// The most a pure writer reaches on the f32 window render's buffer: constant 16-byte words over [items, 84, 84, 3] f32
// (items = T*N, time-major), in maze_window_cta_kernel's address order -- thread t of a 256-thread CTA owns chunk
// column t % 63 of the 1008-byte groups t / 63 + 4j, so every warp store covers 512 contiguous bytes -- with no maze
// logic, no masks and no barrier.  Two grid shapes: one CTA per item (as the render launches), and a persistent grid
// that walks the items in order.  Loaded by scripts/k1_store_ceiling.py.
#include <cuda_runtime.h>
#include <stdint.h>

namespace {
constexpr int kChunksPerGroup = 63;   // 16-byte chunks of one 252-float pixel row
constexpr int kGroups = 84;           // pixel rows of a frame
constexpr int kThreads = 256;
constexpr int R = kThreads / kChunksPerGroup;
constexpr int kFrameChunks = kGroups * kChunksPerGroup;

__device__ __forceinline__ void store_item(uint4* out, size_t b, int tid, uint4 v) {
  const int gsub = tid / kChunksPerGroup, c = tid - gsub * kChunksPerGroup;
  if (gsub >= R) return;
  uint4* o = out + b * kFrameChunks + c;
#pragma unroll
  for (int j = 0; j < kGroups / R; ++j) __stcs(o + (size_t)(gsub + R * j) * kChunksPerGroup, v);
}

__global__ void __launch_bounds__(kThreads) ceiling_cta_per_item(uint4* out) {
  store_item(out, blockIdx.x, threadIdx.x, make_uint4(0x3f800000u, 0u, 0u, 0x3f800000u));
}

__global__ void __launch_bounds__(kThreads) ceiling_persistent(uint4* out, long long items) {
  for (long long b = blockIdx.x; b < items; b += gridDim.x)
    store_item(out, (size_t)b, threadIdx.x, make_uint4(0x3f800000u, 0u, 0u, 0x3f800000u));
}
}  // namespace

extern "C" int k1_ceiling_cta_per_item(void* out, long long items, void* stream) {
  ceiling_cta_per_item<<<(unsigned)items, kThreads, 0, (cudaStream_t)stream>>>(reinterpret_cast<uint4*>(out));
  return (int)cudaGetLastError();
}

extern "C" int k1_ceiling_persistent(void* out, long long items, int grid, void* stream) {
  ceiling_persistent<<<grid, kThreads, 0, (cudaStream_t)stream>>>(reinterpret_cast<uint4*>(out), items);
  return (int)cudaGetLastError();
}
