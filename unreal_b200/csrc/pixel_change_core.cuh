// K2's per-pool-row arithmetic (Environment._calc_pixel_change + _subsample, environment/environment.py:88-99),
// shared by the generic pixel-change kernel (pixel_change.cu) and the host-frame ingest kernel (host_ingest.cu):
// d = |cur - prev| on the 2-pixel-cropped frame, mean over channels, then 4x4 mean (columns first, then rows), in
// exactly numpy's order and roundings -- (d0+d1+d2)/C per pixel, ((m0+m1)+m2)+m3)/4 across a cell row (warp
// shuffles), ((c0+c1)+c2)+c3)/4 down the four rows (shared memory).
#pragma once
#include "common.cuh"

namespace unreal {

constexpr int kMaxCellsPerCta = 64;  // 4 rows x 256 pixels = 1024 threads

template <typename T> struct Px;
template <> struct Px<float> { static __device__ __forceinline__ float load(const float* p) { return __ldcs(p); } };
template <> struct Px<uint8_t> {
  // frames arrive as uint8 and are scaled by /255 like lab_environment.py:99-102
  static __device__ __forceinline__ float load(const uint8_t* p) { return __fdiv_rn((float)__ldcs(p), 255.0f); }
};

// |a-b| channel mean of one pixel, numpy order: ((d0 + d1) + d2) / C
template <int C>
__device__ __forceinline__ float pixel_mean(const float (&a)[C], const float (&b)[C]) {
  float s = fabsf(__fsub_rn(a[0], b[0]));
#pragma unroll
  for (int c = 1; c < C; ++c) s = __fadd_rn(s, fabsf(__fsub_rn(a[c], b[c])));
  return __fdiv_rn(s, (float)C);
}

// after this every lane with (px & 3) == 0 holds the mean of its 4-pixel cell row
__device__ __forceinline__ float cell_row_mean(float m) {
  float v1 = __shfl_down_sync(0xffffffffu, m, 1);
  float v2 = __shfl_down_sync(0xffffffffu, m, 2);
  float v3 = __shfl_down_sync(0xffffffffu, m, 3);
  return __fmul_rn(__fadd_rn(__fadd_rn(__fadd_rn(m, v1), v2), v3), 0.25f);
}

// Threads per block for frames of width w: 4 rows x 4*cells pixels of one pool-row tile, rounded up to whole warps
// (the padding threads only take part in the shuffles).
inline int pool_row_threads(int w) {
  const int pw = (w - 4) / 4;
  const int cells = pw < kMaxCellsPerCta ? pw : kMaxCellsPerCta;
  return (16 * cells + 31) / 32 * 32;
}

// Pool row i, cells j0 .. j0+63 (or up to pw), of the change from frame `prev` to frame `cur` (one [H,W,C] frame each)
// into pc_row[j0 + j].  Every thread of a block of pool_row_threads(W) threads calls it; it contains one __syncthreads
// and leaves s_rows in use by the threads < cells until the caller's next barrier.
template <typename T, int C>
__device__ __forceinline__ void pool_row_change(const T* __restrict__ cur, const T* __restrict__ prev,
                                                float* __restrict__ pc_row, int W, int i, int j0, int pw,
                                                float (&s_rows)[4][kMaxCellsPerCta]) {
  const int cells = min(kMaxCellsPerCta, pw - j0);
  const int tile_px = cells * 4;
  const bool live = threadIdx.x < 4 * tile_px;
  const int r = live ? threadIdx.x / tile_px : 0;  // pixel row inside the pool row, 0..3
  const int p = threadIdx.x - r * tile_px;        // pixel inside the tile
  const size_t off = ((size_t)(4 * i + 2 + r) * W + (size_t)(4 * j0 + 2 + p)) * C;
  float a[C], b[C];
#pragma unroll
  for (int c = 0; c < C; ++c) a[c] = b[c] = 0.f;
  if (live) {
#pragma unroll
    for (int c = 0; c < C; ++c) {
      a[c] = Px<T>::load(cur + off + c);
      b[c] = Px<T>::load(prev + off + c);
    }
  }
  float row = cell_row_mean(pixel_mean<C>(a, b));
  if (live && (p & 3) == 0) s_rows[r][p >> 2] = row;
  __syncthreads();
  if (threadIdx.x < cells) {
    const int j = threadIdx.x;
    float v = __fadd_rn(__fadd_rn(__fadd_rn(s_rows[0][j], s_rows[1][j]), s_rows[2][j]), s_rows[3][j]);
    pc_row[j0 + j] = __fmul_rn(v, 0.25f);
  }
}

}  // namespace unreal
