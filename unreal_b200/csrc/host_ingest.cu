// Host-simulator frames into the device path: everything BatchedFrameEnvironment.process does between the simulator
// calls and its return (environment/frame_environment.py), for N envs in one launch, reading the frames the simulators
// produced straight from the pinned host staging the worker threads wrote (no upload copy).
//
// One CTA per env, K2's block shape (pool_row_threads):
//   1. the new frame row: the step frame (u8 as is, float32 through HostEnvProducer._u8) for an active env; the
//      previous frame for an inactive one when copy_inactive, else the row is left as it is;
//   2. the pixel change of every row over (new row, prev) with K2's arithmetic (pixel_change_core.cuh);
//   3. reward / terminal (0 for inactive envs) and the packed record, as unreal_frame_pack;
//   4. for a terminal active env the reset frame replaces the row and the reset objective the objective;
//   5. last_action / last_reward as the adapter's torch.where updates.
// Reset mode writes the reset frame and objective of every masked env and zeroes its last_action / last_reward.
#include "maze_core.cuh"
#include "pixel_change_core.cuh"

namespace unreal {

struct IngestArgs {
  const void* step_frames;     // [N,H,W,C] staging (device view of pinned host memory)
  const void* reset_frames;
  const float* step_reward;    // [N]
  const uint8_t* step_terminal;
  const float* step_obj;       // [N,G]
  const float* reset_obj;
  const int32_t* action;       // device from here on
  const uint8_t* active;
  const uint8_t* prev;
  uint8_t* out;
  float* pc;
  uint64_t* rec;
  float* reward;
  uint8_t* terminal;
  int32_t* last_action;
  float* last_reward;
  float* objective;
  int h, w, g, copy_inactive;
};

// HostEnvProducer._u8: rint(float64(x) * 255) with round-half-even, clipped to [0, 255] (x finite; the product is exact)
__device__ __forceinline__ uint32_t unit_to_u8(float x) {
  const double d = rint(__dmul_rn((double)x, 255.0));
  return (uint32_t)fmin(fmax(d, 0.0), 255.0);
}

template <typename S> struct Stage;
template <> struct Stage<uint8_t> {   // 16 frame bytes from byte k
  static __device__ __forceinline__ uint4 load16(const uint8_t* src, size_t k) {
    return *reinterpret_cast<const uint4*>(src + k);
  }
};
template <> struct Stage<float> {     // 16 frame bytes from 16 floats at element k
  static __device__ __forceinline__ uint4 load16(const float* src, size_t k) {
    const float4* p = reinterpret_cast<const float4*>(src + k);
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 v = p[j];
      w[j] = unit_to_u8(v.x) | (unit_to_u8(v.y) << 8) | (unit_to_u8(v.z) << 16) | (unit_to_u8(v.w) << 24);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
  }
};

// out[0 .. bytes) <- frame src (bytes % 16 == 0); loads batched so that several PCIe reads per thread are in flight
template <typename S>
__device__ __forceinline__ void ingest_frame(uint8_t* __restrict__ out, const S* __restrict__ src, size_t bytes) {
  constexpr int kB = 4;
  uint4* o = reinterpret_cast<uint4*>(out);
  const size_t n16 = bytes / 16;
  for (size_t k0 = threadIdx.x; k0 < n16; k0 += (size_t)kB * blockDim.x) {
    uint4 v[kB];
#pragma unroll
    for (int j = 0; j < kB; ++j) {
      const size_t k = k0 + (size_t)j * blockDim.x;
      if (k < n16) v[j] = Stage<S>::load16(src, 16 * k);
    }
#pragma unroll
    for (int j = 0; j < kB; ++j) {
      const size_t k = k0 + (size_t)j * blockDim.x;
      if (k < n16) o[k] = v[j];
    }
  }
}

template <typename S, int C, bool kReset>
__global__ void __launch_bounds__(1024) host_frames_ingest_kernel(const IngestArgs g) {
  __shared__ float s_rows[4][kMaxCellsPerCta];
  const int e = blockIdx.x;
  const bool act = g.active == nullptr || g.active[e] != 0;
  const size_t bytes = (size_t)g.h * g.w * C;
  uint8_t* out = g.out + e * bytes;
  const S* reset_frame = static_cast<const S*>(g.reset_frames) + e * bytes;
  if (kReset) {
    if (!act) return;
    ingest_frame<S>(out, reset_frame, bytes);
    for (int k = threadIdx.x; k < g.g; k += blockDim.x) g.objective[(size_t)e * g.g + k] = g.reset_obj[(size_t)e * g.g + k];
    if (threadIdx.x == 0) {
      if (g.last_action) g.last_action[e] = 0;
      if (g.last_reward) g.last_reward[e] = 0.f;
    }
    return;
  }
  const uint8_t* prev = g.prev + e * bytes;
  if (act) ingest_frame<S>(out, static_cast<const S*>(g.step_frames) + e * bytes, bytes);
  else if (g.copy_inactive) ingest_frame<uint8_t>(out, prev, bytes);
  __syncthreads();
  const int ph = (g.h - 4) / 4, pw = (g.w - 4) / 4;
  float* pc = g.pc + (size_t)e * ph * pw;
  for (int i = 0; i < ph; ++i) {
    for (int j0 = 0; j0 < pw; j0 += kMaxCellsPerCta) {
      pool_row_change<uint8_t, C>(out, prev, pc + (size_t)i * pw, g.w, i, j0, pw, s_rows);
      __syncthreads();          // s_rows is reused; after the last row, every read of `out` is done
    }
  }
  const bool term = act && g.step_terminal[e] != 0;
  if (threadIdx.x == 0) {
    const float r = act ? g.step_reward[e] : 0.f;
    const int32_t a = g.action[e];
    g.reward[e] = r;
    g.terminal[e] = term ? 1 : 0;
    g.rec[e] = act ? framed_record(a, r, term ? 1 : 0, g.last_action[e], g.last_reward[e]) : 0ull;
    if (act) {
      g.last_action[e] = term ? 0 : a;
      g.last_reward[e] = term ? 0.f : r;
    }
  }
  if (act) {
    const float* obj = term ? g.reset_obj : g.step_obj;
    for (int k = threadIdx.x; k < g.g; k += blockDim.x) g.objective[(size_t)e * g.g + k] = obj[(size_t)e * g.g + k];
  }
  if (term) ingest_frame<S>(out, reset_frame, bytes);
}

template <typename S, bool kReset>
static void launch_ingest(const IngestArgs& g, int n, int c, cudaStream_t st) {
  const int threads = pool_row_threads(g.w);
  switch (c) {
    case 1: host_frames_ingest_kernel<S, 1, kReset><<<n, threads, 0, st>>>(g); break;
    case 3: host_frames_ingest_kernel<S, 3, kReset><<<n, threads, 0, st>>>(g); break;
    default: host_frames_ingest_kernel<S, 4, kReset><<<n, threads, 0, st>>>(g); break;
  }
}

// the device address of pinned host memory (the same pointer under unified addressing); NULL stays NULL
static int mapped(const void* host, const void** dev, const char* name) {
  *dev = nullptr;
  if (!host) return UNREAL_OK;
  cudaPointerAttributes a;
  const cudaError_t e = cudaPointerGetAttributes(&a, host);
  if (e != cudaSuccess || a.type != cudaMemoryTypeHost || a.devicePointer == nullptr) {
    cudaGetLastError();
    set_error("unreal_host_frames_ingest: %s is not pinned host memory mapped into the device's address space", name);
    return UNREAL_EINVAL;
  }
  *dev = a.devicePointer;
  return UNREAL_OK;
}

}  // namespace unreal

using namespace unreal;

extern "C" int unreal_host_frames_ingest(int mode, const void* step_frames_host, const void* reset_frames_host,
                                         int stage_dtype, const float* step_reward_host,
                                         const uint8_t* step_terminal_host, const float* step_objective_host,
                                         const float* reset_objective_host, const int32_t* action,
                                         const uint8_t* active, const uint8_t* prev, uint8_t* out, int copy_inactive,
                                         float* pc, uint64_t* rec, float* reward, uint8_t* terminal,
                                         int32_t* last_action, float* last_reward, float* objective, int n, int h,
                                         int w, int c, int g, void* stream) {
  const char* fn = "unreal_host_frames_ingest";
  UNREAL_REQUIRE(mode == 0 || mode == 1, "%s: mode %d is not 0 (step) or 1 (reset)", fn, mode);
  UNREAL_REQUIRE(n >= 0 && g >= 0, "%s: n < 0 or g < 0", fn);
  UNREAL_REQUIRE(h >= 8 && w >= 8 && (h - 4) % 4 == 0 && (w - 4) % 4 == 0,
                 "%s: H-4 and W-4 must be positive multiples of 4 (got %dx%d), as _subsample requires", fn, h, w);
  UNREAL_REQUIRE(c == 1 || c == 3 || c == 4, "%s: %d channels not supported (1, 3, 4)", fn, c);
  UNREAL_REQUIRE((w - 4) / 4 <= kMaxCellsPerCta || ((w - 4) / 4) % kMaxCellsPerCta == 0,
                 "%s: frames wider than 260 px need (W-4)/4 to be a multiple of 64", fn);
  UNREAL_REQUIRE(stage_dtype == UNREAL_U8 || stage_dtype == UNREAL_F32, "%s: staging dtype %d is not u8 or f32", fn,
                 stage_dtype);
  if (n == 0) return UNREAL_OK;
  const bool step = mode == 0;
  UNREAL_REQUIRE(reset_frames_host && out, "%s: null reset frames or out", fn);
  UNREAL_REQUIRE(!step || (step_frames_host && step_reward_host && step_terminal_host && action && prev && pc && rec &&
                           reward && terminal && last_action && last_reward),
                 "%s: null argument of the step mode", fn);
  UNREAL_REQUIRE(g == 0 || (objective && reset_objective_host && (!step || step_objective_host)),
                 "%s: g = %d needs the objective buffers", fn, g);
  UNREAL_REQUIRE(aligned16(out) && (!step || aligned16(prev)) && aligned16(reset_frames_host) &&
                     (!step || aligned16(step_frames_host)),
                 "%s: frame buffers must be 16-byte aligned", fn);
  IngestArgs a{};
  int rc = mapped(step_frames_host, &a.step_frames, "step_frames_host");
  if (!rc) rc = mapped(reset_frames_host, &a.reset_frames, "reset_frames_host");
  if (!rc) rc = mapped(step_reward_host, reinterpret_cast<const void**>(&a.step_reward), "step_reward_host");
  if (!rc) rc = mapped(step_terminal_host, reinterpret_cast<const void**>(&a.step_terminal), "step_terminal_host");
  if (!rc && g) rc = mapped(step_objective_host, reinterpret_cast<const void**>(&a.step_obj), "step_objective_host");
  if (!rc && g) rc = mapped(reset_objective_host, reinterpret_cast<const void**>(&a.reset_obj), "reset_objective_host");
  if (rc) return rc;
  a.action = action; a.active = active; a.prev = prev; a.out = out; a.pc = pc; a.rec = rec; a.reward = reward;
  a.terminal = terminal; a.last_action = last_action; a.last_reward = last_reward; a.objective = objective;
  a.h = h; a.w = w; a.g = g; a.copy_inactive = copy_inactive ? 1 : 0;
  cudaStream_t st = as_stream(stream);
  if (stage_dtype == UNREAL_U8) {
    if (step) launch_ingest<uint8_t, false>(a, n, c, st);
    else launch_ingest<uint8_t, true>(a, n, c, st);
  } else {
    if (step) launch_ingest<float, false>(a, n, c, st);
    else launch_ingest<float, true>(a, n, c, st);
  }
  UNREAL_LAUNCH_CHECK("host_frames_ingest_kernel");
  return UNREAL_OK;
}
