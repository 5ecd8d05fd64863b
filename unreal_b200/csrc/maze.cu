// K1: fused maze step + render + pixel-change for thousands of 7x7 mazes (sm_100a).
//
// Replaces, per env and per step, MazeEnvironment.process (environment/maze_environment.py:98-128):
// _move/_clamp/_is_wall (:66-91), reward/terminal (:114-122), _get_current_image (:93-96) and
// Environment._calc_pixel_change (environment/environment.py:88-99).
//
// The kernel is a pure HBM writer: 84 672 B (f32) or 21 168 B (u8) of frame + 1 600 B of
// pixel-change map per env-step against ~30 B of state read.  Two render variants:
//   variant 0 (default): one CTA per env in env order; every thread builds its 128-bit words
//     from per-lane bit masks and stores them directly, 512 contiguous aligned bytes per warp.
//   variant 1: each persistent CTA keeps wall-only frame templates in shared memory, patches
//     the 12x12 agent block (144 elements) and hands the whole frame to the TMA engine with
//     cp.async.bulk (shared -> global), multi-buffered so patching overlaps the store.
//   variant 2: one warp per env, same mask-built words, no shared memory or barriers.
// The default is whichever measured fastest on B200 (profiles/, DESIGN.md).
#include <map>
#include <mutex>

#include "common.cuh"
#include "maze_core.cuh"
#include "tc05.cuh"

namespace unreal {
using namespace tc05;

__constant__ MazeLayout c_maze;

static const char kReferenceMap[] =
    "--+---G"
    "--+-+++"
    "S-+---+"
    "--+++--"
    "--+-+--"
    "--+----"
    "-----++";  // maze_environment.py:18-25

constexpr int kFrameElems = UNREAL_FRAME_HW * UNREAL_FRAME_HW * 3;  // 21168
constexpr int kRowElems = UNREAL_FRAME_HW * 3;                      // 252
constexpr int kPcElems = UNREAL_PC_CELLS * UNREAL_PC_CELLS;         // 400
constexpr int kThreads = 256;

struct StepArgs {
  int32_t* pos;
  const int32_t* action;
  const uint8_t* active;
  float* reward;
  uint8_t* terminal;
  int32_t* last_action;
  float* last_reward;
  void* obs;
  float* pc;
  uint64_t* rec;
  int n;
  int auto_reset;
};

struct EnvInfo {
  int rx, ry;          // cell drawn into obs
  int x0, y0, x1, y1;  // cells defining the pixel change
  int live;            // 0: env skipped, nothing large is written
};

// One thread per env: everything of process() except the two big outputs.
template <bool kStep>
__device__ __forceinline__ EnvInfo env_logic(const StepArgs& a, int e) {
  EnvInfo o;
  int x = a.pos[2 * e], y = a.pos[2 * e + 1];
  o.rx = x; o.ry = y; o.x0 = x; o.y0 = y; o.x1 = x; o.y1 = y; o.live = 1;
  if (!kStep) return o;
  if (a.active != nullptr && a.active[e] == 0) {
    o.live = 0;
    a.reward[e] = 0.f;
    a.terminal[e] = 0;
    if (a.rec) a.rec[e] = 0ull;
    return o;
  }
  int act = a.action[e];
  MazeStep s = maze_step_core(c_maze, x, y, act);
  int la = a.last_action[e];
  float lr = a.last_reward[e];
  if (a.rec) a.rec[e] = frame_pack(x, y, s.x1, s.y1, act, s.reward, s.terminal, la, (int)lr);
  a.reward[e] = (float)s.reward;
  a.terminal[e] = (uint8_t)s.terminal;
  o.x1 = s.x1; o.y1 = s.y1;
  if (s.terminal && a.auto_reset) {  // caller-side reset of trainer.py:201-204,:279-296 + reset() :50-55
    o.rx = c_maze.start_x; o.ry = c_maze.start_y;
    a.last_action[e] = 0;
    a.last_reward[e] = 0.f;
  } else {
    o.rx = s.x1; o.ry = s.y1;
    a.last_action[e] = act;             // :126
    a.last_reward[e] = (float)s.reward; // :127
  }
  a.pos[2 * e] = o.rx;
  a.pos[2 * e + 1] = o.ry;
  return o;
}

// The 4 pool-column weights pc_overlap(j0 + u, c), u = 0..3, as the bytes of one word: along the pool index a cell's
// weights are the run [2, 4, 4, 2] starting at 3c - 1, so the word is that run shifted to byte offset 3c - 1 - j0.
__device__ __forceinline__ uint32_t pc_overlap4(int j0, int c) {
  const int s = 8 * (3 * c - 1 - j0);
  const uint32_t run = 0x02040402u;
  return s >= 0 ? (s < 32 ? run << s : 0u) : (s > -32 ? run >> -s : 0u);
}

// 100 threads write the 20x20 map of one env as float4: k/48 with
// k = ov(i,y0)*ov(j,x0) + ov(i,y1)*ov(j,x1), 0 when the agent did not move.
__device__ __forceinline__ float4 pc_value4(int x0, int y0, int x1, int y1, int q) {
  const int i = q / 5, j0 = (q - i * 5) * 4;
  const bool moved = (x0 != x1) || (y0 != y1);
  // the four k of the float4 as bytes (each an integer <= 32), two multiply-adds for all four
  const uint32_t k4 = moved ? (uint32_t)pc_overlap(i, y0) * pc_overlap4(j0, x0) + (uint32_t)pc_overlap(i, y1) * pc_overlap4(j0, x1)
                            : 0u;
  float v[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const float k = (float)((k4 >> (8 * u)) & 0xffu);
    // k / 48 correctly rounded (= float32 of the reference's float64 means) without the IEEE-division sequence: one
    // Newton correction of k * RN(1/48) with exact FMA residuals; equal to k / 48.0f for every integer k < 200
    // (checked exhaustively; tests/test_gpu_maze.py compares every cell pair with the literal reference computation)
    const float q = k * 0x1.555556p-6f;
    v[u] = __fmaf_rn(__fmaf_rn(-q, 48.0f, k), 0x1.555556p-6f, q);
  }
  return make_float4(v[0], v[1], v[2], v[3]);
}
// the maps are write-once outputs nothing in the pass reads back: streamed, so they do not hold L2 against the frames
__device__ __forceinline__ void write_pc(float* pc, const EnvInfo& f, int q) {
  __stcs(reinterpret_cast<float4*>(pc) + q, pc_value4(f.x0, f.y0, f.x1, f.y1, q));
}

template <typename T> struct One;
template <> struct One<float> { static __device__ __forceinline__ float v() { return 1.0f; } };
template <> struct One<uint8_t> { static __device__ __forceinline__ uint8_t v() { return 255; } };

// ------------------------------------------------------------------------------------
// variant 1: shared-memory frame templates + TMA bulk stores.
// ------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void set_agent(T* buf, int x, int y, int t, T val) {
  // t in [0,144): pixel (12x + t%12, 12y + t/12), channel 1   (_put_pixel :57-60)
  int j = t / 12, i = t - j * 12;
  buf[((12 * y + j) * UNREAL_FRAME_HW + 12 * x + i) * 3 + 1] = val;
}

template <typename T, int kBufs, bool kStep>
__global__ void __launch_bounds__(kThreads) maze_tma_kernel(StepArgs a) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  __shared__ EnvInfo s_info[2];
  T* bufs = reinterpret_cast<T*>(smem_raw);
  const int tid = threadIdx.x;
  constexpr uint32_t kFrameBytes = kFrameElems * sizeof(T);

  // prologue: wall-only template (channel 0) in every buffer   (_setup :30-41)
  for (int i = tid; i < kFrameElems; i += kThreads) {
    int row = i / kRowElems;
    int f = i - row * kRowElems;
    int px = f / 3;
    int chn = f - px * 3;
    bool on = (chn == 0) && ((c_maze.wall_rows[row / 12] >> (px / 12)) & 1u);
    T v = on ? One<T>::v() : (T)0;
#pragma unroll
    for (int b = 0; b < kBufs; ++b) bufs[(size_t)b * kFrameElems + i] = v;
  }
  int drawn[kBufs];  // agent cell currently patched into buffer b (x | y<<4), -1 none
#pragma unroll
  for (int b = 0; b < kBufs; ++b) drawn[b] = -1;
  fence_proxy_async_smem();  // template writes must be visible to the TMA engine too
  __syncthreads();

  int it = 0;
  for (int e = blockIdx.x; e < a.n; e += gridDim.x, ++it) {
    const int b = it % kBufs;
    if (tid == 0) {
      s_info[it & 1] = env_logic<kStep>(a, e);
      bulk_wait_read<kBufs - 1>();  // the store issued kBufs iterations ago has drained buffer b
    }
    __syncthreads();
    const EnvInfo f = s_info[it & 1];
    const bool store = f.live && a.obs != nullptr;
    if (f.live && a.pc != nullptr && tid < kPcElems / 4) write_pc(a.pc + (size_t)e * kPcElems, f, tid);
    if (store) {
      T* buf = bufs + (size_t)b * kFrameElems;
      int want = f.rx | (f.ry << 4);
      int have = -1;
#pragma unroll
      for (int k = 0; k < kBufs; ++k) have = (k == b) ? drawn[k] : have;
      if (have != want && tid < 144) {
        if (have >= 0) set_agent<T>(buf, have & 15, have >> 4, tid, (T)0);
        set_agent<T>(buf, f.rx, f.ry, tid, One<T>::v());
        fence_proxy_async_smem();  // generic-proxy writes -> visible to the async (TMA) proxy
      }
#pragma unroll
      for (int k = 0; k < kBufs; ++k) drawn[k] = (k == b) ? want : drawn[k];
    }
    __syncthreads();
    if (tid == 0) {
      if (store) bulk_store(reinterpret_cast<T*>(a.obs) + (size_t)e * kFrameElems,
                            bufs + (size_t)b * kFrameElems, kFrameBytes);
      bulk_commit();  // one group per iteration (possibly empty) keeps the wait arithmetic uniform
    }
  }
  if (tid == 0) bulk_wait_all();
}

// ------------------------------------------------------------------------------------
// variant 2: one warp per env, no shared memory, no barriers.
// A frame is a sequence of identical-size "groups" of 63 x 16 B = 1008 B: one pixel row for
// f32 (252 floats), four pixel rows for u8 (4 x 252 B).  All groups of one maze-cell row
// ("band", 12 pixel rows) are identical, so a lane computes the two 16-byte chunks it owns
// (lane, lane+32) once per band from per-lane bit masks and stores them to every group of
// the band: 512 contiguous bytes per warp store instruction.
// A 16-byte chunk covers < 6 pixels, hence at most two maze-cell columns (A and B).
// ------------------------------------------------------------------------------------
template <typename T> struct Chunk;
template <> struct Chunk<float> { static constexpr int kElems = 4, kGroupsPerBand = 12; };
template <> struct Chunk<uint8_t> { static constexpr int kElems = 16, kGroupsPerBand = 3; };

struct ChunkMasks {
  uint32_t wallA[4], wallB[4], agentA[4], agentB[4];  // all-ones element patterns
  int cxA, cxB;
};

template <typename T>
__device__ __forceinline__ ChunkMasks make_masks(int chunk) {
  ChunkMasks m;
#pragma unroll
  for (int w = 0; w < 4; ++w) m.wallA[w] = m.wallB[w] = m.agentA[w] = m.agentB[w] = 0u;
  constexpr int E = Chunk<T>::kElems;
  const int first = (chunk * E) % kRowElems;
  m.cxA = (first / 3) / 12;
  m.cxB = m.cxA;
#pragma unroll
  for (int i = 0; i < E; ++i) {
    int col = (chunk * E + i) % kRowElems;
    int px = col / 3, ch = col - px * 3, cx = px / 12;
    uint32_t bits = (sizeof(T) == 4) ? 0x3f800000u : (0xffu << (8 * (i & 3)));
    int w = (sizeof(T) == 4) ? i : (i >> 2);
    bool isA = (cx == m.cxA);
    if (!isA) m.cxB = cx;
    if (ch == 0) { if (isA) m.wallA[w] |= bits; else m.wallB[w] |= bits; }
    if (ch == 1) { if (isA) m.agentA[w] |= bits; else m.agentB[w] |= bits; }
  }
  return m;
}

__device__ __forceinline__ uint4 band_value(const ChunkMasks& m, uint32_t walls, bool agent_band, int ax) {
  uint32_t wa = ((walls >> m.cxA) & 1u) ? 0xffffffffu : 0u;
  uint32_t wb = ((walls >> m.cxB) & 1u) ? 0xffffffffu : 0u;
  uint32_t aa = (agent_band && m.cxA == ax) ? 0xffffffffu : 0u;
  uint32_t ab = (agent_band && m.cxB == ax) ? 0xffffffffu : 0u;
  uint4 v;
  v.x = (m.wallA[0] & wa) | (m.wallB[0] & wb) | (m.agentA[0] & aa) | (m.agentB[0] & ab);
  v.y = (m.wallA[1] & wa) | (m.wallB[1] & wb) | (m.agentA[1] & aa) | (m.agentB[1] & ab);
  v.z = (m.wallA[2] & wa) | (m.wallB[2] & wb) | (m.agentA[2] & aa) | (m.agentB[2] & ab);
  v.w = (m.wallA[3] & wa) | (m.wallB[3] & wb) | (m.agentA[3] & aa) | (m.agentB[3] & ab);
  return v;
}

template <typename T, bool kStep, int kWarps>
__global__ void __launch_bounds__(kWarps * 32) maze_warp_kernel(StepArgs a) {
  const int lane = threadIdx.x & 31;
  const int e = blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (e >= a.n) return;
  int packed = 0;
  if (lane == 0) {
    EnvInfo f = env_logic<kStep>(a, e);
    packed = f.rx | (f.ry << 3) | (f.x0 << 6) | (f.y0 << 9) | (f.x1 << 12) | (f.y1 << 15) | (f.live << 18);
  }
  packed = __shfl_sync(0xffffffffu, packed, 0);
  EnvInfo f;
  f.rx = packed & 7; f.ry = (packed >> 3) & 7; f.x0 = (packed >> 6) & 7; f.y0 = (packed >> 9) & 7;
  f.x1 = (packed >> 12) & 7; f.y1 = (packed >> 15) & 7; f.live = (packed >> 18) & 1;
  if (!f.live) return;
  if (a.pc != nullptr) {
    float* pc = a.pc + (size_t)e * kPcElems;
#pragma unroll
    for (int q = lane; q < kPcElems / 4; q += 32) write_pc(pc, f, q);
  }
  if (a.obs == nullptr) return;
  constexpr int G = Chunk<T>::kGroupsPerBand;
  constexpr int kChunksPerGroup = 63;
  const ChunkMasks m0 = make_masks<T>(lane);
  const ChunkMasks m1 = make_masks<T>(lane + 32);
  const bool has1 = lane + 32 < kChunksPerGroup;
  uint4* out = reinterpret_cast<uint4*>(reinterpret_cast<T*>(a.obs) + (size_t)e * kFrameElems) + lane;
#pragma unroll
  for (int cy = 0; cy < UNREAL_MAZE_GRID; ++cy) {
    const uint32_t walls = c_maze.wall_rows[cy];
    const uint4 v0 = band_value(m0, walls, cy == f.ry, f.rx);
    const uint4 v1 = band_value(m1, walls, cy == f.ry, f.rx);
#pragma unroll
    for (int g = 0; g < G; ++g) {
      uint4* p = out + (size_t)(cy * G + g) * kChunksPerGroup;
      __stcs(p, v0);
      if (has1) __stcs(p + 32, v1);
    }
  }
}

// ------------------------------------------------------------------------------------
// variant 0 (default): one CTA per env, launched non-persistently in env order.
// Thread t owns chunk column t % 63 of groups t / 63 + R*j (R = kThreads / 63), so one pass
// of the CTA writes R whole groups = R*1008 contiguous bytes and every warp store is 512
// contiguous, sector-aligned bytes.  Measured on B200 (profiles/store_patterns_r1.md):
// in-order one-CTA-per-env beats persistent/strided and warp-per-env write patterns.
// ------------------------------------------------------------------------------------
template <typename T, bool kStep, int kThreads>
__global__ void __launch_bounds__(kThreads) maze_cta_kernel(StepArgs a) {
  __shared__ EnvInfo s_info;
  constexpr int kChunksPerGroup = 63;
  constexpr int R = kThreads / kChunksPerGroup;
  constexpr int G = Chunk<T>::kGroupsPerBand;
  constexpr int kGroups = G * UNREAL_MAZE_GRID;
  const int tid = threadIdx.x;
  const int e = blockIdx.x;
  if (tid == 0) s_info = env_logic<kStep>(a, e);
  const int gsub = tid / kChunksPerGroup;
  const int c = tid - gsub * kChunksPerGroup;
  const ChunkMasks m = make_masks<T>(c);   // overlaps the logic thread's global loads
  __syncthreads();
  const EnvInfo f = s_info;
  if (!f.live) return;
  if (a.pc != nullptr && tid >= kThreads - kPcElems / 4) write_pc(a.pc + (size_t)e * kPcElems, f, tid - (kThreads - kPcElems / 4));
  if (a.obs == nullptr || gsub >= R) return;
  uint4* out = reinterpret_cast<uint4*>(reinterpret_cast<T*>(a.obs) + (size_t)e * kFrameElems) + c;
#pragma unroll
  for (int j = 0; j < (kGroups + R - 1) / R; ++j) {
    const int g = gsub + R * j;
    if (g < kGroups) {
      const int cy = g / G;
      __stcs(out + (size_t)g * kChunksPerGroup, band_value(m, c_maze.wall_rows[cy], cy == f.ry, f.rx));
    }
  }
}


// ------------------------------------------------------------------------------------
// Window form: T rollout steps of every env in ONE launch, for callers that hold the T actions up front (scripted
// policies, re-simulation of recorded trajectories, BASELINE configs[1] whose actions are an input of the pass).
// Work item b = t*N + e writes step t of env e into the time-major [T,N,...] buffers, in the same address order as T
// per-step launches -- but without the T launch ramps / drains and without the inter-launch dependency on the state:
// every item re-simulates its env's integer steps 0..t-1 from the window's start state (t <= 31 iterations of a few
// instructions, all lanes of a warp in lock step, actions fetched by lanes 0..t in one load and broadcast by shuffle)
// and then performs step t exactly like env_logic.  The start state is only READ here; maze_window_state_kernel
// (one thread per env, launched after) advances pos / last_action / last_reward by the T steps.
// ------------------------------------------------------------------------------------
struct WindowArgs {
  const int32_t* pos;
  const int32_t* last_action;
  const float* last_reward;
  const int32_t* action;   // [T,N]
  float* reward;           // [T,N]
  uint8_t* terminal;       // [T,N]
  void* obs;               // [T,N,84,84,3] (nullable)
  float* pc;               // [T,N,20,20]   (nullable)
  uint64_t* rec;           // [T,N]         (nullable)
  int n, t, auto_reset;
};

struct MazeCursor { int x, y, la; float lr; };

__device__ __forceinline__ void cursor_advance(MazeCursor& c, const MazeStep& s, int act, int auto_reset) {
  if (s.terminal && auto_reset) { c.x = c_maze.start_x; c.y = c_maze.start_y; c.la = 0; c.lr = 0.f; }
  else { c.x = s.x1; c.y = s.y1; c.la = act; c.lr = (float)s.reward; }
}

// executed by all 32 lanes of a warp (uniform control flow); lane 0 writes the small outputs of item (t, e)
__device__ __forceinline__ EnvInfo window_logic(const WindowArgs& a, int e, int t, int lane) {
  const int mine = (lane <= t) ? a.action[(size_t)lane * a.n + e] : 0;
  MazeCursor c{a.pos[2 * e], a.pos[2 * e + 1], a.last_action[e], a.last_reward[e]};
  for (int s = 0; s < t; ++s) {
    const int act = __shfl_sync(0xffffffffu, mine, s);
    cursor_advance(c, maze_step_core(c_maze, c.x, c.y, act), act, a.auto_reset);
  }
  const int act = __shfl_sync(0xffffffffu, mine, t);
  const MazeStep st = maze_step_core(c_maze, c.x, c.y, act);
  const size_t b = (size_t)t * a.n + e;
  if (lane == 0) {
    if (a.rec) a.rec[b] = frame_pack(c.x, c.y, st.x1, st.y1, act, st.reward, st.terminal, c.la, (int)c.lr);
    a.reward[b] = (float)st.reward;
    a.terminal[b] = (uint8_t)st.terminal;
  }
  EnvInfo o;
  o.x0 = c.x; o.y0 = c.y; o.x1 = st.x1; o.y1 = st.y1; o.live = 1;
  const bool reset = st.terminal && a.auto_reset;
  o.rx = reset ? c_maze.start_x : st.x1;
  o.ry = reset ? c_maze.start_y : st.y1;
  return o;
}

// t <= 32: the actions are all loaded before the recurrence (unrolled, predicated), one memory round trip instead of t
__global__ void maze_window_state_kernel(int32_t* pos, int32_t* last_action, float* last_reward,
                                         const int32_t* __restrict__ action, int n, int t, int auto_reset) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  int acts[32];
#pragma unroll
  for (int s = 0; s < 32; ++s) acts[s] = (s < t) ? __ldg(action + (size_t)s * n + e) : 0;
  MazeCursor c{pos[2 * e], pos[2 * e + 1], last_action[e], last_reward[e]};
#pragma unroll
  for (int s = 0; s < 32; ++s)
    if (s < t) cursor_advance(c, maze_step_core(c_maze, c.x, c.y, acts[s]), acts[s], auto_reset);
  pos[2 * e] = c.x; pos[2 * e + 1] = c.y; last_action[e] = c.la; last_reward[e] = c.lr;
}

// one CTA per item, the render of maze_cta_kernel
template <typename T, int kThreads>
__global__ void __launch_bounds__(kThreads) maze_window_cta_kernel(WindowArgs a) {
  __shared__ EnvInfo s_info;
  constexpr int kChunksPerGroup = 63;
  constexpr int R = kThreads / kChunksPerGroup;
  constexpr int G = Chunk<T>::kGroupsPerBand;
  constexpr int kGroups = G * UNREAL_MAZE_GRID;
  const int tid = threadIdx.x;
  const size_t b = blockIdx.x;
  const int t = (int)(b / a.n), e = (int)(b - (size_t)t * a.n);
  if (tid < 32) {
    const EnvInfo f = window_logic(a, e, t, tid);
    if (tid == 0) s_info = f;
  }
  const int gsub = tid / kChunksPerGroup;
  const int c = tid - gsub * kChunksPerGroup;
  const ChunkMasks m = make_masks<T>(c);
  __syncthreads();
  const EnvInfo f = s_info;
  if (a.pc != nullptr && tid >= kThreads - kPcElems / 4) write_pc(a.pc + b * kPcElems, f, tid - (kThreads - kPcElems / 4));
  if (a.obs == nullptr || gsub >= R) return;
  uint4* out = reinterpret_cast<uint4*>(reinterpret_cast<T*>(a.obs) + b * kFrameElems) + c;
#pragma unroll
  for (int j = 0; j < (kGroups + R - 1) / R; ++j) {
    const int g = gsub + R * j;
    if (g < kGroups) {
      const int cy = g / G;
      __stcs(out + (size_t)g * kChunksPerGroup, band_value(m, c_maze.wall_rows[cy], cy == f.ry, f.rx));
    }
  }
}

// one warp per item, the render of maze_warp_kernel
template <typename T, int kWarps>
__global__ void __launch_bounds__(kWarps * 32) maze_window_warp_kernel(WindowArgs a) {
  const int lane = threadIdx.x & 31;
  const size_t b = (size_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (b >= (size_t)a.n * a.t) return;
  const int t = (int)(b / a.n), e = (int)(b - (size_t)t * a.n);
  const EnvInfo f = window_logic(a, e, t, lane);
  if (a.pc != nullptr) {
    float* pc = a.pc + b * kPcElems;
#pragma unroll
    for (int q = lane; q < kPcElems / 4; q += 32) write_pc(pc, f, q);
  }
  if (a.obs == nullptr) return;
  constexpr int G = Chunk<T>::kGroupsPerBand;
  constexpr int kChunksPerGroup = 63;
  const ChunkMasks m0 = make_masks<T>(lane);
  const ChunkMasks m1 = make_masks<T>(lane + 32);
  const bool has1 = lane + 32 < kChunksPerGroup;
  uint4* out = reinterpret_cast<uint4*>(reinterpret_cast<T*>(a.obs) + b * kFrameElems) + lane;
#pragma unroll
  for (int cy = 0; cy < UNREAL_MAZE_GRID; ++cy) {
    const uint32_t walls = c_maze.wall_rows[cy];
    const uint4 v0 = band_value(m0, walls, cy == f.ry, f.rx);
    const uint4 v1 = band_value(m1, walls, cy == f.ry, f.rx);
#pragma unroll
    for (int g = 0; g < G; ++g) {
      uint4* p = out + (size_t)(cy * G + g) * kChunksPerGroup;
      __stcs(p, v0);
      if (has1) __stcs(p + 32, v1);
    }
  }
}

// Window form, one WARP per env walking its T steps in order (no re-simulation): the warp keeps the env's cursor, its
// two chunk columns' wall patterns of all 7 bands in registers (they do not depend on the env or the step), and per
// step only builds the agent band's two words, writes the 20x20 map and streams the frame out -- ~300 integer
// instructions per 21 KB u8 frame instead of ~1000 (ncu of maze_window_warp_kernel<u8>: ALU pipe 75 % busy at 49 % of
// DRAM: instruction-bound).  Lane 0 writes the small outputs and, after the last step, the env's state.
// (Measured alternative: the wall words in a 7 KB shared-memory table -- 80 registers instead of 128, twice the resident
// warps -- is SLOWER, 0.83 vs 0.89 of HBM: the 14 LDS.128 per frame sit in front of the stores.)
template <typename T, int kWarps>
__global__ void __launch_bounds__(kWarps * 32) maze_window_env_kernel(WindowArgs a, int32_t* pos_out, int32_t* la_out,
                                                                      float* lr_out) {
  const int lane = threadIdx.x & 31;
  const int e = blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (e >= a.n) return;
  constexpr int G = Chunk<T>::kGroupsPerBand;
  constexpr int kChunksPerGroup = 63;
  const ChunkMasks m0 = make_masks<T>(lane);
  const ChunkMasks m1 = make_masks<T>(lane + 32);
  const bool has1 = lane + 32 < kChunksPerGroup;
  uint4 w0[UNREAL_MAZE_GRID], w1[UNREAL_MAZE_GRID];
#pragma unroll
  for (int cy = 0; cy < UNREAL_MAZE_GRID; ++cy) {
    w0[cy] = band_value(m0, c_maze.wall_rows[cy], false, 0);
    w1[cy] = band_value(m1, c_maze.wall_rows[cy], false, 0);
  }
  const int mine = (lane < a.t) ? a.action[(size_t)lane * a.n + e] : 0;
  MazeCursor c{a.pos[2 * e], a.pos[2 * e + 1], a.last_action[e], a.last_reward[e]};
  for (int t = 0; t < a.t; ++t) {
    const int act = __shfl_sync(0xffffffffu, mine, t);
    const MazeStep st = maze_step_core(c_maze, c.x, c.y, act);
    const size_t b = (size_t)t * a.n + e;
    if (lane == 0) {
      if (a.rec) a.rec[b] = frame_pack(c.x, c.y, st.x1, st.y1, act, st.reward, st.terminal, c.la, (int)c.lr);
      a.reward[b] = (float)st.reward;
      a.terminal[b] = (uint8_t)st.terminal;
    }
    EnvInfo f;
    f.x0 = c.x; f.y0 = c.y; f.x1 = st.x1; f.y1 = st.y1; f.live = 1;
    cursor_advance(c, st, act, a.auto_reset);
    f.rx = c.x; f.ry = c.y;                                  // the frame shows the cell the env is in after the step
    if (a.pc != nullptr) {
      float* pc = a.pc + b * kPcElems;
#pragma unroll
      for (int q = lane; q < kPcElems / 4; q += 32) write_pc(pc, f, q);
    }
    if (a.obs == nullptr) continue;
    uint4* out = reinterpret_cast<uint4*>(reinterpret_cast<T*>(a.obs) + b * kFrameElems) + lane;
    const uint4 ag0 = band_value(m0, 0u, true, f.rx), ag1 = band_value(m1, 0u, true, f.rx);   // agent words only
#pragma unroll
    for (int cy = 0; cy < UNREAL_MAZE_GRID; ++cy) {
      uint4 v0 = w0[cy], v1 = w1[cy];
      if (cy == f.ry) {
        v0.x |= ag0.x; v0.y |= ag0.y; v0.z |= ag0.z; v0.w |= ag0.w;
        v1.x |= ag1.x; v1.y |= ag1.y; v1.z |= ag1.z; v1.w |= ag1.w;
      }
#pragma unroll
      for (int g = 0; g < G; ++g) {
        uint4* p = out + (size_t)(cy * G + g) * kChunksPerGroup;
        __stcs(p, v0);
        if (has1) __stcs(p + 32, v1);
      }
    }
  }
  if (lane == 0) { pos_out[2 * e] = c.x; pos_out[2 * e + 1] = c.y; la_out[e] = c.la; lr_out[e] = c.lr; }
}

// ------------------------------------------------------------------------------------
// x'' render: the frame directly in the conv1 kernels' input layout (csrc/conv_tcgen05.cu):
// bf16 planes [6][441][8], x''[q][Y*21+X][e] = frame[4Y+dy, 4X+dx, c] with dy*12+dx*3+c = 8q+e.
// A 4x4 pixel block lies inside one 12-pixel maze cell, so a plane row is one of three constant
// 16-byte patterns (empty / wall: channel 0 / agent: channel 1).  42 336 B per frame instead of
// 84 672 B of f32 plus a separate space-to-depth pass.
// ------------------------------------------------------------------------------------
template <bool kStep>
__global__ void __launch_bounds__(256) maze_s2d_kernel(StepArgs a) {
  __shared__ EnvInfo s_info;
  const int tid = threadIdx.x;
  const int e = blockIdx.x;
  if (tid == 0) s_info = env_logic<kStep>(a, e);
  __syncthreads();
  const EnvInfo f = s_info;
  if (!f.live) return;
  if (a.pc != nullptr && tid >= 256 - kPcElems / 4) write_pc(a.pc + (size_t)e * kPcElems, f, tid - (256 - kPcElems / 4));
  if (a.obs == nullptr) return;
  uint4* out = reinterpret_cast<uint4*>(a.obs) + (size_t)e * (6 * 441);
  // a thread owns pixels tid and tid + 256 of every plane: classify them once (bit0 wall, bit1 agent) ...
  int kind[2];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int pix = tid + h * 256;
    const int Y = pix / 21, X = pix - Y * 21;
    const int cx = X / 3, cy = Y / 3;
    kind[h] = pix < 441 ? (int)((c_maze.wall_rows[cy] >> cx) & 1u) | (((cx == f.rx) && (cy == f.ry)) ? 2 : 0) : -1;
  }
  // ... then per plane the 16-byte row is one of four constants: element i of plane q is channel
  // (8q + i) mod 3; walls set channel 0, the agent channel 1
#pragma unroll
  for (int q = 0; q < 6; ++q) {
    const int base = (2 * q) % 3;
    uint32_t wl[4], ag[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int c0 = (base + 2 * k) % 3, c1 = (base + 2 * k + 1) % 3;
      wl[k] = (c0 == 0 ? 0x3f80u : 0u) | (c1 == 0 ? 0x3f800000u : 0u);
      ag[k] = (c0 == 1 ? 0x3f80u : 0u) | (c1 == 1 ? 0x3f800000u : 0u);
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (kind[h] < 0) continue;
      const uint32_t mw = (kind[h] & 1) ? 0xffffffffu : 0u, ma = (kind[h] & 2) ? 0xffffffffu : 0u;
      __stcs(out + q * 441 + tid + h * 256, make_uint4((wl[0] & mw) | (ag[0] & ma), (wl[1] & mw) | (ag[1] & ma),
                                                       (wl[2] & mw) | (ag[2] & ma), (wl[3] & mw) | (ag[3] & ma)));
    }
  }
}

// pixel change between arbitrary cell pairs (re-materialising maps of replayed frames)
__global__ void __launch_bounds__(128) maze_pc_pairs_kernel(const int32_t* __restrict__ p0,
                                                            const int32_t* __restrict__ p1, float* pc, int m) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  int e = idx / (kPcElems / 4), q = idx - e * (kPcElems / 4);
  if (e >= m) return;
  EnvInfo f;
  f.x0 = p0[2 * e]; f.y0 = p0[2 * e + 1]; f.x1 = p1[2 * e]; f.y1 = p1[2 * e + 1];
  f.rx = f.ry = 0; f.live = 1;
  write_pc(pc + (size_t)e * kPcElems, f, q);
}

// Trainer._process_pc (trainer.py:339-380) on replayed maze cells in ONE pass: pc_R[t] = pixel_change(cell_t, cell_t+1) +
// gamma_pc * pc_R[t+1] with the map's closed form evaluated in registers -- the [L,N,20,20] pixel-change maps
// (maze_pc_pairs_kernel: 262 MB written, then read back by pc_targets_kernel at 8192 envs) never exist.  One thread per
// (env, float4 of the map); the same arithmetic, in the same order, as the two kernels it replaces.
__global__ void __launch_bounds__(128) maze_pc_targets_kernel(const int2* __restrict__ p0, const int2* __restrict__ p1,
                                                              const int32_t* __restrict__ len, const float4* __restrict__ boot,
                                                              float g, float4* __restrict__ tgt, int T, int N) {
  const size_t per_t = (size_t)N * (kPcElems / 4);
  const size_t idx = (size_t)blockIdx.x * 128 + threadIdx.x;
  if (idx >= per_t) return;
  const int n = (int)(idx / (kPcElems / 4)), q = (int)(idx - (size_t)n * (kPcElems / 4));
  const int n_t = len ? max(0, min(len[n], T)) : T;
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 R = boot[idx];
  for (int t = T - 1; t >= n_t; --t) __stcs(tgt + (size_t)t * per_t + idx, zero);
#pragma unroll 4
  for (int t = n_t - 1; t >= 0; --t) {
    const int2 a = __ldg(p0 + (size_t)t * N + n), b = __ldg(p1 + (size_t)t * N + n);
    const float4 pc = pc_value4(a.x, a.y, b.x, b.y, q);
    R.x = __fadd_rn(pc.x, __fmul_rn(g, R.x));   // pc_R = pixel_change + gamma_pc * pc_R   (:361)
    R.y = __fadd_rn(pc.y, __fmul_rn(g, R.y));
    R.z = __fadd_rn(pc.z, __fmul_rn(g, R.z));
    R.w = __fadd_rn(pc.w, __fmul_rn(g, R.w));
    __stcs(tgt + (size_t)t * per_t + idx, R);
  }
}

// The targets of a rollout pass (trainer.py:298-324 and :352-372) from the [T,N] frame records K1 wrote: rewards,
// terminals and both cells of every step are in the record, so the [T,N,20,20] pixel-change maps are evaluated in
// registers (pc_value4, bit-identical to K1's maps) instead of being read back.  A record whose valid bit is 0 counts
// as reward 0, not terminal, map 0 (what the per-step K1 writes for an inactive env).  Blocks [0, ret_blocks) hold
// one thread per env for R / adv (coalesced [T,N] loads); the rest one thread per (env, float4 q and q + 50 of the
// map) for the PC targets: half the threads of one per float4, so the grid fits in one wave of the SMs at 4096 envs
// (measured on B200 at 4096 x 20: 31 us instead of 37 with one float4 per thread).  Both recurrences run in the order
// and with the roundings of nstep_returns_kernel / pc_targets_kernel, so the results are bit-equal to those two kernels
// on the same pass.  Each chunk's loads are issued before its scan.
constexpr int kTgtThreads = 128;
constexpr int kTgtChunk = 10;     // R / adv steps loaded ahead of their scan
constexpr int kTgtPcChunk = 5;    // PC-target steps loaded ahead of theirs
constexpr int kTgtPcPer = 2;      // float4 of the map per thread
constexpr int kTgtPcCols = kPcElems / 4 / kTgtPcPer;

__device__ __forceinline__ uint64_t valid_record(uint64_t r) { return frame_valid(r) ? r : 0ull; }

__global__ void __launch_bounds__(kTgtThreads, 8) maze_rollout_targets_kernel(
    const uint64_t* __restrict__ rec, const float* __restrict__ values, const float* __restrict__ boot_value,
    const float4* __restrict__ boot_q, float gamma, float gamma_pc, float* __restrict__ out_R,
    float* __restrict__ out_adv, float4* __restrict__ tgt, int T, int N, int ret_blocks) {
  if ((int)blockIdx.x < ret_blocks) {
    const int n = blockIdx.x * kTgtThreads + threadIdx.x;
    if (n >= N) return;
    float R = boot_value[n];
    for (int hi = T; hi > 0; hi -= kTgtChunk) {
      const int lo = hi - kTgtChunk;
      int rr[kTgtChunk];        // the reward byte | terminal << 8
      float vv[kTgtChunk];
#pragma unroll
      for (int k = 0; k < kTgtChunk; ++k) {
        if (lo + k >= 0) {
          const size_t o = (size_t)(lo + k) * N + n;
          const uint64_t r = valid_record(__ldg(rec + o));
          rr[k] = (frame_reward(r) & 0xff) | (frame_terminal(r) << 8);
          vv[k] = __ldcs(values + o);
        }
      }
#pragma unroll
      for (int k = kTgtChunk - 1; k >= 0; --k) {
        if (lo + k >= 0) {
          const size_t o = (size_t)(lo + k) * N + n;
          R = (rr[k] & 0x100) ? 0.f : R;                                   // (:298-300)
          R = __fadd_rn((float)(int8_t)rr[k], __fmul_rn(gamma, R));       // R = ri + gamma * R   (:314)
          __stcs(out_R + o, R);
          __stcs(out_adv + o, __fsub_rn(R, vv[k]));                        // adv = R - Vi   (:315)
        }
      }
    }
    return;
  }
  const size_t per_t = (size_t)N * (kPcElems / 4);
  const size_t col = (size_t)(blockIdx.x - ret_blocks) * kTgtThreads + threadIdx.x;   // over N * kTgtPcCols
  if (col >= (size_t)N * kTgtPcCols) return;
  const int n = (int)(col / kTgtPcCols), q0 = (int)(col - (size_t)n * kTgtPcCols);
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 R[kTgtPcPer];
#pragma unroll
  for (int p = 0; p < kTgtPcPer; ++p) R[p] = boot_q[(size_t)n * (kPcElems / 4) + q0 + p * kTgtPcCols];
  for (int hi = T; hi > 0; hi -= kTgtPcChunk) {
    const int lo = hi - kTgtPcChunk;
    uint32_t cc[kTgtPcChunk];   // the record's two cells (its low 16 bits) | terminal << 16
#pragma unroll
    for (int k = 0; k < kTgtPcChunk; ++k) {
      if (lo + k >= 0) {
        const uint64_t r = valid_record(__ldg(rec + (size_t)(lo + k) * N + n));
        cc[k] = (uint32_t)(r & 0xffffu) | ((uint32_t)frame_terminal(r) << 16);
      }
    }
#pragma unroll
    for (int k = kTgtPcChunk - 1; k >= 0; --k) {
      if (lo + k >= 0) {
        const uint64_t r = cc[k];
#pragma unroll
        for (int p = 0; p < kTgtPcPer; ++p) {
          const int q = q0 + p * kTgtPcCols;
          const float4 pc = pc_value4(frame_x0(r), frame_y0(r), frame_x1(r), frame_y1(r), q);
          if (r >> 16) R[p] = zero;
          R[p].x = __fadd_rn(pc.x, __fmul_rn(gamma_pc, R[p].x));   // pc_R = pixel_change + gamma_pc * pc_R   (:361)
          R[p].y = __fadd_rn(pc.y, __fmul_rn(gamma_pc, R[p].y));
          R[p].z = __fadd_rn(pc.z, __fmul_rn(gamma_pc, R[p].z));
          R[p].w = __fadd_rn(pc.w, __fmul_rn(gamma_pc, R[p].w));
          __stcs(tgt + (size_t)(lo + k) * per_t + (size_t)n * (kPcElems / 4) + q, R[p]);
        }
      }
    }
  }
}

__global__ void maze_reset_kernel(int32_t* pos, int32_t* last_action, float* last_reward, const uint8_t* mask,
                                  int n) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n || (mask != nullptr && mask[e] == 0)) return;
  pos[2 * e] = c_maze.start_x;
  pos[2 * e + 1] = c_maze.start_y;
  if (last_action) last_action[e] = 0;
  if (last_reward) last_reward[e] = 0.f;
}

static int parse_map(const char* m, MazeLayout* out) {
  MazeLayout L;
  for (int y = 0; y < UNREAL_MAZE_GRID; ++y) L.wall_rows[y] = 0;
  L.start_x = L.start_y = L.goal_x = L.goal_y = -1;
  for (int i = 0; i < UNREAL_MAZE_GRID * UNREAL_MAZE_GRID; ++i) {
    char c = m[i];
    UNREAL_REQUIRE(c != 0, "maze map shorter than 49 characters");
    int x = i % UNREAL_MAZE_GRID, y = i / UNREAL_MAZE_GRID;
    if (c == '+') L.wall_rows[y] |= 1u << x;
    else if (c == 'S') { L.start_x = x; L.start_y = y; }
    else if (c == 'G') { L.goal_x = x; L.goal_y = y; }
  }
  UNREAL_REQUIRE(L.start_x >= 0, "maze map has no 'S' cell");
  *out = L;
  return UNREAL_OK;
}

// The map is process-wide and h_maze is its one copy on the host.  Each device holds its own c_maze, so a device gets
// h_maze uploaded the first time it needs the map and again after the map changed: h_maze_gen counts the maps set,
// g_dev_gen records the generation each device holds.  Uploads happen in the eager calls that precede a graph capture.
static std::mutex g_maze_mu;
static MazeLayout h_maze = [] {
  MazeLayout L;
  parse_map(kReferenceMap, &L);
  return L;
}();
static unsigned h_maze_gen = 1;
static std::map<int, unsigned> g_dev_gen;

static int upload_map_locked() {
  int dev = 0;
  UNREAL_CUDA(cudaGetDevice(&dev));
  unsigned& have = g_dev_gen[dev];
  if (have == h_maze_gen) return UNREAL_OK;
  UNREAL_CUDA(cudaMemcpyToSymbol(c_maze, &h_maze, sizeof(h_maze)));
  have = h_maze_gen;
  return UNREAL_OK;
}

// every entry point whose kernels read c_maze calls this first
static int ensure_map() {
  std::lock_guard<std::mutex> lk(g_maze_mu);
  return upload_map_locked();
}

template <bool kStep>
static int launch_render(const StepArgs& a, int obs_dtype, cudaStream_t st) {
  if (a.n == 0) return UNREAL_OK;
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  if (obs_dtype == UNREAL_BF16) {
    maze_s2d_kernel<kStep><<<a.n, 256, 0, st>>>(a);
    UNREAL_LAUNCH_CHECK("maze_s2d_kernel");
    return UNREAL_OK;
  }
  // defaults = fastest measured on B200 (profiles/microbench_r1.md): f32 -> CTA per env with
  // 256 threads (99% of measured HBM peak), u8 -> warp per env.
  int variant = get_tunable("maze_render_variant", -1);
  // no frame to write (cell observations / K1 as a pure stepper): one WARP per env -- a 256-thread CTA per env costs
  // 33 us per step at 8192 envs for 13 MB of pixel-change maps
  if (variant < 0) variant = (a.obs == nullptr || obs_dtype == UNREAL_U8) ? 2 : 0;
  if (a.obs == nullptr && variant == 1) variant = 0;  // nothing to stage through shared memory
  if (variant == 2) {
    const int warps = get_tunable("maze_warps_per_cta", 4);
    if (obs_dtype == UNREAL_F32) {
      maze_warp_kernel<float, kStep, 4><<<(a.n + 3) / 4, 128, 0, st>>>(a);
    } else if (warps == 16) {
      maze_warp_kernel<uint8_t, kStep, 16><<<(a.n + 15) / 16, 512, 0, st>>>(a);
    } else if (warps == 8) {
      maze_warp_kernel<uint8_t, kStep, 8><<<(a.n + 7) / 8, 256, 0, st>>>(a);
    } else if (warps == 2) {
      maze_warp_kernel<uint8_t, kStep, 2><<<(a.n + 1) / 2, 64, 0, st>>>(a);
    } else {
      maze_warp_kernel<uint8_t, kStep, 4><<<(a.n + 3) / 4, 128, 0, st>>>(a);
    }
    UNREAL_LAUNCH_CHECK("maze_warp_kernel");
    return UNREAL_OK;
  }
  if (variant == 0) {
    if (obs_dtype == UNREAL_F32) {
      if (get_tunable("maze_cta_threads", 256) == 512) maze_cta_kernel<float, kStep, 512><<<a.n, 512, 0, st>>>(a);
      else maze_cta_kernel<float, kStep, 256><<<a.n, 256, 0, st>>>(a);
    } else {
      if (get_tunable("maze_cta_threads", 256) == 512) maze_cta_kernel<uint8_t, kStep, 512><<<a.n, 512, 0, st>>>(a);
      else maze_cta_kernel<uint8_t, kStep, 256><<<a.n, 256, 0, st>>>(a);
    }
    UNREAL_LAUNCH_CHECK("maze_cta_kernel");
    return UNREAL_OK;
  }
  if (obs_dtype == UNREAL_F32) {
    constexpr int kBufs = 2;
    size_t smem = (size_t)kBufs * kFrameElems * sizeof(float);
    auto k = maze_tma_kernel<float, kBufs, kStep>;
    const int rc = allow_dynamic_smem((const void*)k, (int)smem);
    if (rc != UNREAL_OK) return rc;
    int grid = a.n < sms ? a.n : sms;
    k<<<grid, kThreads, smem, st>>>(a);
    UNREAL_LAUNCH_CHECK("maze_tma_kernel<f32>");
  } else {
    constexpr int kBufs = 4;
    size_t smem = (size_t)kBufs * kFrameElems * sizeof(uint8_t);
    auto k = maze_tma_kernel<uint8_t, kBufs, kStep>;
    const int rc = allow_dynamic_smem((const void*)k, (int)smem);
    if (rc != UNREAL_OK) return rc;
    int per_sm = get_tunable("maze_u8_ctas_per_sm", 2);
    int grid = a.n < sms * per_sm ? a.n : sms * per_sm;
    k<<<grid, kThreads, smem, st>>>(a);
    UNREAL_LAUNCH_CHECK("maze_tma_kernel<u8>");
  }
  return UNREAL_OK;
}

}  // namespace unreal

using namespace unreal;

extern "C" int unreal_maze_set_map(const char* map49_host) {
  MazeLayout L;
  int rc = parse_map(map49_host ? map49_host : kReferenceMap, &L);
  if (rc != UNREAL_OK) return rc;
  std::lock_guard<std::mutex> lk(g_maze_mu);
  h_maze = L;
  ++h_maze_gen;
  return upload_map_locked();
}

namespace unreal {
MazeLayout maze_layout_host() {
  std::lock_guard<std::mutex> lk(g_maze_mu);
  return h_maze;
}

uint64_t maze_walls49() {
  const MazeLayout L = maze_layout_host();
  uint64_t w = 0;
  for (int cy = 0; cy < UNREAL_MAZE_GRID; ++cy) w |= (uint64_t)(L.wall_rows[cy] & 0x7fu) << (7 * cy);
  return w;
}
}  // namespace unreal

extern "C" int unreal_maze_get_layout(int* sx, int* sy, int* gx, int* gy, uint8_t* walls49_host) {
  int rc = ensure_map();
  if (rc) return rc;
  const MazeLayout L = maze_layout_host();
  if (sx) *sx = L.start_x;
  if (sy) *sy = L.start_y;
  if (gx) *gx = L.goal_x;
  if (gy) *gy = L.goal_y;
  if (walls49_host)
    for (int i = 0; i < 49; ++i) walls49_host[i] = (L.wall_rows[i / 7] >> (i % 7)) & 1u;
  return UNREAL_OK;
}

extern "C" int unreal_maze_reset(int32_t* pos, int32_t* last_action, float* last_reward, const uint8_t* mask,
                                 int n, void* stream) {
  UNREAL_REQUIRE(pos != nullptr && n >= 0, "unreal_maze_reset: pos is null or n < 0");
  int rc = ensure_map();
  if (rc) return rc;
  if (n == 0) return UNREAL_OK;
  maze_reset_kernel<<<(n + 255) / 256, 256, 0, as_stream(stream)>>>(pos, last_action, last_reward, mask, n);
  UNREAL_LAUNCH_CHECK("maze_reset_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_maze_step(int32_t* pos, const int32_t* action, const uint8_t* active, float* reward,
                                uint8_t* terminal, int32_t* last_action, float* last_reward, void* obs,
                                int obs_dtype, float* pc, uint64_t* frame_rec, int n, int auto_reset,
                                void* stream) {
  UNREAL_REQUIRE(n >= 0, "unreal_maze_step: n < 0");
  UNREAL_REQUIRE(pos && action && reward && terminal && last_action && last_reward,
                 "unreal_maze_step: pos/action/reward/terminal/last_action/last_reward must be non-null");
  UNREAL_REQUIRE(obs_dtype == UNREAL_F32 || obs_dtype == UNREAL_U8 || obs_dtype == UNREAL_BF16,
                 "unreal_maze_step: bad obs_dtype %d", obs_dtype);
  UNREAL_REQUIRE(aligned16(obs) && aligned16(pc), "unreal_maze_step: obs and pc must be 16-byte aligned");
  int rc = ensure_map();
  if (rc) return rc;
  StepArgs a{pos, action, active, reward, terminal, last_action, last_reward, obs, pc, frame_rec, n, auto_reset};
  return launch_render<true>(a, obs_dtype, as_stream(stream));
}

extern "C" int unreal_maze_render(const int32_t* pos, void* obs, int obs_dtype, int m, void* stream) {
  UNREAL_REQUIRE(pos && obs && m >= 0, "unreal_maze_render: null argument or m < 0");
  UNREAL_REQUIRE(obs_dtype == UNREAL_F32 || obs_dtype == UNREAL_U8 || obs_dtype == UNREAL_BF16,
                 "unreal_maze_render: bad obs_dtype %d", obs_dtype);
  UNREAL_REQUIRE(aligned16(obs), "unreal_maze_render: obs must be 16-byte aligned");
  int rc = ensure_map();
  if (rc) return rc;
  StepArgs a{const_cast<int32_t*>(pos), nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, obs, nullptr, nullptr, m, 0};
  return launch_render<false>(a, obs_dtype, as_stream(stream));
}

extern "C" int unreal_maze_pixel_change(const int32_t* pos0, const int32_t* pos1, float* pc, int m, void* stream) {
  UNREAL_REQUIRE(pos0 && pos1 && pc && m >= 0, "unreal_maze_pixel_change: null argument or m < 0");
  UNREAL_REQUIRE(aligned16(pc), "unreal_maze_pixel_change: pc must be 16-byte aligned");
  if (m == 0) return UNREAL_OK;
  long long threads = (long long)m * (kPcElems / 4);
  maze_pc_pairs_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, as_stream(stream)>>>(pos0, pos1, pc, m);
  UNREAL_LAUNCH_CHECK("maze_pc_pairs_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_maze_pc_targets(const int32_t* pos0, const int32_t* pos1, const int32_t* len, const float* boot,
                                      float gamma_pc, float* tgt, int t, int n, void* stream) {
  UNREAL_REQUIRE(t >= 0 && n >= 0, "unreal_maze_pc_targets: negative size");
  if (t == 0 || n == 0) return UNREAL_OK;
  UNREAL_REQUIRE(pos0 && pos1 && boot && tgt, "unreal_maze_pc_targets: pos0, pos1, boot and tgt must be non-null");
  UNREAL_REQUIRE(aligned16(boot) && aligned16(tgt) && (reinterpret_cast<uintptr_t>(pos0) & 7u) == 0 &&
                 (reinterpret_cast<uintptr_t>(pos1) & 7u) == 0, "unreal_maze_pc_targets: alignment (16 bytes; cells 8)");
  const long long cols = (long long)n * (kPcElems / 4);
  maze_pc_targets_kernel<<<(unsigned)((cols + 127) / 128), 128, 0, as_stream(stream)>>>(
      reinterpret_cast<const int2*>(pos0), reinterpret_cast<const int2*>(pos1), len, reinterpret_cast<const float4*>(boot),
      gamma_pc, reinterpret_cast<float4*>(tgt), t, n);
  UNREAL_LAUNCH_CHECK("maze_pc_targets_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_maze_rollout_targets(const uint64_t* rec, const float* values, const float* boot_value,
                                           const float* boot_q, float gamma, float gamma_pc, float* out_R, float* out_adv,
                                           float* pc_tgt, int t, int n, void* stream) {
  UNREAL_REQUIRE(t >= 0 && n >= 0, "unreal_maze_rollout_targets: negative size");
  if (t == 0 || n == 0) return UNREAL_OK;
  UNREAL_REQUIRE(rec && values && boot_value && boot_q && out_R && out_adv && pc_tgt,
                 "unreal_maze_rollout_targets: null argument");
  UNREAL_REQUIRE(aligned16(boot_q) && aligned16(pc_tgt) && (reinterpret_cast<uintptr_t>(rec) & 7u) == 0,
                 "unreal_maze_rollout_targets: alignment (boot_q / pc_tgt 16 bytes; rec 8)");
  const long long cols = (long long)n * kTgtPcCols;
  const int ret_blocks = (n + kTgtThreads - 1) / kTgtThreads;
  const long long blocks = ret_blocks + (cols + kTgtThreads - 1) / kTgtThreads;
  maze_rollout_targets_kernel<<<(unsigned)blocks, kTgtThreads, 0, as_stream(stream)>>>(
      rec, values, boot_value, reinterpret_cast<const float4*>(boot_q), gamma, gamma_pc, out_R, out_adv,
      reinterpret_cast<float4*>(pc_tgt), t, n, ret_blocks);
  UNREAL_LAUNCH_CHECK("maze_rollout_targets_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_maze_window(int32_t* pos, const int32_t* action, float* reward, uint8_t* terminal, int32_t* last_action,
                                  float* last_reward, void* obs, int obs_dtype, float* pc, uint64_t* frame_rec, int n, int t,
                                  int auto_reset, void* stream) {
  UNREAL_REQUIRE(n >= 0 && t >= 0, "unreal_maze_window: negative size");
  UNREAL_REQUIRE(t <= 32, "unreal_maze_window: at most 32 steps per window (got %d)", t);
  UNREAL_REQUIRE(pos && action && reward && terminal && last_action && last_reward,
                 "unreal_maze_window: pos/action/reward/terminal/last_action/last_reward must be non-null");
  UNREAL_REQUIRE(obs_dtype == UNREAL_F32 || obs_dtype == UNREAL_U8, "unreal_maze_window: obs_dtype must be f32 or u8");
  UNREAL_REQUIRE(aligned16(obs) && aligned16(pc), "unreal_maze_window: obs and pc must be 16-byte aligned");
  UNREAL_REQUIRE((long long)n * t < 2147483647LL / 4, "unreal_maze_window: window too large for one launch");
  int rc = ensure_map();
  if (rc) return rc;
  if (n == 0 || t == 0) return UNREAL_OK;
  cudaStream_t st = as_stream(stream);
  WindowArgs a{pos, last_action, last_reward, action, reward, terminal, obs, pc, frame_rec, n, t, auto_reset};
  const long long items = (long long)n * t;
  int variant = get_tunable("maze_render_variant", -1);
  // u8 frames: one warp per env walking its T steps (variant 3); f32 frames: one CTA per (step, env) item (variant 0)
  if (variant < 0 || variant == 1) variant = (obs == nullptr || obs_dtype == UNREAL_U8) ? 3 : 0;
  if (variant == 3) {
    const int warps = get_tunable("maze_warps_per_cta", 8);
    if (obs_dtype == UNREAL_F32) maze_window_env_kernel<float, 4><<<(n + 3) / 4, 128, 0, st>>>(a, pos, last_action, last_reward);
    else if (warps == 4) maze_window_env_kernel<uint8_t, 4><<<(n + 3) / 4, 128, 0, st>>>(a, pos, last_action, last_reward);
    else if (warps == 2) maze_window_env_kernel<uint8_t, 2><<<(n + 1) / 2, 64, 0, st>>>(a, pos, last_action, last_reward);
    else if (warps == 1) maze_window_env_kernel<uint8_t, 1><<<n, 32, 0, st>>>(a, pos, last_action, last_reward);
    else maze_window_env_kernel<uint8_t, 8><<<(n + 7) / 8, 256, 0, st>>>(a, pos, last_action, last_reward);
    UNREAL_LAUNCH_CHECK("maze_window_env_kernel");
    return UNREAL_OK;                       // the env kernel advances the state itself
  }
  if (variant == 2) {
    if (obs_dtype == UNREAL_F32) maze_window_warp_kernel<float, 4><<<(unsigned)((items + 3) / 4), 128, 0, st>>>(a);
    else if (get_tunable("maze_warps_per_cta", 4) == 8) maze_window_warp_kernel<uint8_t, 8><<<(unsigned)((items + 7) / 8), 256, 0, st>>>(a);
    else maze_window_warp_kernel<uint8_t, 4><<<(unsigned)((items + 3) / 4), 128, 0, st>>>(a);
    UNREAL_LAUNCH_CHECK("maze_window_warp_kernel");
  } else {
    if (obs_dtype == UNREAL_F32) maze_window_cta_kernel<float, 256><<<(unsigned)items, 256, 0, st>>>(a);
    else maze_window_cta_kernel<uint8_t, 256><<<(unsigned)items, 256, 0, st>>>(a);
    UNREAL_LAUNCH_CHECK("maze_window_cta_kernel");
  }
  maze_window_state_kernel<<<(n + 127) / 128, 128, 0, st>>>(pos, last_action, last_reward, action, n, t, auto_reset);
  UNREAL_LAUNCH_CHECK("maze_window_state_kernel");
  return UNREAL_OK;
}
