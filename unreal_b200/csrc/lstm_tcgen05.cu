// K7 LSTM steps with the BasicLSTMCell arithmetic in the GEMM epilogue (model/model.py:110, :343-351 -- dynamic_rnn over
// BasicLSTMCell(256): gates = [x, h] W + b split into i | j | f | o, c' = c sigma(f + 1) + sigma(i) tanh(j),
// h' = tanh(c') sigma(o)).
//
// The separate-kernel form (gemm_tcgen05_kernel + lstm_cell_fwd8_kernel) wrote the [N,1024] gate pre-activations to HBM
// and read them back once per step, and its epilogue (one warp per 32 rows x 256 columns) was what paced the step GEMM
// (ncu, profiles/r2_lstm_step_8192envs_ncu_summary.txt: 18.1 us with the tensor pipe 34 % busy, nothing else above
// 26 %; cell kernel 19.2 us).  Here one tile holds ALL FOUR gates of 64 units -- the B operand of a tile is four
// 64-column boxes of W taken 256 columns apart (no permuted weight copy) -- so the cell is computed on the accumulator
// as it leaves TMEM, by SIXTEEN cell warps (four per TMEM lane quarter, 16 units each), and the only things written are what
// the next step and the backward pass read: c', h', h' as bf16 straight into the next step's operand, the gate activations
// as bf16.
//
//   forward   unreal_lstm_step_fwd:  acc[128 rows, (gate, 64 units)] = xh_t[rows, :] W[:, gate*256 + units]
//   backward  unreal_lstm_step_bwd:  acc[128 rows, BN units]          = dgates_{t+1}[rows, :] Wh[units, :]^T  (= dh_rec)
//             epilogue: the cell's backward pass of step t on dh_t + dh_rec -> dgates_t (bf16), dc in place.
//
// Warp roles: 0 = TMA producer, 1 = MMA issuer (one thread), 2..17 = cell warps.  Two TMEM accumulators, so the cell
// arithmetic of tile i overlaps the MMAs of tile i+1.  The cell arithmetic is what the kernels are made of (ncu,
// profiles/r2_lstm_fused_8192envs_ncu_summary.txt: the cell's backward pass alone, without the product, took 23 us with
// eight cell warps -- a chain of load, wait, compute, store per warp with nothing to overlap it), hence four warps per
// scheduler working on 8-unit chunks, and branch-free activations so that a lane's 8 units interleave.
//
// Memory access of the cell warps.  An accumulator row lives in one TMEM lane, so a lane owns one env row, and with
// row-major [n,256] / [n,1024] buffers every 16-byte access of a warp touches 32 different 128-byte lines: the L1 tag
// stage (one line per cycle) paced the first build of these kernels (36 us per step at 8192 envs against 31 us for the
// two-kernel path; profiles/r2_lstm_step_bench.jsonl).  Two remedies, both used by the unroll ("tiled" mode):
//   * buffers only these kernels touch (c of every step, the gate activations, the running dc) are kept in the layout
//     the cell warps access them in -- see tiled_off();
//   * buffers with other readers (h f32 for the heads, h bf16 in the next step's operand, dh from the heads, dgates for
//     the next product and the filter gradient) go through per-warp swizzled shared-memory tiles and the TMA engine.
// The row-major mode (direct 16-byte accesses) remains for the acting step, which updates the persistent state in place
// under an `active` mask.
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "tc05.cuh"

namespace unreal {
using namespace tc05;

namespace {

constexpr int kLsCellWarps = 16;
constexpr int kLsThreads = 32 * (2 + kLsCellWarps);
constexpr int kLsBM = 128, kLsBK = 64;
constexpr uint32_t kLsDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);   // SBO 1024 B, version 1, 128-byte swizzle

// Branch-free activations.  What hides latency in a cell warp is instruction-level parallelism over a lane's 8 units --
// which tanhf (a branch between its polynomial and exponential ranges) and the IEEE division (a branch to its
// special-case path) prevent: with them the first build measured ~700 cycles per unit.
//   sigmoid: MUFU.EX2 + MUFU.RCP, <= 3 ulp.
//   tanh:    |x| <  0.2: x - x^3/3 + 2x^5/15 - 17x^7/315 (next term < 6e-8 relative)
//            |x| >= 0.2: 1 - 2 / (exp(2x) + 1), absolute error ~1e-7 = <= 5e-7 relative there; +-1 at the overflow ends.
__device__ __forceinline__ float sigmoid_(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float tanh_(float x) {
  const float x2 = x * x;
  const float p = fmaf(x * x2, fmaf(x2, fmaf(x2, -17.0f / 315.0f, 2.0f / 15.0f), -1.0f / 3.0f), x);
  const float r = 1.0f - __fdividef(2.0f, __expf(2.0f * x) + 1.0f);
  return fabsf(x) < 0.2f ? p : r;
}

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&p);
}
__device__ __forceinline__ uint4 pack8(const float (&v)[8]) {
  return make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
}
__device__ __forceinline__ void unpack8(const uint4 u, float (&v)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int j = 0; j < 4; ++j) { const float2 f = __bfloat1622float2(h[j]); v[2 * j] = f.x; v[2 * j + 1] = f.y; }
}
// 8 consecutive units of one row: two 16-byte f32 chunks `step` floats apart (4 = a row-major row), or one bf16 chunk
__device__ __forceinline__ void ld8f(const float* p, float (&v)[8], int step) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + step);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void st8f(float* p, const float (&v)[8], int step) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + step) = make_float4(v[4], v[5], v[6], v[7]);
}

// "Tiled" buffers: blocks of 32 rows; inside a block the 16-byte chunks of a row lie 512 bytes apart and the 32 rows of
// a chunk are consecutive:
//     chunk (row, ch) at 16 bytes * ((row / 32 * chunks_per_row + ch) * 32 + row % 32)
// so one warp access (lane = row % 32) is 512 contiguous bytes.  Rows are padded to a multiple of 32.
__device__ __forceinline__ size_t tiled_off(int row_block, int chunks_per_row, int chunk, int lane) {
  return ((size_t)(row_block * chunks_per_row + chunk) * 32 + lane);        // in 16-byte chunks
}

// Staging tiles of one cell warp (its 32 rows x 16 units), lane = row.  f32: [32 rows x 64 B] with the 64-byte swizzle
// (16-byte chunk j of row r at chunk j ^ ((r >> 1) & 3)); bf16: [32 rows x 32 B] with the 32-byte swizzle (chunk j at
// j ^ ((r >> 2) & 1)).  Both are what a TMA box {16 columns, 32 rows} of that swizzle mode reads / writes, and both are
// bank-conflict free for lane = row.  `ch` = which 8-unit half of the warp's 16 units.
__device__ __forceinline__ void stage8f(uint32_t tile, int lane, int ch, const float (&v)[8]) {
  const uint32_t rowp = tile + (uint32_t)lane * 64u, sw = (uint32_t)((lane >> 1) & 3);
  st_shared_v4(rowp + (((uint32_t)(2 * ch)) ^ sw) * 16u, __float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3]));
  st_shared_v4(rowp + (((uint32_t)(2 * ch + 1)) ^ sw) * 16u, __float_as_uint(v[4]), __float_as_uint(v[5]), __float_as_uint(v[6]), __float_as_uint(v[7]));
}
__device__ __forceinline__ void unstage8f(uint32_t tile, int lane, int ch, float (&v)[8]) {
  const uint32_t rowp = tile + (uint32_t)lane * 64u, sw = (uint32_t)((lane >> 1) & 3);
  const float4 a = lds_v4(rowp + (((uint32_t)(2 * ch)) ^ sw) * 16u), b = lds_v4(rowp + (((uint32_t)(2 * ch + 1)) ^ sw) * 16u);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void stage8h(uint32_t tile, int lane, int ch, const float (&v)[8]) {
  const uint4 p = pack8(v);
  st_shared_v4(tile + (uint32_t)lane * 32u + (((uint32_t)ch) ^ (uint32_t)((lane >> 2) & 1)) * 16u, p.x, p.y, p.z, p.w);
}

struct LstmFwdArgs {
  const float* bias;        // [1024]
  const float* c_prev;      // [n,256]
  float* c_out;             // [n,256] (may alias c_prev: the acting step updates the persistent state in place)
  float* h_out;             // [n,256] f32 or null
  float* h_copy;            // [n,256] f32 or null: h of every row -- the new one, or (inactive rows) what h_out holds
  __nv_bfloat16* h16_out;   // bf16 h, rows h16_ld apart (the next step's operand columns), or null
  __nv_bfloat16* acts;      // [n,1024] gate activations for the backward pass, or null
  const uint8_t* active;    // [n] or null: rows with 0 keep their state
  int n, k, h16_ld;
  int tiled;                // c_prev, c_out and acts are tiled; h_out / h16_out leave through the TMA engine
};

constexpr int kFwdBN = 256;
constexpr int kFwdStages = 3;
constexpr int kFwdStageBytes = kLsBM * kLsBK * 2 + kFwdBN * kLsBK * 2;     // 16 KB of xh + 32 KB of W
constexpr int kFwdStagingBytes = kLsCellWarps * (2048 + 1024);             // per cell warp: h f32 tile + h bf16 tile
constexpr int kFwdSmem = kFwdStages * kFwdStageBytes + 1024 /*barriers*/ + 4096 /*bias*/ + kFwdStagingBytes + 1024 /*alignment*/;

__global__ void __launch_bounds__(kLsThreads, 1)
lstm_step_fwd_tcgen05_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                             const __grid_constant__ CUtensorMap tma_h, const __grid_constant__ CUtensorMap tma_h16,
                             const LstmFwdArgs g) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + kFwdStages * kFwdStageBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kFwdStages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * kFwdStages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * kFwdStages + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * kFwdStages + 4);
  float* s_bias = reinterpret_cast<float*>(smem_raw + (bar_base + 1024u - smem_u32(smem_raw)));
  const uint32_t stg_base = bar_base + 1024u + 4096u;      // 1024-byte aligned

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_m = (g.n + kLsBM - 1) / kLsBM;
  const int kb_total = (g.k + kLsBK - 1) / kLsBK;
  const int work_total = num_m * 4;             // (row block, block of 64 units)

  for (int i = threadIdx.x; i < 1024; i += kLsThreads) s_bias[i] = g.bias[i];
  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tma_a);
    prefetch_tensormap(&tma_b);
    if (g.tiled) { prefetch_tensormap(&tma_h); prefetch_tensormap(&tma_h16); }
    for (int s = 0; s < kFwdStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), kLsCellWarps); }
    fence_mbar_init();
  } else if (warp == 2) {
    tmem_alloc<512>(tmem_slot);
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = tmem_base_at(tmem_slot);

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int w = blockIdx.x; w < work_total; w += gridDim.x) {
        const int ub = w & 3, m_blk = w >> 2;
        for (int kb = 0; kb < kb_total; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sa = smem_base + stage * kFwdStageBytes, sb = sa + kLsBM * kLsBK * 2;
          mbar_arrive_expect_tx(full_bar(stage), kFwdStageBytes);
          tma_load_2d(sa, &tma_a, full_bar(stage), kb * kLsBK, m_blk * kLsBM);
#pragma unroll
          for (int gate = 0; gate < 4; ++gate)       // accumulator columns [64 gate, 64 gate + 64) = units ub*64.. of that gate
            tma_load_2d(sb + gate * (kLsBK * 128), &tma_b, full_bar(stage), gate * 256 + ub * 64, kb * kLsBK);
          if (++stage == kFwdStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = idesc_bf16_f32(kLsBM, kFwdBN, false, true);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int w = blockIdx.x; w < work_total; w += gridDim.x) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        fence_after_sync();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * kFwdBN);
        for (int kb = 0; kb < kb_total; ++kb) {
          mbar_wait(full_bar(stage), phase);
          fence_after_sync();
          const uint32_t sa = smem_base + stage * kFwdStageBytes, sb = sa + kLsBM * kLsBK * 2;
          const uint32_t a_lo = (sa >> 4) | (1u << 16);
          const uint32_t b_lo = (sb >> 4) | (((uint32_t)(kLsBK * 128) >> 4) << 16);
          // the last block of K = 520 holds 8 columns: one UMMA instead of four over zero fill
          const int kk = min(kLsBK / 16, (g.k - kb * kLsBK + 15) >> 4);
#pragma unroll
          for (int k = 0; k < kLsBK / 16; ++k)
            if (k < kk)
              mma_f16_lohi(tmem_d, a_lo + (uint32_t)k * 2u, kLsDescHi, b_lo + (uint32_t)k * 128u, kLsDescHi, idesc,
                           (kb > 0 || k > 0) ? 1u : 0u);
          mma_commit(empty_bar(stage));
          if (++stage == kFwdStages) { stage = 0; phase ^= 1u; }
        }
        mma_commit(tfull_bar(acc));
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else {
    // ===== cell warps: warp w owns TMEM lanes 32 (w % 4) .. +31; the four warps of a quarter take 16 units each =====
    const int quarter = warp & 3, part = (warp - 2) >> 2;
    const uint32_t s_h = stg_base + (uint32_t)(warp - 2) * 2048u;
    const uint32_t s_h16 = stg_base + (uint32_t)kLsCellWarps * 2048u + (uint32_t)(warp - 2) * 1024u;
    const bool out_h = g.tiled && g.h_out != nullptr, out_h16 = g.tiled && g.h16_out != nullptr;
    const int cstep = g.tiled ? 128 : 4;
    int acc = 0; uint32_t acc_phase = 0;
    for (int w = blockIdx.x; w < work_total; w += gridDim.x) {
      const int ub = w & 3, m_blk = w >> 2;
      const int row0 = m_blk * kLsBM + quarter * 32;
      const int row = row0 + lane;
      const bool row_ok = row < g.n;
      const bool on = row_ok && (g.active == nullptr || g.active[row] != 0);
      const int u0 = ub * 64 + part * 16;                    // this warp's 16 units
      // c_{t-1} of both chunks does not depend on the product: in flight while the MMAs run
      float c[2][8];
#pragma unroll
      for (int ch = 0; ch < 2; ++ch) {
        const int u = u0 + ch * 8;
        if (on) ld8f(g.c_prev + (g.tiled ? tiled_off(m_blk * 4 + quarter, 64, u >> 2, lane) * 4 : (size_t)row * 256 + u), c[ch], cstep);
      }
      if (g.tiled) {                         // the staging tiles are free once the previous tile's stores have read them
        if (lane == 0) bulk_wait_read<0>();
        __syncwarp();
      }
      mbar_wait(tfull_bar(acc), acc_phase);
      fence_after_sync();
      const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * kFwdBN + part * 16);
#pragma unroll
      for (int ch = 0; ch < 2; ++ch) {
        const int u = u0 + ch * 8;
        const size_t so = (size_t)row * 256 + u;
        float zi[8], zj[8], zf[8], zo[8], h[8];
        tmem_ld8(trow + (uint32_t)(ch * 8), zi);
        tmem_ld8(trow + (uint32_t)(64 + ch * 8), zj);
        tmem_ld8(trow + (uint32_t)(128 + ch * 8), zf);
        tmem_ld8(trow + (uint32_t)(192 + ch * 8), zo);
        tmem_ld_wait();
        if (on) {
#pragma unroll
          for (int q4 = 0; q4 < 2; ++q4) {
            const float4 b4i = *reinterpret_cast<const float4*>(s_bias + u + 4 * q4);
            const float4 b4j = *reinterpret_cast<const float4*>(s_bias + 256 + u + 4 * q4);
            const float4 b4f = *reinterpret_cast<const float4*>(s_bias + 512 + u + 4 * q4);
            const float4 b4o = *reinterpret_cast<const float4*>(s_bias + 768 + u + 4 * q4);
            const float bi[4] = {b4i.x, b4i.y, b4i.z, b4i.w}, bj[4] = {b4j.x, b4j.y, b4j.z, b4j.w};
            const float bf[4] = {b4f.x, b4f.y, b4f.z, b4f.w}, bo[4] = {b4o.x, b4o.y, b4o.z, b4o.w};
#pragma unroll
            for (int r = 0; r < 4; ++r) {
              const int q = 4 * q4 + r;
              const float i = sigmoid_(zi[q] + bi[r]);
              const float j = tanh_(zj[q] + bj[r]);
              const float f = sigmoid_(zf[q] + bf[r] + 1.0f);   // forget_bias = 1.0
              const float o = sigmoid_(zo[q] + bo[r]);
              zi[q] = i; zj[q] = j; zf[q] = f; zo[q] = o;
              c[ch][q] = c[ch][q] * f + i * j;
              h[q] = tanh_(c[ch][q]) * o;
            }
          }
          st8f(g.c_out + (g.tiled ? tiled_off(m_blk * 4 + quarter, 64, u >> 2, lane) * 4 : so), c[ch], cstep);
          if (g.acts != nullptr) {
            // gate blocks 256 columns apart: 32 chunks of 8 bf16
            __nv_bfloat16* ar = g.acts + (g.tiled ? tiled_off(m_blk * 4 + quarter, 128, u >> 3, lane) * 8 : (size_t)row * 1024 + u);
            const int gstep = g.tiled ? 32 * 256 : 256;
            *reinterpret_cast<uint4*>(ar) = pack8(zi); *reinterpret_cast<uint4*>(ar + gstep) = pack8(zj);
            *reinterpret_cast<uint4*>(ar + 2 * gstep) = pack8(zf); *reinterpret_cast<uint4*>(ar + 3 * gstep) = pack8(zo);
          }
          if (!g.tiled) {
            if (g.h_out != nullptr) st8f(g.h_out + so, h, 4);
            if (g.h_copy != nullptr) st8f(g.h_copy + so, h, 4);
            if (g.h16_out != nullptr) *reinterpret_cast<uint4*>(g.h16_out + (size_t)row * g.h16_ld + u) = pack8(h);
          }
        } else if (!g.tiled && row_ok && g.h_copy != nullptr && g.h_out != nullptr) {
          ld8f(g.h_out + so, h, 4);
          st8f(g.h_copy + so, h, 4);
        }
        if (out_h) stage8f(s_h, lane, ch, h);            // rows >= n: garbage the TMA store clips
        if (out_h16) stage8h(s_h16, lane, ch, h);
      }
      fence_before_sync();
      if (g.tiled) fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(tempty_bar(acc));
        if (out_h) tma_store_2d(&tma_h, s_h, u0, row0);
        if (out_h16) tma_store_2d(&tma_h16, s_h16, u0, row0);
        if (g.tiled) bulk_commit();
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
    if (g.tiled && lane == 0) bulk_wait_all();
  }
  __syncwarp();
  fence_before_sync();
  __syncthreads();
  if (warp == 2) {
    fence_after_sync();
    tmem_dealloc<512>(tmem_base);
  }
}

struct LstmBwdArgs {
  const __nv_bfloat16* acts;   // [n,1024] gate activations of step t (i | j | f | o)
  const float* c_prev;         // [n,256] c_{t-1}
  const float* c;              // [n,256] c_t
  const float* dh;             // [n,256] gradient wrt h_t from the heads
  float* dc;                   // [n,256] in: gradient wrt c_t from step t+1, out: wrt c_{t-1}
  __nv_bfloat16* dgates;       // [n,1024] out: gradient wrt step t's pre-activations (row-major: the next GEMM's operand)
  const float* dh2;            // skip_gemm: optional second gradient wrt h_t [n,256] (the unroll's dh_last)
  int n;
  int tiled;                   // acts, c_prev, c and dc are tiled; dh arrives and dgates leaves through the TMA engine
  int skip_gemm;               // last step of the unroll: no recurrent gradient, the accumulator is not read
};

// 64 units per tile: acc[128 rows, 64] = dgates_{t+1}[rows, 0..1024) Wh[units, 0..1024)^T.  (128-unit tiles measured
// slower at every batch size: fewer, longer tiles with nothing to overlap the cell warps' work with.)
constexpr int kBwdBN = 64;
constexpr int kBwdStages = 5;
constexpr int kBwdStageBytes = kLsBM * kLsBK * 2 + kBwdBN * kLsBK * 2;      // 16 KB of dgates + 8 KB of Wh
constexpr int kBwdStagingBytes = kLsCellWarps * (2048 + 4 * 1024);          // per cell warp: dh f32 tile + four dgates bf16 tiles
constexpr int kBwdSmem = kBwdStages * kBwdStageBytes + 1024 + kBwdStagingBytes + 1024;

__global__ void __launch_bounds__(kLsThreads, 1)
lstm_step_bwd_tcgen05_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                             const __grid_constant__ CUtensorMap tma_dh, const __grid_constant__ CUtensorMap tma_dg,
                             const LstmBwdArgs g) {
  constexpr int BN = kBwdBN;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + kBwdStages * kBwdStageBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kBwdStages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * kBwdStages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * kBwdStages + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * kBwdStages + 4);
  auto dh_bar = [&](int e) { return bar_base + 8u * (2 * kBwdStages + 5 + e); };
  const uint32_t stg_base = bar_base + 1024u;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_m = (g.n + kLsBM - 1) / kLsBM;
  constexpr int kNumN = 256 / BN;
  constexpr int kKb = 1024 / kLsBK;
  const int work_total = num_m * kNumN;

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tma_a);
    prefetch_tensormap(&tma_b);
    if (g.tiled) { prefetch_tensormap(&tma_dh); prefetch_tensormap(&tma_dg); }
    for (int s = 0; s < kBwdStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), kLsCellWarps); }
    for (int e = 0; e < kLsCellWarps; ++e) mbar_init(dh_bar(e), 1);
    fence_mbar_init();
  } else if (warp == 2) {
    tmem_alloc<2 * BN>(tmem_slot);
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = tmem_base_at(tmem_slot);

  if (warp == 0) {
    if (lane == 0 && !g.skip_gemm) {
      int stage = 0; uint32_t phase = 0;
      for (int w = blockIdx.x; w < work_total; w += gridDim.x) {
        const int n_blk = w % kNumN, m_blk = w / kNumN;
        for (int kb = 0; kb < kKb; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sa = smem_base + stage * kBwdStageBytes, sb = sa + kLsBM * kLsBK * 2;
          mbar_arrive_expect_tx(full_bar(stage), kBwdStageBytes);
          tma_load_2d(sa, &tma_a, full_bar(stage), kb * kLsBK, m_blk * kLsBM);
          tma_load_2d(sb, &tma_b, full_bar(stage), kb * kLsBK, n_blk * BN);
          if (++stage == kBwdStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && !g.skip_gemm) {
      constexpr uint32_t idesc = idesc_bf16_f32(kLsBM, BN, false, false);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int w = blockIdx.x; w < work_total; w += gridDim.x) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        fence_after_sync();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
        for (int kb = 0; kb < kKb; ++kb) {
          mbar_wait(full_bar(stage), phase);
          fence_after_sync();
          const uint32_t sa = smem_base + stage * kBwdStageBytes, sb = sa + kLsBM * kLsBK * 2;
          const uint32_t a_lo = (sa >> 4) | (1u << 16), b_lo = (sb >> 4) | (1u << 16);
#pragma unroll
          for (int k = 0; k < kLsBK / 16; ++k)
            mma_f16_lohi(tmem_d, a_lo + (uint32_t)k * 2u, kLsDescHi, b_lo + (uint32_t)k * 2u, kLsDescHi, idesc,
                         (kb > 0 || k > 0) ? 1u : 0u);
          mma_commit(empty_bar(stage));
          if (++stage == kBwdStages) { stage = 0; phase ^= 1u; }
        }
        mma_commit(tfull_bar(acc));
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else {
    // ===== cell warps: the backward pass of the cell on dh_t + acc; a warp owns 32 rows x 16 units of the tile =====
    const int quarter = warp & 3, part = (warp - 2) >> 2;
    const int cw = warp - 2;
    const uint32_t s_dh = stg_base + (uint32_t)cw * 2048u;
    const uint32_t s_dg = stg_base + (uint32_t)kLsCellWarps * 2048u + (uint32_t)cw * 4096u;
    const int cstep = g.tiled ? 128 : 4;
    int acc = 0; uint32_t acc_phase = 0, dh_phase = 0;
    for (int w = blockIdx.x; w < work_total; w += gridDim.x) {
      const int n_blk = w % kNumN, m_blk = w / kNumN;
      const int row0 = m_blk * kLsBM + quarter * 32;
      const int row = row0 + lane;
      const bool row_ok = row < g.n;
      const int u0 = n_blk * BN + part * 16;
      if (g.tiled) {
        if (lane == 0) {
          bulk_wait_read<0>();              // the previous tile's dgates stores have read the staging tiles
          mbar_arrive_expect_tx(dh_bar(cw), 2048);
          tma_load_2d(s_dh, &tma_dh, dh_bar(cw), u0, row0);     // rows >= n arrive as zeros
        }
        __syncwarp();
      }
#pragma unroll 1
      for (int ch = 0; ch < 2; ++ch) {
        const int u = u0 + ch * 8;
        const size_t so = (size_t)row * 256 + u;
        const size_t co = g.tiled ? tiled_off(m_blk * 4 + quarter, 64, u >> 2, lane) * 4 : so;
        // everything the cell needs besides the product: in flight before the accumulator is waited for
        float gi[8], gj[8], gf[8], go[8], cp[8], cc[8], dcv[8], dhh[8], dhv[8];
        uint4 pi = make_uint4(0, 0, 0, 0), pj = pi, pf = pi, po = pi;
        if (row_ok) {
          const __nv_bfloat16* ar = g.acts + (g.tiled ? tiled_off(m_blk * 4 + quarter, 128, u >> 3, lane) * 8 : (size_t)row * 1024 + u);
          const int gstep = g.tiled ? 32 * 256 : 256;
          pi = *reinterpret_cast<const uint4*>(ar); pj = *reinterpret_cast<const uint4*>(ar + gstep);
          pf = *reinterpret_cast<const uint4*>(ar + 2 * gstep); po = *reinterpret_cast<const uint4*>(ar + 3 * gstep);
          ld8f(g.c_prev + co, cp, cstep); ld8f(g.c + co, cc, cstep); ld8f(g.dc + co, dcv, cstep);
          if (!g.tiled) ld8f(g.dh + so, dhh, 4);
        }
        if (ch == 0) {
          if (!g.skip_gemm) {
            mbar_wait(tfull_bar(acc), acc_phase);
            fence_after_sync();
          }
          if (g.tiled) mbar_wait(dh_bar(cw), dh_phase);
        }
        if (!g.skip_gemm) {
          tmem_ld8(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN + part * 16 + ch * 8), dhv);
        } else {
#pragma unroll
          for (int q = 0; q < 8; ++q) dhv[q] = 0.f;
          if (row_ok && g.dh2 != nullptr) ld8f(g.dh2 + so, dhv, 4);
        }
        if (g.tiled) unstage8f(s_dh, lane, ch, dhh);
        unpack8(pi, gi); unpack8(pj, gj); unpack8(pf, gf); unpack8(po, go);
        if (!g.skip_gemm) tmem_ld_wait();
        if (row_ok) {
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            // = model_ops.cu:lstm_cell_bwd_kernel
            const float i = gi[q], j = gj[q], f = gf[q], o = go[q];
            const float tc = tanh_(cc[q]);
            const float d = dhh[q] + dhv[q];
            const float d_o = d * tc;
            const float dct = dcv[q] + d * o * (1.0f - tc * tc);
            gi[q] = dct * j * i * (1.0f - i);
            gj[q] = dct * i * (1.0f - j * j);
            gf[q] = dct * cp[q] * f * (1.0f - f);
            go[q] = d_o * o * (1.0f - o);
            dcv[q] = dct * f;
          }
          st8f(g.dc + co, dcv, cstep);
          if (!g.tiled) {
            __nv_bfloat16* dg = g.dgates + (size_t)row * 1024 + u;
            *reinterpret_cast<uint4*>(dg) = pack8(gi); *reinterpret_cast<uint4*>(dg + 256) = pack8(gj);
            *reinterpret_cast<uint4*>(dg + 512) = pack8(gf); *reinterpret_cast<uint4*>(dg + 768) = pack8(go);
          }
        }
        if (g.tiled) {                       // rows >= n: garbage the TMA store clips
          stage8h(s_dg, lane, ch, gi); stage8h(s_dg + 1024u, lane, ch, gj);
          stage8h(s_dg + 2048u, lane, ch, gf); stage8h(s_dg + 3072u, lane, ch, go);
        }
      }
      fence_before_sync();
      if (g.tiled) fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(tempty_bar(acc));
        if (g.tiled) {
#pragma unroll
          for (int gate = 0; gate < 4; ++gate) tma_store_2d(&tma_dg, s_dg + (uint32_t)gate * 1024u, gate * 256 + u0, row0);
          bulk_commit();
        }
      }
      dh_phase ^= 1u;
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
    if (g.tiled && lane == 0) bulk_wait_all();
  }
  __syncwarp();
  fence_before_sync();
  __syncthreads();
  if (warp == 2) {
    fence_after_sync();
    tmem_dealloc<2 * BN>(tmem_base);
  }
}

}  // namespace
}  // namespace unreal

using namespace unreal;

extern "C" int unreal_lstm_step_fwd(const void* xh, int64_t ld_xh, const void* w, const float* bias, const float* c_prev,
                                    float* c_out, float* h_out, float* h_copy, void* h16_out, int h16_ld, void* acts,
                                    const uint8_t* active, int tiled, int n, int k, void* stream) {
  UNREAL_REQUIRE(xh && w && bias && c_prev && c_out, "unreal_lstm_step_fwd: null operand");
  UNREAL_REQUIRE(n > 0 && k > 0, "unreal_lstm_step_fwd: empty problem (n %d, k %d)", n, k);
  UNREAL_REQUIRE((ld_xh & 7) == 0 && ld_xh >= k, "unreal_lstm_step_fwd: ld_xh %lld must be a multiple of 8 and >= k %d",
                 (long long)ld_xh, k);
  UNREAL_REQUIRE(aligned16(xh) && aligned16(w) && aligned16(c_prev) && aligned16(c_out) && aligned16(h_out) &&
                     aligned16(h_copy) && aligned16(h16_out) && aligned16(acts) && aligned16(bias),
                 "unreal_lstm_step_fwd: buffers must be 16-byte aligned");
  UNREAL_REQUIRE(h16_out == nullptr || (h16_ld >= 256 && (h16_ld & 7) == 0),
                 "unreal_lstm_step_fwd: h16_ld %d must be a multiple of 8 and >= 256", h16_ld);
  UNREAL_REQUIRE(h_copy == nullptr || h_out != nullptr, "unreal_lstm_step_fwd: h_copy needs h_out");
  UNREAL_REQUIRE(!(tiled && (active != nullptr || h_copy != nullptr || c_prev == c_out)),
                 "unreal_lstm_step_fwd: the in-place acting step (active, h_copy, c_out == c_prev) is row-major");
  CUtensorMap ta, tb, th, th16;
  int rc = make_tma_2d(&ta, xh, n, k, ld_xh, kLsBM, false);
  if (rc != UNREAL_OK) return rc;
  rc = make_tma_2d(&tb, w, k, 1024, 1024, kLsBK, false);
  if (rc != UNREAL_OK) return rc;
  th = ta; th16 = ta;
  const uint32_t box[2] = {16, 32};        // a cell warp's 32 rows x 16 units
  if (tiled && h_out != nullptr) {
    const uint64_t dims[2] = {256, (uint64_t)n}, strides[1] = {1024};
    rc = make_tma_nd(&th, true, h_out, 2, dims, strides, box, 64);          // 64-byte rows, 64-byte swizzle
    if (rc != UNREAL_OK) return rc;
  }
  if (tiled && h16_out != nullptr) {
    const uint64_t dims[2] = {256, (uint64_t)n}, strides[1] = {(uint64_t)h16_ld * 2};
    rc = make_tma_nd(&th16, false, h16_out, 2, dims, strides, box, 32);     // 32-byte rows, 32-byte swizzle
    if (rc != UNREAL_OK) return rc;
  }
  rc = allow_dynamic_smem((const void*)lstm_step_fwd_tcgen05_kernel, kFwdSmem);
  if (rc != UNREAL_OK) return rc;
  LstmFwdArgs g{bias, c_prev, c_out, h_out, h_copy, static_cast<__nv_bfloat16*>(h16_out), static_cast<__nv_bfloat16*>(acts),
                active, n, k, h16_ld, tiled ? 1 : 0};
  const int work = (n + kLsBM - 1) / kLsBM * 4;
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  lstm_step_fwd_tcgen05_kernel<<<work < sms ? work : sms, kLsThreads, kFwdSmem, as_stream(stream)>>>(ta, tb, th, th16, g);
  UNREAL_LAUNCH_CHECK("lstm_step_fwd_tcgen05_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_lstm_step_bwd(const void* dgates_next, const void* wh, int64_t ld_wh, const void* acts,
                                    const float* c_prev, const float* c, const float* dh, const float* dh2, float* dc,
                                    void* dgates, int tiled, int n, void* stream) {
  UNREAL_REQUIRE(wh && acts && c_prev && c && dh && dc && dgates, "unreal_lstm_step_bwd: null operand");
  UNREAL_REQUIRE(dgates_next == nullptr || dh2 == nullptr, "unreal_lstm_step_bwd: dh2 is the last step's (dgates_next NULL) extra gradient");
  UNREAL_REQUIRE(n > 0, "unreal_lstm_step_bwd: n %d", n);
  UNREAL_REQUIRE((ld_wh & 7) == 0 && ld_wh >= 1024, "unreal_lstm_step_bwd: ld_wh %lld must be a multiple of 8 and >= 1024",
                 (long long)ld_wh);
  UNREAL_REQUIRE(aligned16(dgates_next) && aligned16(wh) && aligned16(acts) && aligned16(c_prev) && aligned16(c) &&
                     aligned16(dh) && aligned16(dh2) && aligned16(dc) && aligned16(dgates),
                 "unreal_lstm_step_bwd: buffers must be 16-byte aligned");
  const bool skip = dgates_next == nullptr;        // the unroll's last step: the cell's backward pass alone
  CUtensorMap ta, tb, tdh, tdg;
  int rc = make_tma_2d(&ta, skip ? wh : dgates_next, skip ? 256 : n, 1024, skip ? ld_wh : 1024, kLsBM, false);
  if (rc != UNREAL_OK) return rc;
  rc = make_tma_2d(&tb, wh, 256, 1024, ld_wh, kBwdBN, false);
  if (rc != UNREAL_OK) return rc;
  tdh = ta; tdg = ta;
  if (tiled) {
    const uint32_t box[2] = {16, 32};      // a cell warp's 32 rows x 16 units
    const uint64_t dims_h[2] = {256, (uint64_t)n}, strides_h[1] = {1024};
    rc = make_tma_nd(&tdh, true, dh, 2, dims_h, strides_h, box, 64);
    if (rc != UNREAL_OK) return rc;
    const uint64_t dims_g[2] = {1024, (uint64_t)n}, strides_g[1] = {2048};
    rc = make_tma_nd(&tdg, false, dgates, 2, dims_g, strides_g, box, 32);
    if (rc != UNREAL_OK) return rc;
  }
  rc = allow_dynamic_smem((const void*)lstm_step_bwd_tcgen05_kernel, kBwdSmem);
  if (rc != UNREAL_OK) return rc;
  LstmBwdArgs g{static_cast<const __nv_bfloat16*>(acts), c_prev, c, dh, dc, static_cast<__nv_bfloat16*>(dgates), dh2, n,
                tiled ? 1 : 0, skip ? 1 : 0};
  const int work = (n + kLsBM - 1) / kLsBM * (256 / kBwdBN);
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  lstm_step_bwd_tcgen05_kernel<<<work < sms ? work : sms, kLsThreads, kBwdSmem, as_stream(stream)>>>(ta, tb, tdh, tdg, g);
  UNREAL_LAUNCH_CHECK("lstm_step_bwd_tcgen05_kernel");
  return UNREAL_OK;
}
