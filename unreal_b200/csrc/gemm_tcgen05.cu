// K7: bf16 x bf16 -> fp32 GEMM on the sm_100a tensor path (tcgen05.mma, TMEM accumulators, TMA).
//
// The dense layers of UnrealModel (model/model.py:281-598) are tf.matmul / tf.nn.conv2d calls in
// the reference; batched over envs x time they become the GEMMs
//     fc1      [S, 2592] x [2592, 256]      (model.py:337-340)
//     LSTM     [S, 256+A+1+G] x [., 1024] and per step [N, 256] x [256, 1024]   (:110, :346-351)
//     pc_fc1   [S, 256] x [256, 2592]       (:424)
//     conv1/2  im2col [S*400, 192] x [192, 16], [S*81, 256] x [256, 32]          (:283-289)
//     deconv   [S*81, 32] x [32, 16*(1+A)]  (:425-430)
// plus their dgrad / wgrad transposes.  One kernel serves all of them:
//
//     C[M,N] (=|+=) act( A * B + bias ),   fp32 accumulation in TMEM
//
//   A: "K-major"  = row-major [M,K] (K contiguous)   or "MN-major" = row-major [K,M] (M contiguous)
//   B: "K-major"  = row-major [N,K] (K contiguous)   or "MN-major" = row-major [K,N] (N contiguous)
// so forward (X * W, W stored [in,out] like TF), dgrad (dY * W^T) and wgrad (X^T * dY) all read
// the operands where they lie, with no transposed copies.
//
// Structure (one persistent CTA per SM, 192 threads):
//   warp 0   TMA producer: cp.async.bulk.tensor.2d with 128-byte swizzle into a ring of kStages
//            shared-memory stages, one mbarrier pair (full/empty) per stage;
//   warp 1   MMA issuer: ONE thread issues tcgen05.mma.cta_group::1.kind::f16 (UMMA 128 x BN x 16),
//            tcgen05.commit releases the stage / publishes the accumulator;
//   warps 2-5 epilogue: tcgen05.ld (32 lanes x 32 columns) -> bias / ReLU / convert -> global.
//            Two TMEM accumulator buffers, so the epilogue of tile i overlaps the MMAs of tile i+1.
// Split-K (wgrad: K = samples is the long dimension) adds the partial tiles with red.global.add.f32.
#include <cuda.h>
#include <cuda_bf16.h>

#include <mutex>

#include "common.cuh"
#include "tc05.cuh"

namespace unreal {
using namespace tc05;

constexpr int kBM = 128;        // UMMA M (cta_group::1): accumulator row i lives in TMEM lane i
constexpr int kBK = 64;         // bf16 elements per stage along K = one 128-byte swizzle row
constexpr int kUmmaK = 16;      // K per tcgen05.mma for 16-bit operands
constexpr int kGemmThreads = 192;
constexpr uint32_t kDescHiSw128 = (1024u >> 4) | (1u << 14) | (2u << 29);   // SBO 1024 B, version 1, 128-byte swizzle

struct GemmArgs {
  void* c;
  const float* bias;
  const void* add;  // optional [M,N] f32 addend read by the epilogue (ld = ldc)
  int64_t ldc;
  int m, n, k;
  int split_k;
  int c_bf16;       // 1: C is bf16, 0: f32
  int relu;
  int accumulate;   // 1: C += result (red.global.add.f32); implied by split_k > 1
  int tma_store;    // 1: epilogue stages tiles in shared memory and stores / reduces them with TMA
};

// DEEP: short-K, output-dominated products (pc_fc1 forward: K = 256, 849 MB out; the LSTM acting step).  Their tiles
// spend ~1 us in the MMAs and then wait for the epilogue -- ncu of pc_fc1 forward (profiles/r2_pcfc1_fwd_ncu_summary.txt):
// 342 us with the tensor pipe 35 % busy, DRAM 31 %, L2 43 %, the ONE epilogue warp per scheduler issuing 28 % of the
// cycles and stalled on fixed-latency dependencies for most of the rest (~1800 dependent instructions per 32 x 256
// accumulator slice).  The deep build runs EIGHT epilogue warps (two per TMEM lane quarter, half the columns each; 320
// threads), paid for with a pipeline stage a 4-block K loop cannot use anyway.
template <int BN, bool DEEP = false>
struct GemmCfg {
  static constexpr int kABytes = kBM * kBK * 2;
  static constexpr int kBBytes = BN * kBK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = DEEP ? ((BN >= 256) ? 3 : (BN >= 128 ? 5 : 6)) : ((BN >= 256) ? 4 : (BN >= 128 ? 6 : 8));
  static constexpr int kTmemCols = (2 * BN <= 32) ? 32 : (2 * BN <= 64 ? 64 : (2 * BN <= 128 ? 128 : (2 * BN <= 256 ? 256 : 512)));
  static constexpr int kEpiWarps = DEEP ? 8 : 4;
  static constexpr int kThreads = 32 * (2 + kEpiWarps);
  static constexpr int kEpiBytes = kEpiWarps * 2 * 4096;  // epilogue warps x 2 buffers x [32 rows x 128 B]
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*barriers, tmem slot*/ + kEpiBytes + 1024 /*alignment slack*/;
};

// One accumulator tile [32 rows of this warp x BN columns]: TMEM -> registers -> bias / addend /
// ReLU -> C.  `lead` = this work item applies bias / addend (first K split).  TMA-store path: the
// warp stages [32 rows x 128 bytes] (64 bf16 or 32 f32 columns) in its own double-buffered,
// 128B-swizzled shared-memory tile and hands it to the TMA engine, which writes whole 128-byte
// lines and clips rows / columns outside C.
template <int BN>
__device__ __forceinline__ void epilogue_tile(const GemmArgs& g, const CUtensorMap* tma_c, uint32_t tmem_row,
                                              uint32_t ebuf, uint32_t& ebuf_it, int lane, int warp_row0, int n_blk,
                                              bool lead, int c_begin = 0, int c_end = BN) {
  const bool atomic = g.accumulate || g.split_k > 1;
  const int row = warp_row0 + lane;
  const bool row_ok = row < g.m;
  if (g.tma_store) {
    const int group = g.c_bf16 ? 64 : 32;          // columns per 128-byte staged row
#pragma unroll 1
    for (int c0 = c_begin; c0 < c_end; c0 += group) {
      const int gcol0 = n_blk * BN + c0;
      if (gcol0 >= g.n) break;                     // uniform: the rest of the tile is outside C
      const uint32_t buf = ebuf + (ebuf_it & 1u) * 4096u;
      ++ebuf_it;
      if (lane == 0) bulk_wait_read<1>();          // the store issued two groups ago has read `buf`
      __syncwarp();
      const uint32_t rowp = buf + (uint32_t)lane * 128u;
#pragma unroll 1
      for (int half = 0; half * 32 < group; ++half) {
        uint32_t r[32];
        tmem_ld32(tmem_row + (uint32_t)(c0 + half * 32), r);
        tmem_ld_wait();
        const int col0 = gcol0 + half * 32;
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
        if (g.bias != nullptr && lead) {
          if (col0 + 32 <= g.n) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 t = __ldg(reinterpret_cast<const float4*>(g.bias + col0 + j));
              v[j] += t.x; v[j + 1] += t.y; v[j + 2] += t.z; v[j + 3] += t.w;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) if (col0 + j < g.n) v[j] += __ldg(g.bias + col0 + j);
          }
        }
        if (g.add != nullptr && lead && row_ok) {
          const float* ap = reinterpret_cast<const float*>(g.add) + (size_t)row * g.ldc + col0;
#pragma unroll
          for (int j = 0; j < 32; ++j) if (col0 + j < g.n) v[j] += ap[j];
        }
        if (g.relu) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        if (g.c_bf16) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            __nv_bfloat162 p0 = __floats2bfloat162_rn(v[8 * q], v[8 * q + 1]);
            __nv_bfloat162 p1 = __floats2bfloat162_rn(v[8 * q + 2], v[8 * q + 3]);
            __nv_bfloat162 p2 = __floats2bfloat162_rn(v[8 * q + 4], v[8 * q + 5]);
            __nv_bfloat162 p3 = __floats2bfloat162_rn(v[8 * q + 6], v[8 * q + 7]);
            const uint32_t chunk = (uint32_t)(half * 4 + q) ^ (uint32_t)(lane & 7);
            st_shared_v4(rowp + chunk * 16u, *reinterpret_cast<uint32_t*>(&p0), *reinterpret_cast<uint32_t*>(&p1),
                         *reinterpret_cast<uint32_t*>(&p2), *reinterpret_cast<uint32_t*>(&p3));
          }
        } else {
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const uint32_t chunk = (uint32_t)q ^ (uint32_t)(lane & 7);
            st_shared_v4(rowp + chunk * 16u, __float_as_uint(v[4 * q]), __float_as_uint(v[4 * q + 1]),
                         __float_as_uint(v[4 * q + 2]), __float_as_uint(v[4 * q + 3]));
          }
        }
      }
      fence_proxy_async_smem();                    // generic-proxy writes -> visible to the TMA engine
      __syncwarp();
      if (lane == 0) {
        if (atomic) tma_reduce_add_2d(tma_c, buf, gcol0, warp_row0);
        else tma_store_2d(tma_c, buf, gcol0, warp_row0);
        bulk_commit();
      }
    }
  } else {
#pragma unroll 1
  for (int c0 = c_begin; c0 < c_end; c0 += 32) {
    uint32_t r[32];
    tmem_ld32(tmem_row + (uint32_t)c0, r);
    tmem_ld_wait();
    const int col0 = n_blk * BN + c0;
    if (row_ok && col0 < g.n) {
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
      if (g.bias != nullptr && lead) {
#pragma unroll
        for (int j = 0; j < 32; ++j) if (col0 + j < g.n) v[j] += __ldg(g.bias + col0 + j);
      }
      if (g.add != nullptr && lead) {
        const float* ap = reinterpret_cast<const float*>(g.add) + (size_t)row * g.ldc + col0;
#pragma unroll
        for (int j = 0; j < 32; ++j) if (col0 + j < g.n) v[j] += ap[j];
      }
      if (g.relu) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
      }
      // unaligned / odd leading dimensions: plain element stores
      if (g.c_bf16) {
        __nv_bfloat16* cp = reinterpret_cast<__nv_bfloat16*>(g.c) + (size_t)row * g.ldc + col0;
#pragma unroll
        for (int j = 0; j < 32; ++j) if (col0 + j < g.n) cp[j] = __float2bfloat16_rn(v[j]);
      } else {
        float* cp = reinterpret_cast<float*>(g.c) + (size_t)row * g.ldc + col0;
        if (atomic) {
#pragma unroll
          for (int j = 0; j < 32; ++j) if (col0 + j < g.n) atomicAdd(cp + j, v[j]);
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) if (col0 + j < g.n) cp[j] = v[j];
        }
      }
    }
  }
  }
}

template <int BN, bool A_MN, bool B_MN, bool DEEP = false>
__global__ void __launch_bounds__(GemmCfg<BN, DEEP>::kThreads, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                    const __grid_constant__ CUtensorMap tma_c, const GemmArgs g) {
  using Cfg = GemmCfg<BN, DEEP>;
  extern __shared__ uint8_t smem_raw[];
  // 128-byte swizzle atoms are 1024 bytes: every operand tile starts on a 1024-byte boundary
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + Cfg::kStages * Cfg::kStageBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::kStages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * Cfg::kStages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * Cfg::kStages + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * Cfg::kStages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_m = (g.m + kBM - 1) / kBM, num_n = (g.n + BN - 1) / BN;
  const int kb_total = (g.k + kBK - 1) / kBK;
  const int kb_per = (kb_total + g.split_k - 1) / g.split_k;
  const int work_total = num_m * num_n * g.split_k;

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tma_a);
    prefetch_tensormap(&tma_b);
    if (g.tma_store) prefetch_tensormap(&tma_c);
    for (int s = 0; s < Cfg::kStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), Cfg::kEpiWarps); }
    fence_mbar_init();
  } else if (warp == 2) {
    tmem_alloc<Cfg::kTmemCols>(tmem_slot);
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = tmem_base_at(tmem_slot);

  if (warp == 0) {
    if (lane == 0) {
      // ===== TMA producer =====
      int stage = 0; uint32_t phase = 0;
      for (int w = blockIdx.x; w < work_total; w += gridDim.x) {
        const int n_blk = w % num_n, m_blk = (w / num_n) % num_m, sp = w / (num_n * num_m);
        const int kb0 = sp * kb_per, kb1 = min(kb0 + kb_per, kb_total);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sa = smem_base + stage * Cfg::kStageBytes, sb = sa + Cfg::kABytes;
          mbar_arrive_expect_tx(full_bar(stage), Cfg::kStageBytes);
          if (A_MN) {
#pragma unroll
            for (int b = 0; b < kBM / 64; ++b)
              tma_load_2d(sa + b * (kBK * 128), &tma_a, full_bar(stage), m_blk * kBM + b * 64, kb * kBK);
          } else {
            tma_load_2d(sa, &tma_a, full_bar(stage), kb * kBK, m_blk * kBM);
          }
          if (B_MN) {
#pragma unroll
            for (int b = 0; b < BN / 64; ++b)
              tma_load_2d(sb + b * (kBK * 128), &tma_b, full_bar(stage), n_blk * BN + b * 64, kb * kBK);
          } else {
            tma_load_2d(sb, &tma_b, full_bar(stage), kb * kBK, n_blk * BN);
          }
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===== MMA issuer =====
      constexpr uint32_t idesc = idesc_bf16_f32(kBM, BN, A_MN, B_MN);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int w = blockIdx.x; w < work_total; w += gridDim.x) {
        const int sp = w / (num_n * num_m);
        const int kb0 = sp * kb_per, kb1 = min(kb0 + kb_per, kb_total);
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);   // epilogue has drained this accumulator
        fence_after_sync();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar(stage), phase);
          fence_after_sync();
          const uint32_t sa = smem_base + stage * Cfg::kStageBytes, sb = sa + Cfg::kABytes;
          // K-major: 16 elements = 32 bytes further inside the swizzle row; 8-row groups 1024 B apart.
          // MN-major: 16 k-rows = two 8-row groups = 2048 bytes; 64-element MN chunks kBK*128 B apart.
          // Descriptors as (lo, hi) words: hi is constant, lo = (address >> 4) | LBO field.
          const uint32_t a_lo = (sa >> 4) | ((A_MN ? (uint32_t)(kBK * 128) >> 4 : 1u) << 16);
          const uint32_t b_lo = (sb >> 4) | ((B_MN ? (uint32_t)(kBK * 128) >> 4 : 1u) << 16);
#pragma unroll
          for (int k = 0; k < kBK / kUmmaK; ++k)
            mma_f16_lohi(tmem_d, a_lo + (uint32_t)k * (A_MN ? 128u : 2u), kDescHiSw128, b_lo + (uint32_t)k * (B_MN ? 128u : 2u),
                         kDescHiSw128, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          mma_commit(empty_bar(stage));               // stage is free once these MMAs have read it
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1u; }
        }
        mma_commit(tfull_bar(acc));                   // accumulator complete
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else {
    // ===== epilogue (warps 2..5): warp w may touch TMEM lanes 32*(w%4) .. +31 =====
    const int quarter = warp & 3;
    int acc = 0; uint32_t acc_phase = 0;
    const uint32_t ebuf = smem_base + Cfg::kStages * Cfg::kStageBytes + 1024u + (uint32_t)(warp - 2) * 8192u;
    uint32_t ebuf_it = 0;
    constexpr int kColsPerWarp = BN / (Cfg::kEpiWarps / 4);      // deep build: the two warps of a lane quarter split the columns
    const int c_begin = ((warp - 2) >> 2) * kColsPerWarp;
    for (int w = blockIdx.x; w < work_total; w += gridDim.x) {
      const int n_blk = w % num_n, m_blk = (w / num_n) % num_m, sp = w / (num_n * num_m);
      mbar_wait(tfull_bar(acc), acc_phase);
      fence_after_sync();
      epilogue_tile<BN>(g, &tma_c, tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN), ebuf, ebuf_it,
                        lane, m_blk * kBM + quarter * 32, n_blk, sp == 0, c_begin, c_begin + kColsPerWarp);
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
    if (lane == 0) bulk_wait_all();                    // staged tiles must be read before the CTA exits
  }
  __syncwarp();
  fence_before_sync();
  __syncthreads();
  if (warp == 2) {
    fence_after_sync();
    tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
}


// ---- CTA-pair variant: 256 x 256 tile per cluster of two CTAs (tcgen05.mma.cta_group::2) ----------
// Each CTA loads its own 128 rows of A and its own 128 of the tile's 256 B rows (so operand traffic
// from L2 per SM is half that of two independent 128x256 tiles), the leader CTA issues the MMAs for
// both, every CTA's TMEM receives its 128 accumulator rows and runs its own epilogue.
// BN = 256: A 16 KB + B half 16 KB per stage, 6 stages; BN = 128 (256 x 128 tiles, used when the
// 256-wide tiling would leave the last wave of CTA pairs mostly empty): B half 8 KB, 8 stages.
template <int BN> struct Cfg2 {
  static constexpr int kStages = BN == 256 ? 6 : 8;
  static constexpr int kStageBytes = kBM * kBK * 2 + (BN / 2) * kBK * 2;
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 + 4 * 2 * 4096 + 1024;
  static constexpr int kTmemCols = 2 * BN;
};

template <int BN, bool A_MN, bool B_MN>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
gemm2sm_tcgen05_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                       const __grid_constant__ CUtensorMap tma_c, const GemmArgs g) {
  constexpr int k2Stages = Cfg2<BN>::kStages, k2StageBytes = Cfg2<BN>::kStageBytes;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + k2Stages * k2StageBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (k2Stages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * k2Stages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * k2Stages + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * k2Stages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
  const int num_m = (g.m + 2 * kBM - 1) / (2 * kBM), num_n = (g.n + BN - 1) / BN;
  const int kb_total = (g.k + kBK - 1) / kBK;
  const int kb_per = (kb_total + g.split_k - 1) / g.split_k;
  const int work_total = num_m * num_n * g.split_k;

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tma_a);
    prefetch_tensormap(&tma_b);
    if (g.tma_store) prefetch_tensormap(&tma_c);
    for (int s = 0; s < k2Stages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 8); }
    fence_mbar_init();
  } else if (warp == 2) {
    tmem_alloc_2sm<Cfg2<BN>::kTmemCols>(tmem_slot);
  }
  fence_before_sync();
  cluster_sync_all();                 // both CTAs' barriers exist before any remote arrive / TMA signal
  fence_after_sync();
  const uint32_t tmem_base = tmem_base_at(tmem_slot);

  if (warp == 0) {
    if (lane == 0) {
      // ===== TMA producer (both CTAs): own A rows, own half of the B rows =====
      int stage = 0; uint32_t phase = 0;
      for (int w = cluster_id; w < work_total; w += num_clusters) {
        const int n_blk = w % num_n, m_blk = (w / num_n) % num_m, sp = w / (num_n * num_m);
        const int kb0 = sp * kb_per, kb1 = min(kb0 + kb_per, kb_total);
        const int m0 = m_blk * 2 * kBM + (int)rank * kBM, n0 = n_blk * BN + (int)rank * (BN / 2);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sa = smem_base + stage * k2StageBytes, sb = sa + kBM * kBK * 2;
          if (leader) mbar_arrive_expect_tx(full_bar(stage), 2 * k2StageBytes);   // both CTAs' bytes
          if (A_MN) {
#pragma unroll
            for (int b = 0; b < kBM / 64; ++b)
              tma_load_2d_2sm(sa + b * (kBK * 128), &tma_a, full_bar(stage), m0 + b * 64, kb * kBK);
          } else {
            tma_load_2d_2sm(sa, &tma_a, full_bar(stage), kb * kBK, m0);
          }
          if (B_MN) {
#pragma unroll
            for (int b = 0; b < BN / 2 / 64; ++b)
              tma_load_2d_2sm(sb + b * (kBK * 128), &tma_b, full_bar(stage), n0 + b * 64, kb * kBK);
          } else {
            tma_load_2d_2sm(sb, &tma_b, full_bar(stage), kb * kBK, n0);
          }
          if (++stage == k2Stages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && leader) {
      // ===== MMA issuer (leader CTA only) =====
      constexpr uint32_t idesc = idesc_bf16_f32(2 * kBM, BN, A_MN, B_MN);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int w = cluster_id; w < work_total; w += num_clusters) {
        const int sp = w / (num_n * num_m);
        const int kb0 = sp * kb_per, kb1 = min(kb0 + kb_per, kb_total);
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);   // both CTAs' epilogues have drained this accumulator
        fence_after_sync();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar(stage), phase);
          fence_after_sync();
          const uint32_t sa = smem_base + stage * k2StageBytes, sb = sa + kBM * kBK * 2;
#pragma unroll
          for (int k = 0; k < kBK / kUmmaK; ++k) {
            const uint64_t ad = A_MN ? smem_desc_sw128(sa + k * 2048, kBK * 128, 1024)
                                     : smem_desc_sw128(sa + k * 32, 16, 1024);
            const uint64_t bd = B_MN ? smem_desc_sw128(sb + k * 2048, kBK * 128, 1024)
                                     : smem_desc_sw128(sb + k * 32, 16, 1024);
            mma_f16_2sm(tmem_d, ad, bd, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          mma_commit_2sm(empty_bar(stage), 3);        // frees the stage in BOTH CTAs
          if (++stage == k2Stages) { stage = 0; phase ^= 1u; }
        }
        mma_commit_2sm(tfull_bar(acc), 3);            // accumulator complete, both epilogues may read
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else {
    // ===== epilogue (warps 2..5 of both CTAs): this CTA's 128 accumulator rows =====
    const int quarter = warp & 3;
    int acc = 0; uint32_t acc_phase = 0;
    const uint32_t ebuf = smem_base + k2Stages * k2StageBytes + 1024u + (uint32_t)(warp - 2) * 8192u;
    uint32_t ebuf_it = 0;
    for (int w = cluster_id; w < work_total; w += num_clusters) {
      const int n_blk = w % num_n, m_blk = (w / num_n) % num_m, sp = w / (num_n * num_m);
      mbar_wait(tfull_bar(acc), acc_phase);
      fence_after_sync();
      epilogue_tile<BN>(g, &tma_c, tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN), ebuf, ebuf_it,
                        lane, m_blk * 2 * kBM + (int)rank * kBM + quarter * 32, n_blk, sp == 0);
      fence_before_sync();
      __syncwarp();
      if (lane == 0) {
        if (leader) mbar_arrive(tempty_bar(acc));
        else mbar_arrive_remote(mapa_cluster(tempty_bar(acc), 0));
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
    if (lane == 0) bulk_wait_all();
  }
  __syncwarp();
  fence_before_sync();
  cluster_sync_all();                 // the peer may still be read by the leader's MMAs / signal its barriers
  if (warp == 2) {
    fence_after_sync();
    tmem_dealloc_2sm<Cfg2<BN>::kTmemCols>(tmem_base);
  }
}

// ---- host side -------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

int make_tma_2d(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows, bool f32) {
  EncodeTiledFn fn = encode_tiled();
  if (fn == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from the CUDA driver");
    return UNREAL_ECUDA;
  }
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * (f32 ? 4 : 2)};
  cuuint32_t box[2] = {f32 ? 32u : 64u, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = fn(map, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for a [%lld x %lld] matrix, ld %lld", (int)r, (long long)rows,
              (long long)cols, (long long)ld);
    return UNREAL_ECUDA;
  }
  return UNREAL_OK;
}

int make_tma_nd(CUtensorMap* map, bool f32, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                const uint32_t* box, int swizzle_bytes) {
  EncodeTiledFn fn = encode_tiled();
  if (fn == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from the CUDA driver");
    return UNREAL_ECUDA;
  }
  cuuint64_t d[5]; cuuint64_t st[4]; cuuint32_t b[5]; cuuint32_t e[5];
  for (int i = 0; i < rank; ++i) { d[i] = dims[i]; b[i] = box[i]; e[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) st[i] = strides_bytes[i];
  const CUtensorMapSwizzle sw = swizzle_bytes == 0 ? CU_TENSOR_MAP_SWIZZLE_NONE
                                : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B;
  CUresult r = fn(map, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank,
                  const_cast<void*>(base), d, st, b, e, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for a rank-%d %s tensor", (int)r, rank, f32 ? "f32" : "bf16");
    return UNREAL_ECUDA;
  }
  return UNREAL_OK;
}

int make_tma_nd_bf16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                     const uint32_t* box, int swizzle_bytes) {
  return make_tma_nd(map, false, base, rank, dims, strides_bytes, box, swizzle_bytes);
}

template <int BN, bool A_MN, bool B_MN, bool DEEP = false>
static int launch_gemm(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const GemmArgs& g,
                       cudaStream_t st) {
  using Cfg = GemmCfg<BN, DEEP>;
  auto kern = gemm_tcgen05_kernel<BN, A_MN, B_MN, DEEP>;
  const int rc = allow_dynamic_smem((const void*)kern, Cfg::kSmemBytes);
  if (rc != UNREAL_OK) return rc;
  const int num_m = (g.m + kBM - 1) / kBM, num_n = (g.n + BN - 1) / BN;
  const int64_t work = (int64_t)num_m * num_n * g.split_k;
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  const int grid = (int)(work < sms ? work : sms);
  kern<<<grid, Cfg::kThreads, Cfg::kSmemBytes, st>>>(ta, tb, tc, g);
  UNREAL_LAUNCH_CHECK("gemm_tcgen05_kernel");
  return UNREAL_OK;
}

template <int BN, bool A_MN, bool B_MN>
static int launch_gemm_2sm(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const GemmArgs& g,
                           cudaStream_t st) {
  auto kern = gemm2sm_tcgen05_kernel<BN, A_MN, B_MN>;
  const int rc = allow_dynamic_smem((const void*)kern, Cfg2<BN>::kSmemBytes);
  if (rc != UNREAL_OK) return rc;
  const int num_m = (g.m + 2 * kBM - 1) / (2 * kBM), num_n = (g.n + BN - 1) / BN;
  const int64_t work = (int64_t)num_m * num_n * g.split_k;
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  const int clusters = (int)(work < sms / 2 ? work : sms / 2);
  kern<<<2 * clusters, kGemmThreads, Cfg2<BN>::kSmemBytes, st>>>(ta, tb, tc, g);
  UNREAL_LAUNCH_CHECK("gemm2sm_tcgen05_kernel");
  return UNREAL_OK;
}

}  // namespace unreal

using namespace unreal;

extern "C" int unreal_gemm_bf16(const void* a, int64_t lda, int a_mn_major, const void* b, int64_t ldb,
                                int b_mn_major, void* c, int64_t ldc, int c_dtype, const float* bias,
                                const float* add, int relu, int accumulate, int split_k, int m, int n, int k,
                                void* stream) {
  UNREAL_REQUIRE(a && b && c, "unreal_gemm_bf16: null operand");
  UNREAL_REQUIRE(m > 0 && n > 0 && k > 0, "unreal_gemm_bf16: empty problem %d x %d x %d", m, n, k);
  // the TMA-store epilogue reads the bias as float4
  UNREAL_REQUIRE(aligned16(a) && aligned16(b) && aligned16(c) && (bias == nullptr || aligned16(bias)),
                 "unreal_gemm_bf16: operands and bias must be 16-byte aligned");
  UNREAL_REQUIRE((lda & 7) == 0 && (ldb & 7) == 0, "unreal_gemm_bf16: lda/ldb must be multiples of 8 elements (TMA)");
  UNREAL_REQUIRE(lda >= (a_mn_major ? m : k) && ldb >= (b_mn_major ? n : k) && ldc >= n,
                 "unreal_gemm_bf16: leading dimension smaller than the row length");
  UNREAL_REQUIRE(c_dtype == UNREAL_GEMM_OUT_F32 || c_dtype == UNREAL_GEMM_OUT_BF16, "unreal_gemm_bf16: bad c_dtype");
  if (split_k < 1) split_k = 1;
  const int kb_total = (k + kBK - 1) / kBK;
  if (split_k > kb_total) split_k = kb_total;
  // every split must own at least one K block
  while (split_k > 1 && (int64_t)((kb_total + split_k - 1) / split_k) * (split_k - 1) >= kb_total) --split_k;
  UNREAL_REQUIRE(!(c_dtype == UNREAL_GEMM_OUT_BF16 && (accumulate || split_k > 1)),
                 "unreal_gemm_bf16: accumulate / split-K need an f32 output");
  UNREAL_REQUIRE(!(relu && (accumulate || split_k > 1)), "unreal_gemm_bf16: ReLU cannot be fused with accumulation");
  // tile width: wide tiles for wide outputs; MN-major B needs whole 64-column boxes
  int bn = (n > 128) ? 256 : ((n > 64) ? 128 : (n > 32 ? 64 : 32));
  // small-M problems (the LSTM step at 1024-2048 envs, acting-side layers): a wide tile leaves most SMs idle and the
  // launch is one pipeline fill long whatever the tile does -- narrow the tile until the grid is about one wave
  // (measured, profiles/r2_gemm_small_tiles.jsonl: [1024,520]x[520,1024] 11.1 us at BN 256, 7.2 us at BN 64;
  // [2048,...] 11.4 -> 8.6 us at BN 128; at 8192 rows BN 256 stays best)
  {
    const int64_t m_tiles = (m + kBM - 1) / kBM;
    const int64_t want = (int64_t)sm_count() * 4 / 5;
    // (not for split-K products -- the wgrad GEMMs are bound by operand traffic per flop, where the wide tile wins:
    // the LSTM's [520,S]x[S,1024] filter gradient measured 250 us at BN 256 and 361 us at BN 128)
    while (split_k == 1 && bn > 64 && m_tiles * ((n + bn - 1) / bn) < want) bn /= 2;
  }
  { int forced = get_tunable("gemm_bn", 0); if (forced == 32 || forced == 64 || forced == 128 || forced == 256) bn = forced; }
  if (b_mn_major && bn < 64) bn = 64;
  // a bf16 output row of the TMA-store epilogue is staged and stored 64 columns at a time: a 32-column tile would read
  // the other accumulator's TMEM columns and store them over the next tile
  if (c_dtype == UNREAL_GEMM_OUT_BF16 && bn < 64) bn = 64;
  // CTA-pair kernel (256 x 256 tiles) once there is at least one full wave of pairs
  const int64_t work2 = (int64_t)((m + 255) / 256) * ((n + 255) / 256) * split_k;
  // ... and the problem is compute-bound (long K): short-K, output-dominated shapes are paced by the
  // epilogue, where independent CTAs measured faster (profiles/r1_gemm_bench_v4_2sm.jsonl)
  int use_2sm = (n > 128) && work2 >= sm_count() / 2 && kb_total >= 16;
  if (split_k > 1) {
    // split-K products (filter gradients) are a handful of tiles times the split the caller chose for ONE wave of single
    // CTAs: as pairs that count must fill a wave of the 74 pairs about as well, or the second, nearly empty wave costs
    // more than pairing saves (the LSTM's [520,S]x[S,1024] gradient at split 7: 140 single-CTA items = 0.95 of a wave,
    // 181 us; 84 pair items = 1.14 waves, 285 us; pc_fc1's [256,S]x[S,2592] at split 6: 132 items / 66 pairs, 223 vs
    // 199 us -- profiles/r2_wgrad_split_bench.jsonl)
    const int sms = sm_count(), pairs = sms / 2;
    const int64_t work1 = (int64_t)((m + kBM - 1) / kBM) * ((n + 255) / 256) * split_k;
    const double eff1 = (double)work1 / (double)(((work1 + sms - 1) / sms) * sms);
    const double eff2 = (double)work2 / (double)(((work2 + pairs - 1) / pairs) * pairs);
    use_2sm = (n > 128) && kb_total / split_k >= 16 && eff2 >= eff1 - 0.05;
  }
  { int forced = get_tunable("gemm_2sm", -1); if (forced == 0) use_2sm = 0; else if (forced == 1 && n > 128) use_2sm = 1; }
  if (use_2sm) {
    // 256 x 256 tiles.  256 x 128 tiles fill the last wave of the 74 CTA pairs better (fc1: 8.6 waves
    // instead of 4.3) but measured SLOWER everywhere (fc1 830 vs 1134 TFLOP/s, 4096^3 920 vs 1303,
    // profiles/r1_gemm_bench_v5_2sm_bn128.jsonl): operand traffic per flop from L2 is what bounds this
    // kernel, not the tail.  The narrow variant stays selectable with the tunable for experiments.
    bn = 256;
    int forced = get_tunable("gemm_2sm_bn", 0);
    if (forced == 128 || forced == 256) bn = forced;
  }
  CUtensorMap ta, tb, tc;
  int rc;
  if (a_mn_major) rc = make_tma_2d(&ta, a, k, m, lda, kBK, false); else rc = make_tma_2d(&ta, a, m, k, lda, kBM, false);
  if (rc != UNREAL_OK) return rc;
  if (b_mn_major) rc = make_tma_2d(&tb, b, k, n, ldb, kBK, false);
  else rc = make_tma_2d(&tb, b, n, k, ldb, use_2sm ? bn / 2 : bn, false);   // a CTA of a pair loads half the B rows
  if (rc != UNREAL_OK) return rc;
  const bool c_bf16 = c_dtype == UNREAL_GEMM_OUT_BF16;
  // TMA epilogue needs a 16-byte row pitch and rows of whole 16-byte chunks: a bf16 C of n = 52 (104-byte rows) inside
  // a wider buffer had the columns past n written by the TMA store.  Other shapes fall back to element stores.
  const int c_esize = c_bf16 ? 2 : 4;
  int tma_store = ((ldc * c_esize) % 16 == 0) && (((int64_t)n * c_esize) % 16 == 0) && get_tunable("gemm_tma_store", 1) != 0;
  if (tma_store) {
    rc = make_tma_2d(&tc, c, m, n, ldc, 32, !c_bf16);
    if (rc != UNREAL_OK) return rc;
  } else {
    tc = ta;
  }
  GemmArgs g{c, bias, add, ldc, m, n, k, split_k, c_bf16 ? 1 : 0, relu ? 1 : 0, accumulate ? 1 : 0, tma_store};
  cudaStream_t st = as_stream(stream);
  if (use_2sm) {
#define UNREAL_GEMM2_CASE(BN_, AMN_, BMN_) \
  if (bn == BN_ && (a_mn_major != 0) == AMN_ && (b_mn_major != 0) == BMN_) return launch_gemm_2sm<BN_, AMN_, BMN_>(ta, tb, tc, g, st);
    UNREAL_GEMM2_CASE(256, false, false) UNREAL_GEMM2_CASE(256, false, true)
    UNREAL_GEMM2_CASE(256, true, false) UNREAL_GEMM2_CASE(256, true, true)
    UNREAL_GEMM2_CASE(128, false, false) UNREAL_GEMM2_CASE(128, false, true)
    UNREAL_GEMM2_CASE(128, true, false) UNREAL_GEMM2_CASE(128, true, true)
#undef UNREAL_GEMM2_CASE
  }
  // short-K, output-dominated forward / dgrad products: the deep-epilogue build (GemmCfg<BN, true>)
  int deep = split_k == 1 && !accumulate && !a_mn_major && kb_total <= 8 && tma_store && bn >= 128 &&
             (int64_t)((m + kBM - 1) / kBM) * ((n + bn - 1) / bn) >= 2 * sm_count();
  { int forced = get_tunable("gemm_deep_epilogue", -1); if (forced == 0) deep = 0; else if (forced == 1 && !a_mn_major && bn >= 128 && tma_store) deep = 1; }
  if (deep) {
    if (bn == 256 && b_mn_major) return launch_gemm<256, false, true, true>(ta, tb, tc, g, st);
    if (bn == 256) return launch_gemm<256, false, false, true>(ta, tb, tc, g, st);
    if (bn == 128 && b_mn_major) return launch_gemm<128, false, true, true>(ta, tb, tc, g, st);
    if (bn == 128) return launch_gemm<128, false, false, true>(ta, tb, tc, g, st);
  }
#define UNREAL_GEMM_CASE(BN_, AMN_, BMN_) \
  if (bn == BN_ && (a_mn_major != 0) == AMN_ && (b_mn_major != 0) == BMN_) return launch_gemm<BN_, AMN_, BMN_>(ta, tb, tc, g, st);
  UNREAL_GEMM_CASE(32, false, false)
  UNREAL_GEMM_CASE(64, false, false)
  UNREAL_GEMM_CASE(128, false, false)
  UNREAL_GEMM_CASE(256, false, false)
  UNREAL_GEMM_CASE(256, false, true)
  UNREAL_GEMM_CASE(256, true, false)
  UNREAL_GEMM_CASE(256, true, true)
  UNREAL_GEMM_CASE(64, false, true)
  UNREAL_GEMM_CASE(128, false, true)
  UNREAL_GEMM_CASE(32, true, false)
  UNREAL_GEMM_CASE(64, true, false)
  UNREAL_GEMM_CASE(128, true, false)
  UNREAL_GEMM_CASE(64, true, true)
  UNREAL_GEMM_CASE(128, true, true)
#undef UNREAL_GEMM_CASE
  set_error("unreal_gemm_bf16: no kernel for tile %d, a_mn %d, b_mn %d", bn, a_mn_major, b_mn_major);
  return UNREAL_EINVAL;
}
