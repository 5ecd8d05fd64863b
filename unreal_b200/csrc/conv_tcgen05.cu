// K7 convolutions (model/model.py:281-289: conv 8x8x3->16 stride 4, conv 4x4x16->32 stride 2, VALID,
// NHWC) as implicit GEMMs on tcgen05 with the im2col done by the TMA engine -- no patch matrix ever
// exists in memory.
//
// A stride-s KxK convolution with K = 2s is a 2x2 stride-1 convolution over the space-to-depth view
//     x'[Y, X, (dy, dx, c)] = x[s*Y + dy, s*X + dx, c]:
//     out[oy, ox, :] = sum over the four taps (by, bx) of  x'[oy+by, ox+bx, :] . Wtap[by, bx]
// so for one tap the GEMM A operand is just a shifted window of x':
//   conv1: x'' = x' as six 8-channel planes [S,6,441,8] bf16 (s2d_frames_kernel, or rendered directly by
//          K1's maze_s2d_kernel) is the UN-SWIZZLED K-major UMMA layout with a uniform 16-byte row
//          pitch.  One work item (5 output rows) bulk-copies its 6 x 126-row tile ONCE; each tap is the
//          same tile with the descriptor start address advanced by (by*21 + bx) rows
//          (conv1_fwd_tcgen05_kernel).  conv1_wgrad_tcgen05_kernel reads the same tiles as the MN-major
//          B operand of the filter gradient, with the masked dY as two 8-channel planes.
//   conv2: x' is only a VIEW of h1 [S,20,20,16]: for each dy a 4-D tensor map {32 (dx,c), 10 X, 10 Y, S}
//          based at row dy (TMA needs hierarchical strides, so dy cannot be a box dimension between
//          the channel run and X; measured with scripts/probes/tma5d_probe.cu) with box {32, 9, 9, 1}
//          lands 81 rows x 32 channels (one sample, half a tap) as 64-byte rows with the 64-byte
//          swizzle = a K-major UMMA SW64 tile as it lands (conv_fwd_tcgen05_kernel<32, 2>).
// Tap filters stay resident in shared memory for the whole (persistent) kernel.  Rows of the 128-row
// UMMA tile that a box does not cover hold stale data; they only produce accumulator rows that the
// row-clipped TMA store / the epilogue never writes.
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "maze_core.cuh"
#include "tc05.cuh"

namespace unreal {
using namespace tc05;

// Render-fused conv1 input (maze env type): the x'' tile of a work item (6 planes x 126 pixel rows x 16 B, rows
// rb*105.. of the 21x21 space-to-depth grid) is a pure function of the agent cell and the constant wall map --
// a 4x4 pixel block lies inside one 12-pixel maze cell, so each plane row is one of three constant 16-byte
// patterns (csrc/maze.cu:maze_s2d_kernel writes the same bytes to HBM).  One warp writes it straight into
// the stage the UMMA reads: the frame never exists in HBM, neither for the forward nor for the filter gradient.
__device__ __forceinline__ void maze_tile_to_smem(uint32_t dst, uint64_t walls49, int ax, int ay, int rb, int lane) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int p = lane + 32 * j;
    if (p < 126) {
      const int gp = rb * 105 + p;
      const int Y = gp / 21, X = gp - Y * 21;
      const int cx = X / 3, cy = Y / 3;
      const uint32_t mw = ((walls49 >> (cy * 7 + cx)) & 1ull) ? 0xffffffffu : 0u;
      const uint32_t ma = (cx == ax && cy == ay) ? 0xffffffffu : 0u;
#pragma unroll
      for (int q = 0; q < 6; ++q) {
        // element i of plane q is channel (8q + i) mod 3; walls set channel 0, the agent channel 1 (bf16 1.0 = 0x3f80)
        const int base = (2 * q) % 3;
        uint32_t v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int c0 = (base + 2 * k) % 3, c1 = (base + 2 * k + 1) % 3;
          const uint32_t wl = (c0 == 0 ? 0x3f80u : 0u) | (c1 == 0 ? 0x3f800000u : 0u);
          const uint32_t ag = (c0 == 1 ? 0x3f80u : 0u) | (c1 == 1 ? 0x3f800000u : 0u);
          v[k] = (wl & mw) | (ag & ma);
        }
        st_shared_v4(dst + (uint32_t)(q * 126 * 16 + p * 16), v[0], v[1], v[2], v[3]);
      }
    }
  }
}

constexpr int kConvThreads = 192;
constexpr int kConvAcc = 4;       // TMEM accumulator buffers of 32 columns
template <int MODE, int C = 16> struct ConvCfg;   // MODE 2 = conv2 (conv1 has its own single-copy kernel below)
template <int C> struct ConvCfg<2, C> {      // conv2: one step per filter row ky = 2by+dy; a box row is the 4 pixels
  // 2X..2X+3 of image row 2(Y+by)+dy = 64 (kx,c) K-columns = 128 bytes (rows of neighbouring X OVERLAP in
  // global memory: dim-1 stride 64 B under a 128-byte dim-0 extent; scripts/probes/tma_overlap_probe.cu), so a
  // sample is 4 boxes of 81 x 128 B instead of 8 of 81 x 64 B: half the TMA instructions, barrier round trips
  // and row requests.  A stage holds the 81 landed rows (88 = next multiple of the 8-row swizzle atom); the
  // 128-row UMMA reads on into the next stage, producing accumulator rows nobody stores.
  // C = 8 input channels (the pixel-control loss gradient without its 8 padding channels): 64-byte rows under the
  // 64-byte swizzle, two UMMAs per step, stages of 96 rows (a multiple of 1024 bytes) and twice as many of them.
  static_assert(C == 16 || C == 8, "conv2 geometry with 16 or 8 input channels");
  static constexpr int kSteps = 4, kRowBytes = 8 * C, kStageBytes = (C == 16 ? 88 : 96) * kRowBytes, kMmaPerStep = C / 4;
  static constexpr int kStages = C == 16 ? 6 : 12;  // 1.5 (3) samples in flight per CTA, two CTAs per SM
  static constexpr int kEpiWarps = 3;   // 81 rows: quarters 0..2 store
  // K-major UMMA descriptor high word: SBO (8 rows), version 1, swizzle mode (2: 128-byte, 4: 64-byte)
  static constexpr uint32_t kDescHi = C == 16 ? ((1024u >> 4) | (1u << 14) | (2u << 29)) : ((512u >> 4) | (1u << 14) | (4u << 29));
};

struct ConvArgs {
  const float* bias;
  int items;          // work items: one per sample
  int rows;           // valid GEMM rows per item: 81
  int box_bytes;      // bytes one A box delivers
  int mode;           // 2: conv2 over h1
  int relu;           // apply max(., 0) in the epilogue
  const float* scale; // nullable device scalar multiplied into the accumulators (the upstream gradient of a backward conv)
  const __nv_bfloat16* mask_y;   // MASKED build: [items][rows][N] activations of the layer the result is a gradient of
  float* db;                     // MASKED build: [rows][N] += the masked, rounded result summed over items (its bias gradient)
};

// MASKED: the result is the gradient w.r.t. a ReLU layer's output `mask_y` (pc_fc1 seen as [S,9,9,32] behind the pixel-control
// deconv): the epilogue zeroes it where mask_y <= 0 and sums the rounded values over items into db -- the ReLU-gradient /
// bias-gradient pass over the [S,2592] gradient (2.5 GB of traffic per update at 8192 envs) disappears.
// SPLIT (split-bf16 conv2, C = 16 only): tma_alo / tma_alo2 are the boxes of h1_lo, tma_wlo the filter residual; a stage
// holds the hi box then the lo box (two stages keep two CTAs per SM), the filters are resident as hi then lo, and every
// K step accumulates a_hi.w_hi + a_hi.w_lo + a_lo.w_hi.  Other builds ignore the three extra maps.
template <int N, int MODE, bool MASKED = false, int C = 16, bool SPLIT = false>   // N output channels: 32 (conv2, MODE 2); C input channels
__global__ void __launch_bounds__(kConvThreads, 2)
conv_fwd_tcgen05_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_a2,
                        const __grid_constant__ CUtensorMap tma_w, const __grid_constant__ CUtensorMap tma_c,
                        const ConvArgs g, const __grid_constant__ CUtensorMap tma_alo,
                        const __grid_constant__ CUtensorMap tma_alo2, const __grid_constant__ CUtensorMap tma_wlo) {
  using Cfg = ConvCfg<MODE, C>;
  static_assert(!SPLIT || (C == 16 && !MASKED), "split conv2: the encoder's geometry only");
  constexpr int kStages = SPLIT ? 2 : Cfg::kStages;
  constexpr int kStageBytes = SPLIT ? 2 * Cfg::kStageBytes : Cfg::kStageBytes;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  constexpr int kWTileBytes = N * Cfg::kRowBytes;          // one resident filter slice [N rows x kRowBytes]
  constexpr int kWBytes = (Cfg::kSteps * kWTileBytes + 1023) / 1024 * 1024;
  const uint32_t w_smem = smem_base;
  const uint32_t a_smem = smem_base + (SPLIT ? 2 : 1) * kWBytes;
  const uint32_t bar_base = a_smem + kStages * kStageBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kStages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * kStages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * kStages + kConvAcc + a); };
  const uint32_t w_bar = bar_base + 8u * (2 * kStages + 2 * kConvAcc);
  const uint32_t tmem_slot = bar_base + 8u * (2 * kStages + 2 * kConvAcc + 1);
  const uint32_t ebuf_base = bar_base + 1024u;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tma_a);
    prefetch_tensormap(&tma_a2);
    prefetch_tensormap(&tma_w);
    prefetch_tensormap(&tma_c);
    if constexpr (SPLIT) { prefetch_tensormap(&tma_alo); prefetch_tensormap(&tma_alo2); prefetch_tensormap(&tma_wlo); }
    for (int s = 0; s < kStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < kConvAcc; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4); }
    mbar_init(w_bar, 1);
    fence_mbar_init();
  } else if (warp == 2) {
    tmem_alloc<kConvAcc * 32>(tmem_slot);
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = tmem_base_at(tmem_slot);

  if (warp == 0) {
    if (lane == 0) {
      // ===== TMA producer: resident filter slices once, then one box per (item, step) =====
      mbar_arrive_expect_tx(w_bar, (SPLIT ? 2 : 1) * Cfg::kSteps * kWTileBytes);
#pragma unroll
      for (int t = 0; t < Cfg::kSteps; ++t) {
        tma_load_2d(w_smem + t * kWTileBytes, &tma_w, w_bar, t * (Cfg::kRowBytes / 2), 0);
        if constexpr (SPLIT) tma_load_2d(w_smem + kWBytes + t * kWTileBytes, &tma_wlo, w_bar, t * (Cfg::kRowBytes / 2), 0);
      }
      int stage = 0; uint32_t phase = 0;
      for (int it = blockIdx.x; it < g.items; it += gridDim.x) {
#pragma unroll 1
        for (int st = 0; st < Cfg::kSteps; ++st) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          mbar_arrive_expect_tx(full_bar(stage), (SPLIT ? 2 : 1) * g.box_bytes);
          const uint32_t dst = a_smem + stage * kStageBytes;
          const int by = st >> 1, dy = st & 1;
          tma_load_4d(dst, dy ? &tma_a2 : &tma_a, full_bar(stage), 0, 0, by, it);
          if constexpr (SPLIT) tma_load_4d(dst + Cfg::kStageBytes, dy ? &tma_alo2 : &tma_alo, full_bar(stage), 0, 0, by, it);
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===== MMA issuer: UMMA 128 x N x 16 over every step's K columns =====
      constexpr uint32_t idesc = idesc_bf16_f32(128, N, false, false);
      constexpr uint32_t kDescHiSw64 = Cfg::kDescHi;
      mbar_wait(w_bar, 0);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int it = blockIdx.x; it < g.items; it += gridDim.x) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        fence_after_sync();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * 32);
#pragma unroll
        for (int st = 0; st < Cfg::kSteps; ++st) {
          mbar_wait(full_bar(stage), phase);
          fence_after_sync();
          // SW64 K-major descriptors as (lo, hi) words: hi is constant (SBO 512 B, version 1, 64-byte swizzle),
          // lo = (address >> 4) | LBO field; one add per UMMA instead of rebuilding 64-bit descriptors
          const uint32_t a_lo = ((a_smem + stage * kStageBytes) >> 4) | (1u << 16);
          const uint32_t b_lo = ((w_smem + st * kWTileBytes) >> 4) | (1u << 16);
#pragma unroll
          for (int k = 0; k < Cfg::kMmaPerStep; ++k) {
            mma_f16_lohi(tmem_d, a_lo + 2u * k, kDescHiSw64, b_lo + 2u * k, kDescHiSw64, idesc, (st > 0 || k > 0) ? 1u : 0u);
            if constexpr (SPLIT) {
              mma_f16_lohi(tmem_d, a_lo + 2u * k, kDescHiSw64, b_lo + (uint32_t)(kWBytes >> 4) + 2u * k, kDescHiSw64, idesc, 1u);
              mma_f16_lohi(tmem_d, a_lo + (uint32_t)(Cfg::kStageBytes >> 4) + 2u * k, kDescHiSw64, b_lo + 2u * k, kDescHiSw64, idesc, 1u);
            }
          }
          mma_commit(empty_bar(stage));
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
        mma_commit(tfull_bar(acc));
        if (++acc == kConvAcc) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else {
    // ===== epilogue: bias + ReLU + bf16, staged per warp, TMA store clipped to the item's rows =====
    const int quarter = warp & 3;
    const uint32_t ebuf = ebuf_base + (uint32_t)(quarter < Cfg::kEpiWarps ? quarter : 0) * 8192u;
    uint32_t ebuf_it = 0;
    int acc = 0; uint32_t acc_phase = 0;
    float b[N];       // MASKED: the bias-gradient partial sums of this thread's row instead (the masked build has no bias)
#pragma unroll
    for (int j = 0; j < N; ++j) b[j] = (!MASKED && g.bias) ? __ldg(g.bias + j) : 0.f;
    const float sc = g.scale ? __ldg(g.scale) : 1.f;
    const int row = quarter * 32 + lane;
    const bool row_ok = row < g.rows;
    for (int it = blockIdx.x; it < g.items; it += gridDim.x) {
      uint4 yv[N / 8];
      if constexpr (MASKED) {       // the mask row, requested before the accumulator wait
        const uint4* ysrc = reinterpret_cast<const uint4*>(g.mask_y + ((int64_t)it * g.rows + (row_ok ? row : 0)) * N);
#pragma unroll
        for (int q = 0; q < N / 8; ++q) yv[q] = __ldg(ysrc + q);
      }
      mbar_wait(tfull_bar(acc), acc_phase);
      fence_after_sync();
      if (quarter * 32 < g.rows) {
        uint32_t r[32];
        tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * 32), r);
        tmem_ld_wait();
        const uint32_t buf = ebuf + (ebuf_it & 1u) * 4096u;
        ++ebuf_it;
        if (lane == 0) bulk_wait_read<1>();
        __syncwarp();
        const uint32_t rowp = buf + (uint32_t)lane * 128u;
#pragma unroll
        for (int q = 0; q < N / 8; ++q) {
          uint32_t pk[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if constexpr (MASKED) {
              const uint32_t yw = j == 0 ? yv[q].x : (j == 1 ? yv[q].y : (j == 2 ? yv[q].z : yv[q].w));
              const float2 yf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&yw));
              const float v0 = yf.x > 0.f ? __uint_as_float(r[8 * q + 2 * j]) * sc : 0.f;
              const float v1 = yf.y > 0.f ? __uint_as_float(r[8 * q + 2 * j + 1]) * sc : 0.f;
              __nv_bfloat162 p = __floats2bfloat162_rn(v0, v1);
              pk[j] = *reinterpret_cast<uint32_t*>(&p);
              if (row_ok) {                               // the bias gradient sums the ROUNDED values (as unreal_relu_grad does)
                const float2 f = __bfloat1622float2(p);
                b[8 * q + 2 * j] += f.x; b[8 * q + 2 * j + 1] += f.y;
              }
            } else {
              float v0 = __uint_as_float(r[8 * q + 2 * j]) * sc + b[8 * q + 2 * j];
              float v1 = __uint_as_float(r[8 * q + 2 * j + 1]) * sc + b[8 * q + 2 * j + 1];
              if (g.relu) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); }
              __nv_bfloat162 p = __floats2bfloat162_rn(v0, v1);
              pk[j] = *reinterpret_cast<uint32_t*>(&p);
            }
          }
          const uint32_t chunk = (uint32_t)q ^ (uint32_t)(lane & 7);
          st_shared_v4(rowp + chunk * 16u, pk[0], pk[1], pk[2], pk[3]);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_3d(&tma_c, buf, 0, quarter * 32, it);
          bulk_commit();
        }
      }
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
      if (++acc == kConvAcc) { acc = 0; acc_phase ^= 1u; }
    }
    if constexpr (MASKED) {
      if (row_ok && g.db != nullptr) {
#pragma unroll
        for (int j = 0; j < N; ++j) atomicAdd(g.db + row * N + j, b[j]);
      }
    }
    if (lane == 0) bulk_wait_all();
  }
  __syncwarp();
  fence_before_sync();
  __syncthreads();
  if (warp == 2) {
    fence_after_sync();
    tmem_dealloc<kConvAcc * 32>(tmem_base);
  }
}

// space-to-depth + bf16 conversion of frames: in [S,84,84,3] f32 / u8 (/255) -> x'' [S,6,441,8]
// (pixel (Y,X) = Y*21+X, channel dy*12 + dx*3 + c split into six 8-channel planes).  One thread per
// x' pixel: four 48-byte (f32) row pieces in, six coalesced 16-byte plane rows out.
// u8 frames: two adjacent bytes of a word -> (v0/255, v1/255) as correctly rounded float32 without a divide, like the u8
// pixel-change kernel (csrc/pixel_change84.cu: PRMT into the mantissa of 2^23, one FADD2, fma(v, hi, RN(v * lo)) on the
// packed fp32x2 pipe; exhaustively checked by unreal_selfcheck_arith) -- the kernel was instruction-bound on 48
// __fdiv_rn per thread (0.39 of HBM).  `magic` = 0x4B000000 arrives as a kernel parameter so the PRMT selectors stay immediates.
__device__ __forceinline__ float2 u8pair_to_f32x2(uint32_t word, int byte0, uint32_t magic) {
  float2 m;
  m.x = __uint_as_float(__byte_perm(word, magic, 0x7540u | (uint32_t)byte0));
  m.y = __uint_as_float(__byte_perm(word, magic, 0x7540u | (uint32_t)(byte0 + 1)));
  const float2 v = __fadd2_rn(m, make_float2(-8388608.0f, -8388608.0f));
  return __ffma2_rn(v, make_float2(0x1.010102p-8f, 0x1.010102p-8f),
                    __fmul2_rn(v, make_float2(-0x1.fdfdfep-33f, -0x1.fdfdfep-33f)));
}
__device__ __forceinline__ uint32_t u8pair_to_bf16x2(uint32_t word, int byte0, uint32_t magic) {
  const float2 q = u8pair_to_f32x2(word, byte0, magic);
  __nv_bfloat162 p2 = __floats2bfloat162_rn(q.x, q.y);
  return *reinterpret_cast<uint32_t*>(&p2);
}

// LO (split-bf16 encoder): also writes the residual planes out_lo = bf16(x - bf16(x)) in the same layout, so that
// hi + lo carries the frame to about 16 mantissa bits.
template <typename T, bool LO = false>
__global__ void __launch_bounds__(256) s2d_frames_kernel(const T* __restrict__ in, __nv_bfloat16* __restrict__ out,
                                                         int64_t total, uint32_t magic, __nv_bfloat16* __restrict__ out_lo) {
  for (int64_t id = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; id < total; id += (int64_t)gridDim.x * blockDim.x) {
    const int X = (int)(id % 21);
    const int Y = (int)((id / 21) % 21);
    const int64_t s = id / 441;
    const T* src = in + ((s * 84 + 4 * Y) * 84 + 4 * X) * 3;
    uint32_t pk[24];
    uint32_t pl[LO ? 24 : 1];
#pragma unroll
    for (int dy = 0; dy < 4; ++dy) {
      float v[12];
      if (sizeof(T) == 1 && !LO) {
        const uint32_t* p = reinterpret_cast<const uint32_t*>(src + dy * 252);   // 12 bytes, 4-byte aligned
#pragma unroll
        for (int w = 0; w < 3; ++w) {
          const uint32_t u = __ldcs(p + w);
          pk[dy * 6 + 2 * w] = u8pair_to_bf16x2(u, 0, magic);
          pk[dy * 6 + 2 * w + 1] = u8pair_to_bf16x2(u, 2, magic);
        }
        continue;
      }
      if (sizeof(T) == 4) {
        const float4* p = reinterpret_cast<const float4*>(src + dy * 252);
        const float4 a = __ldcs(p), b = __ldcs(p + 1), c = __ldcs(p + 2);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
        v[8] = c.x; v[9] = c.y; v[10] = c.z; v[11] = c.w;
      } else if (LO) {
        const uint32_t* p = reinterpret_cast<const uint32_t*>(src + dy * 252);   // 12 bytes, 4-byte aligned
#pragma unroll
        for (int w = 0; w < 3; ++w) {
          const uint32_t u = __ldcs(p + w);
          const float2 a = u8pair_to_f32x2(u, 0, magic), b = u8pair_to_f32x2(u, 2, magic);
          v[4 * w] = a.x; v[4 * w + 1] = a.y; v[4 * w + 2] = b.x; v[4 * w + 3] = b.y;
        }
      } else {
        const uint32_t* p = reinterpret_cast<const uint32_t*>(src + dy * 252);   // 12 bytes, 4-byte aligned
#pragma unroll
        for (int w = 0; w < 3; ++w) {
          const uint32_t u = __ldcs(p + w);
#pragma unroll
          for (int j = 0; j < 4; ++j) v[4 * w + j] = __fdiv_rn((float)((u >> (8 * j)) & 255u), 255.0f);
        }
      }
#pragma unroll
      for (int j = 0; j < 6; ++j) {
        __nv_bfloat162 p2 = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
        pk[dy * 6 + j] = *reinterpret_cast<uint32_t*>(&p2);
        if constexpr (LO) {
          const float2 h = __bfloat1622float2(p2);
          __nv_bfloat162 l2 = __floats2bfloat162_rn(v[2 * j] - h.x, v[2 * j + 1] - h.y);
          pl[dy * 6 + j] = *reinterpret_cast<uint32_t*>(&l2);
        }
      }
    }
    // plane-major: x'' [S][6 chunks of 8 channels][441 pixels][8]; consecutive threads (pixels) write
    // consecutive 16-byte rows of each plane
    const int pix = Y * 21 + X;
    uint4* dst = reinterpret_cast<uint4*>(out) + (s * 6) * 441 + pix;
#pragma unroll
    for (int j = 0; j < 6; ++j) dst[(int64_t)j * 441] = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
    if constexpr (LO) {
      uint4* dlo = reinterpret_cast<uint4*>(out_lo) + (s * 6) * 441 + pix;
#pragma unroll
      for (int j = 0; j < 6; ++j) dlo[(int64_t)j * 441] = make_uint4(pl[4 * j], pl[4 * j + 1], pl[4 * j + 2], pl[4 * j + 3]);
    }
  }
}

// ---- conv1, single-copy variant ----------------------------------------------------------------
// x'' is stored plane-major (8-channel chunks as separate [441 x 16 B] planes), which is exactly the
// un-swizzled K-major UMMA layout with a UNIFORM 16-byte row pitch.  One 3-D TMA box {8 ch, 126
// pixels (6 x' rows), 6 planes} per work item (5 output rows) lands once in shared memory and all four
// taps read it in place: tap (by,bx) is the same tile with the descriptor start address advanced by
// (by*21 + bx) rows.  GEMM rows follow the 21-wide x' grid (row m' = oy*21 + ox); the column ox = 20
// and rows >= 105 are garbage accumulator rows the epilogue skips.  HBM/L2 traffic per frame:
// 42 KB of x'' in (each byte once) + 12.8 KB of h1 out.
constexpr int kC1Stages = 6;      // x 12 KB; two CTAs per SM (each has ONE MMA-issuing thread, which is what bounds it)
constexpr int kC1Acc = 4;        // TMEM accumulator buffers (32 columns each): the MMA -> epilogue -> MMA hand-back
                                 // costs ~2 us of barrier latency per item, so 2 buffers capped the kernel
constexpr int kC1PlaneBytes = 126 * 16;
constexpr int kC1BoxBytes = 6 * kC1PlaneBytes;      // 12096
constexpr int kC1StageBytes = 12288;
constexpr int kC1WBytes = 4 * 6 * 16 * 16;          // [tap][chunk][16 out rows][8 ch] bf16
constexpr int kC1Smem = kC1WBytes + kC1Stages * kC1StageBytes + 1024 /*barriers*/ + 1024 /*tail reads*/ + 1024 /*align*/;
// SPLIT (split-bf16, "bf16x3"): operands a = a_hi + a_lo as two bf16 tensors; a stage holds the hi tile then the lo
// tile, the filters are resident as hi then lo, and a.b ~ a_hi.b_hi + a_hi.b_lo + a_lo.b_hi accumulates in the same
// TMEM columns (the a_lo.b_lo term is below fp32 rounding).  Four stages keep two CTAs per SM.
constexpr int kC1SplitStages = 4;
constexpr int kC1SplitSmem = 2 * kC1WBytes + kC1SplitStages * 2 * kC1StageBytes + 1024 + 1024 + 1024;

template <bool SPLIT>
__global__ void __launch_bounds__(kConvThreads, 2)
conv1_fwd_tcgen05_kernel(const __nv_bfloat16* __restrict__ xpp, const __nv_bfloat16* __restrict__ w_planes,
                         const float* __restrict__ bias, __nv_bfloat16* __restrict__ out, int items,
                         const int32_t* __restrict__ maze_pos, uint64_t walls49,
                         const __nv_bfloat16* __restrict__ xpp_lo, const __nv_bfloat16* __restrict__ w_planes_lo,
                         __nv_bfloat16* __restrict__ out_lo) {
  // SPLIT: xpp_lo may be NULL (input exactly bf16: rendered maze tiles, pre-converted planes): two passes instead of three
  constexpr int kStages = SPLIT ? kC1SplitStages : kC1Stages;
  constexpr int kStageBytes = SPLIT ? 2 * kC1StageBytes : kC1StageBytes;
  constexpr int kWB = SPLIT ? 2 * kC1WBytes : kC1WBytes;
  const bool has_lo = SPLIT && xpp_lo != nullptr;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t w_smem = smem_base;
  const uint32_t a_smem = smem_base + kWB;
  const uint32_t bar_base = a_smem + kStages * kStageBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kStages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * kStages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * kStages + kC1Acc + a); };
  const uint32_t w_bar = bar_base + 8u * (2 * kStages + 2 * kC1Acc);
  const uint32_t tmem_slot = bar_base + 8u * (2 * kStages + 2 * kC1Acc + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < kStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < kC1Acc; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4); }
    mbar_init(w_bar, 1);
    fence_mbar_init();
  } else if (warp == 2) {
    tmem_alloc<kC1Acc * 32>(tmem_slot);
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = tmem_base_at(tmem_slot);

  if (warp == 0 && maze_pos != nullptr) {
    // ===== render-fused producer (maze): the warp WRITES each item's x'' tile from the agent cell =====
    if (lane == 0) {
      mbar_arrive_expect_tx(w_bar, kWB);
      bulk_load(w_smem, w_planes, kC1WBytes, w_bar);
      if constexpr (SPLIT)
        bulk_load(w_smem + kC1WBytes, w_planes_lo, kC1WBytes, w_bar);
    }
    int stage = 0; uint32_t phase = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int2 cell = __ldg(reinterpret_cast<const int2*>(maze_pos) + (it >> 2));
      mbar_wait(empty_bar(stage), phase ^ 1u);
      maze_tile_to_smem(a_smem + stage * kStageBytes, walls49, cell.x, cell.y, it & 3, lane);
      fence_proxy_async_smem();            // generic-proxy writes -> visible to the tensor core's async-proxy reads
      __syncwarp();
      if (lane == 0) mbar_arrive(full_bar(stage));
      if (++stage == kStages) { stage = 0; phase ^= 1u; }
    }
  } else if (warp == 0) {
    if (lane == 0) {
      // ===== producer: resident filters (one bulk copy), then ONE box per item =====
      mbar_arrive_expect_tx(w_bar, kWB);
      bulk_load(w_smem, w_planes, kC1WBytes, w_bar);
      if constexpr (SPLIT)
        bulk_load(w_smem + kC1WBytes, w_planes_lo, kC1WBytes, w_bar);
      int stage = 0; uint32_t phase = 0;
      for (int it = blockIdx.x; it < items; it += gridDim.x) {
        mbar_wait(empty_bar(stage), phase ^ 1u);
        mbar_arrive_expect_tx(full_bar(stage), has_lo ? 2 * kC1BoxBytes : kC1BoxBytes);
        // each plane's 126 pixel rows are 2016 contiguous bytes in x'': six 1-D bulk copies (a tensor
        // box with a 16-byte inner dimension costs the TMA engine one request per row: measured 2.3x slower)
        const uint8_t* src = reinterpret_cast<const uint8_t*>(xpp) + ((int64_t)(it >> 2) * 6 * 441 + (it & 3) * 105) * 16;
        const uint32_t dst = a_smem + stage * kStageBytes;
#pragma unroll
        for (int q = 0; q < 6; ++q)
          bulk_load(dst + q * kC1PlaneBytes, src + (int64_t)q * 441 * 16, kC1PlaneBytes, full_bar(stage));
        if (has_lo) {
          const uint8_t* src_lo = reinterpret_cast<const uint8_t*>(xpp_lo) + (src - reinterpret_cast<const uint8_t*>(xpp));
#pragma unroll
          for (int q = 0; q < 6; ++q)
            bulk_load(dst + kC1StageBytes + q * kC1PlaneBytes, src_lo + (int64_t)q * 441 * 16, kC1PlaneBytes, full_bar(stage));
        }
        if (++stage == kStages) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===== MMA issuer: 4 taps x 3 UMMA (128 x 16 x 16) on the one resident tile =====
      constexpr uint32_t idesc = idesc_bf16_f32(128, 16, false, false);
      constexpr uint32_t desc_hi = (128u >> 4) | (1u << 14);        // SBO = 128 B, descriptor version 1, no swizzle
      const uint32_t w_lo0 = (w_smem >> 4) | ((256u >> 4) << 16);  // filter tiles: LBO = 256 B
      mbar_wait(w_bar, 0);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int it = blockIdx.x; it < items; it += gridDim.x) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        mbar_wait(full_bar(stage), phase);
        fence_after_sync();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * 32);
        // descriptor low words: (address >> 4) | LBO field; every offset below is a multiple of 16 bytes
        const uint32_t a_lo0 = ((a_smem + stage * kStageBytes) >> 4) | ((uint32_t)(kC1PlaneBytes >> 4) << 16);
#pragma unroll
        for (int tap = 0; tap < 4; ++tap) {
          const uint32_t shift16 = (uint32_t)((tap >> 1) * 21 + (tap & 1));
#pragma unroll
          for (int j = 0; j < 3; ++j) {
            const uint32_t a = a_lo0 + (uint32_t)(2 * j * kC1PlaneBytes >> 4) + shift16;
            const uint32_t w = w_lo0 + (uint32_t)((tap * 1536 + 2 * j * 256) >> 4);
            mma_f16_lohi(tmem_d, a, desc_hi, w, desc_hi, idesc, (tap > 0 || j > 0) ? 1u : 0u);
            if constexpr (SPLIT) {
              mma_f16_lohi(tmem_d, a, desc_hi, w + (uint32_t)(kC1WBytes >> 4), desc_hi, idesc, 1u);        // a_hi . w_lo
              if (has_lo) mma_f16_lohi(tmem_d, a + (uint32_t)(kC1StageBytes >> 4), desc_hi, w, desc_hi, idesc, 1u);  // a_lo . w_hi
            }
          }
        }
        mma_commit(empty_bar(stage));
        mma_commit(tfull_bar(acc));
        if (++stage == kStages) { stage = 0; phase ^= 1u; }
        if (++acc == kC1Acc) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else {
    // ===== epilogue: bias + ReLU + bf16; row m' = oy*21 + ox -> h1[(item*5 + oy), ox, 0..15] =====
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const int oyl = r / 21, ox = r - oyl * 21;
    const bool valid = r < 105 && ox < 20;
    int acc = 0; uint32_t acc_phase = 0;
    float b[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) b[j] = bias ? __ldg(bias + j) : 0.f;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      mbar_wait(tfull_bar(acc), acc_phase);
      fence_after_sync();
      uint32_t v[32];
      tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * 32), v);
      tmem_ld_wait();
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
      if (valid) {
        uint32_t pk[8], pl[SPLIT ? 8 : 1];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float f0 = fmaxf(__uint_as_float(v[2 * j]) + b[2 * j], 0.f), f1 = fmaxf(__uint_as_float(v[2 * j + 1]) + b[2 * j + 1], 0.f);
          __nv_bfloat162 p = __floats2bfloat162_rn(f0, f1);
          pk[j] = *reinterpret_cast<uint32_t*>(&p);
          if constexpr (SPLIT) {          // h1 = hi + lo: the residual of the rounding as a second bf16
            const float2 h = __bfloat1622float2(p);
            __nv_bfloat162 l = __floats2bfloat162_rn(f0 - h.x, f1 - h.y);
            pl[j] = *reinterpret_cast<uint32_t*>(&l);
          }
        }
        const int64_t o = ((int64_t)it * 100 + oyl * 20 + ox) * 16;
        uint4* dst = reinterpret_cast<uint4*>(out + o);
        dst[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        dst[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
        if constexpr (SPLIT) {
          uint4* dlo = reinterpret_cast<uint4*>(out_lo + o);
          dlo[0] = make_uint4(pl[0], pl[1], pl[2], pl[3]);
          dlo[1] = make_uint4(pl[4], pl[5], pl[6], pl[7]);
        }
      }
      if (++acc == kC1Acc) { acc = 0; acc_phase ^= 1u; }
    }
  }
  __syncwarp();
  fence_before_sync();
  __syncthreads();
  if (warp == 2) {
    fence_after_sync();
    tmem_dealloc<kC1Acc * 32>(tmem_base);
  }
}


// ---- conv1 weight gradient, fused ---------------------------------------------------------------
// dW[tap][o][(dy,dx,c)] = sum over samples and output pixels of dY[pix, o] * x'[pix + shift(tap), (dy,dx,c)]
// -- the reduction runs over PIXELS, so both operands are "MN-major" for the tensor core and the same
// plane-major tiles serve again: x'' planes are the A operand (M = 48 channels = 6 chunks of the 16 a
// 128-row UMMA reads, rows at a 16-byte pitch, tap = start address shift), dY planes [2][S*400][8]
// (written by unreal_conv2_dgrad_relu / unreal_relu_grad) are the B operand (N = 16 outputs = 2 chunks).  One work item = 5 output rows = 112 grid rows (K): rows with ox = 20 and rows >= 105
// are zero in the dY tile (zero-initialised once; bulk copies only ever write the twenty real rows
// of each output row), so whatever finite data x'' holds there contributes nothing.  Each CTA keeps
// its four [48 x 16] accumulators in TMEM across ALL its items and adds them to global once.
// Traffic per frame: 42 KB of x'' + 12.8 KB of dY, each read once; no patch matrix.
// The four taps share ONE x'' tile and differ only by a pixel shift; instead of shifting A (four UMMAs per K step,
// each re-reading 2 KB of x'' from shared memory -- the tensor core's operand fetch was 90 % busy at 30 % math,
// profiles/r1_conv_s3_kernels_summary.txt) the dY tile is landed FOUR times, plane (tap, half) at row offset
// shift(tap): B[q, (tap,o)] = dY[q - shift(tap), o], N = 64, and one UMMA per K step reads x'' once.
constexpr int kWgStages = 2;      // three CTAs per SM (58 KB and 64 TMEM columns each)
constexpr int kWgStageBytes = 28672;            // x'' tile 12 096 (+192 pad) | dY: 4 taps x 2 halves x 128 rows x 16 B
constexpr int kWgDyOff = 12288;
constexpr int kWgDyPlane = 128 * 16;
constexpr int kWgTail = 0;
constexpr int kWgSmem = kWgStages * kWgStageBytes + kWgTail + 1024 + 1024;

__global__ void __launch_bounds__(96, 3)
conv1_wgrad_tcgen05_kernel(const __nv_bfloat16* __restrict__ xpp, const __nv_bfloat16* __restrict__ dyp,
                           float* __restrict__ dw, int items, int64_t dy_plane_elems, int pitch21,
                           const int32_t* __restrict__ maze_pos, uint64_t walls49) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + kWgStages * kWgStageBytes + kWgTail;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kWgStages + s); };
  const uint32_t done_bar = bar_base + 8u * (2 * kWgStages);
  const uint32_t tmem_slot = bar_base + 8u * (2 * kWgStages + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // zero every tile byte once: padding rows of the x'' tiles and the never-written rows of the dY tiles
  for (uint32_t off = threadIdx.x * 16u; off < (uint32_t)(kWgStages * kWgStageBytes + kWgTail); off += 96u * 16u)
    st_shared_v4(smem_base + off, 0u, 0u, 0u, 0u);
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < kWgStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    mbar_init(done_bar, 1);
    fence_mbar_init();
  } else if (warp == 2) {
    tmem_alloc<64>(tmem_slot);
  }
  fence_proxy_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = tmem_base_at(tmem_slot);

  if (warp == 0 && maze_pos != nullptr) {
    // ===== render-fused producer (maze): the x'' tile is written by the warp, only dY comes from HBM =====
    int stage = 0; uint32_t phase = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int64_t smp = it >> 2;
      const int rb = it & 3;
      const int2 cell = __ldg(reinterpret_cast<const int2*>(maze_pos) + smp);
      mbar_wait(empty_bar(stage), phase ^ 1u);
      const uint32_t dst = smem_base + stage * kWgStageBytes;
      maze_tile_to_smem(dst, walls49, cell.x, cell.y, rb, lane);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive_expect_tx(full_bar(stage), 8 * 1680);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const uint8_t* ds = reinterpret_cast<const uint8_t*>(dyp) + ((int64_t)c * dy_plane_elems / 8 + smp * 420 + rb * 105) * 16;
#pragma unroll
          for (int t = 0; t < 4; ++t)
            bulk_load(dst + kWgDyOff + (t * 2 + c) * kWgDyPlane + ((t >> 1) * 21 + (t & 1)) * 16, ds, 1680, full_bar(stage));
        }
      }
      if (++stage == kWgStages) { stage = 0; phase ^= 1u; }
    }
  } else if (warp == 0) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int it = blockIdx.x; it < items; it += gridDim.x) {
        mbar_wait(empty_bar(stage), phase ^ 1u);
        mbar_arrive_expect_tx(full_bar(stage), kC1BoxBytes + (pitch21 ? 8 * 1680 : 40 * 320));
        const int64_t smp = it >> 2;
        const int rb = it & 3;
        const uint32_t dst = smem_base + stage * kWgStageBytes;
        const uint8_t* xs = reinterpret_cast<const uint8_t*>(xpp) + (smp * 6 * 441 + rb * 105) * 16;
#pragma unroll
        for (int q = 0; q < 6; ++q)
          bulk_load(dst + q * kC1PlaneBytes, xs + (int64_t)q * 441 * 16, kC1PlaneBytes, full_bar(stage));
        if (pitch21) {
          // planes already on the x'' grid's 21-pixel row pitch (column 20 zero): ONE 1680-byte copy per plane
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            const uint8_t* ds = reinterpret_cast<const uint8_t*>(dyp) + ((int64_t)c * dy_plane_elems / 8 + smp * 420 + rb * 105) * 16;
#pragma unroll
            for (int t = 0; t < 4; ++t)
              bulk_load(dst + kWgDyOff + (t * 2 + c) * kWgDyPlane + ((t >> 1) * 21 + (t & 1)) * 16, ds, 1680, full_bar(stage));
          }
        } else {
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            const uint8_t* ds = reinterpret_cast<const uint8_t*>(dyp) + ((int64_t)c * dy_plane_elems / 8 + smp * 400 + rb * 100) * 16;
#pragma unroll 1
            for (int t = 0; t < 4; ++t)
#pragma unroll
              for (int oyl = 0; oyl < 5; ++oyl)
                bulk_load(dst + kWgDyOff + (t * 2 + c) * kWgDyPlane + ((t >> 1) * 21 + (t & 1) + oyl * 21) * 16, ds + oyl * 320,
                          320, full_bar(stage));
          }
        }
        if (++stage == kWgStages) { stage = 0; phase ^= 1u; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0) {
      // x'' is the A operand (M = (dy,dx,c) channels: 6 real 8-channel chunks of the 16 a 128-row UMMA reads, the
      // rest land in accumulator rows nobody reads), dY the B operand (N = 16 outputs): a UMMA costs
      // max(M,128) * N / 256 cycles, so N = 16 is a third of the tensor-pipe time of the transposed form (N = 48)
      // M = 64, not 128: the MN-major A operand is read from shared memory chunk by chunk, and at 128 B/clk a
      // 128-row read (16 chunks x 16 pixels x 16 B = 4 KB per UMMA, 10 of the 16 chunks garbage) is what bounds
      // the kernel; 64 rows (6 real chunks of 8) halve it
      // N = 64 = (tap, o): the four shifted dY copies are the 8 chunks of ONE B operand
      constexpr uint32_t idesc = idesc_bf16_f32(64, 64, true, true);
      int stage = 0; uint32_t phase = 0;
      bool first = true;
      for (int it = blockIdx.x; it < items; it += gridDim.x) {
        mbar_wait(full_bar(stage), phase);
        fence_after_sync();
        const uint32_t sx = smem_base + stage * kWgStageBytes, sd = sx + kWgDyOff;
        // MN-major un-swizzled descriptors: LBO = 128 B (next 8 pixel rows), SBO = plane stride
        const uint32_t a_lo0 = (sx >> 4) | ((128u >> 4) << 16), b_lo0 = (sd >> 4) | ((128u >> 4) << 16);
        constexpr uint32_t a_hi = ((uint32_t)kC1PlaneBytes >> 4) | (1u << 14), b_hi = ((uint32_t)kWgDyPlane >> 4) | (1u << 14);
        // K = 128 grid rows: x'' rows 0..125 (+2 zero pad rows) against dY rows shifted by up to 22
#pragma unroll
        for (int ks = 0; ks < 8; ++ks)
          mma_f16_lohi(tmem_base, a_lo0 + (uint32_t)(ks * 16), a_hi, b_lo0 + (uint32_t)(ks * 16), b_hi, idesc,
                       (first && ks == 0) ? 0u : 1u);
        first = false;
        mma_commit(empty_bar(stage));
        if (++stage == kWgStages) { stage = 0; phase ^= 1u; }
      }
      mma_commit(done_bar);
    }
    __syncwarp();
  }
  {
    // ===== final epilogue: a 64-row accumulator keeps row m = (dy,dx,c) in lane 32*(m/16) + m%16, i.e. 16 rows in
    // each warp's TMEM sub-partition (warps 0..2: m = 0..47; rows 48..63 are the garbage chunks), columns t*16 + o =====
    mbar_wait(done_bar, 0);
    fence_after_sync();
    const int m = warp * 16 + lane;
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
      uint32_t v[32];
      tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(half * 32), v);     // taps 2*half, 2*half+1
      tmem_ld_wait();
      if (lane < 16) {
#pragma unroll
        for (int j = 0; j < 32; ++j) atomicAdd(dw + ((2 * half) * 16 + j) * 48 + m, __uint_as_float(v[j]));
      }
    }
  }
  __syncwarp();
  fence_before_sync();
  __syncthreads();
  if (warp == 2) {
    fence_after_sync();
    tmem_dealloc<64>(tmem_base);
  }
}


// ---- conv2 weight gradient, fused ---------------------------------------------------------------
// dW2[ky][(kx,c), o] = sum over samples and output pixels of h1box[pix, (kx,c)] * dY2[pix, o]:
// the SAME four 4-D TMA boxes per sample as the forward kernel (81 overlapping rows x 128 B, 128-byte
// swizzle) are now the MN-major A operand (M = 64 (kx,c) values, K = pixels), the sample's masked dY2 [81, 32]
// lands through a 3-D box of 96 rows (rows 81..95 are out of bounds = TMA zero fill) as the MN-major
// B operand.  Tile rows the boxes never write were zeroed once, so K rows 81..95 contribute exactly 0.
// Four [64 x 32] accumulators live in TMEM across ALL samples of a CTA and are added to global
// once.  Replaces unreal_im2col (41 KB per sample written and re-read) + the split-K GEMM.
// C = 8 (the pixel-control head's filter gradient, the loss gradient [S,400,8] in the activation's role): 64-byte A rows under
// the 64-byte swizzle = 32 (kx,c) values; the 64-row UMMA's second 32-row chunk (LBO) reads the next stage and lands in
// accumulator rows nobody stores.
template <int C> struct W2Cfg {
  static constexpr int kAStages = C == 16 ? 6 : 10;   // 1.5 (2.5) samples in flight per CTA, two CTAs per SM
  static constexpr int kBStages = C == 16 ? 3 : 4;
  static constexpr int kABytes = 96 * 8 * C;          // 81 landed rows of 128 (64) B (+ rows the zero dY rows cancel)
  static constexpr int kBBytes = 8192;                // 96 rows x 64 B used
  static constexpr int kTail = kABytes;               // the ignored A rows 64..127 of the last stage read here
  static constexpr int kSmem = kAStages * kABytes + kBStages * kBBytes + kTail + 1024 + 1024;
};

template <int C>
__global__ void __launch_bounds__(128, 2)
conv2_wgrad_tcgen05_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_a2,
                           const __grid_constant__ CUtensorMap tma_dy, float* __restrict__ dw, int samples) {
  constexpr int kW2AStages = W2Cfg<C>::kAStages, kW2BStages = W2Cfg<C>::kBStages, kW2ABytes = W2Cfg<C>::kABytes,
                kW2BBytes = W2Cfg<C>::kBBytes, kW2Tail = W2Cfg<C>::kTail;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t a_smem = smem_base;
  const uint32_t b_smem = a_smem + kW2AStages * kW2ABytes;
  const uint32_t bar_base = b_smem + kW2BStages * kW2BBytes + kW2Tail;
  auto fullA = [&](int s) { return bar_base + 8u * s; };
  auto emptyA = [&](int s) { return bar_base + 8u * (kW2AStages + s); };
  auto fullB = [&](int s) { return bar_base + 8u * (2 * kW2AStages + s); };
  auto emptyB = [&](int s) { return bar_base + 8u * (2 * kW2AStages + kW2BStages + s); };
  const uint32_t done_bar = bar_base + 8u * (2 * kW2AStages + 2 * kW2BStages);
  const uint32_t tmem_slot = done_bar + 8u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  for (uint32_t off = threadIdx.x * 16u; off < (uint32_t)(kW2AStages * kW2ABytes + kW2BStages * kW2BBytes + kW2Tail); off += 128u * 16u)
    st_shared_v4(smem_base + off, 0u, 0u, 0u, 0u);
  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tma_a); prefetch_tensormap(&tma_a2); prefetch_tensormap(&tma_dy);
    for (int s = 0; s < kW2AStages; ++s) { mbar_init(fullA(s), 1); mbar_init(emptyA(s), 1); }
    for (int s = 0; s < kW2BStages; ++s) { mbar_init(fullB(s), 1); mbar_init(emptyB(s), 1); }
    mbar_init(done_bar, 1);
    fence_mbar_init();
  } else if (warp == 2) {
    tmem_alloc<256>(tmem_slot);
  }
  fence_proxy_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = tmem_base_at(tmem_slot);

  if (warp == 0) {
    if (lane == 0) {
      int sa = 0; uint32_t pa = 0; int sb = 0; uint32_t pb = 0;
      for (int it = blockIdx.x; it < samples; it += gridDim.x) {
        mbar_wait(emptyB(sb), pb ^ 1u);
        mbar_arrive_expect_tx(fullB(sb), 96 * 64);
        tma_load_3d(b_smem + sb * kW2BBytes, &tma_dy, fullB(sb), 0, 0, it);
        if (++sb == kW2BStages) { sb = 0; pb ^= 1u; }
#pragma unroll 1
        for (int st = 0; st < 4; ++st) {          // st = filter row ky = 2by + dy
          const int by = st >> 1, dy = st & 1;
          mbar_wait(emptyA(sa), pa ^ 1u);
          mbar_arrive_expect_tx(fullA(sa), 4 * C * 9 * 9 * 2);
          tma_load_4d(a_smem + sa * kW2ABytes, dy ? &tma_a2 : &tma_a, fullA(sa), 0, 0, by, it);
          if (++sa == kW2AStages) { sa = 0; pa ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = idesc_bf16_f32(64, 32, true, true);   // 64 rows: all of them real, half the A read
      // MN-major descriptors.  A (h1 box, 128-byte rows, SW128): lo = (addr >> 4) | LBO (stride of the next
      // 64-element M chunk; only the first chunk is real, the second reads the next stage / the tail),
      // hi = SBO 1024 B (next 8 pixel rows).  B (dY2, 64-byte rows, SW64): SBO 512 B.
      constexpr uint32_t hi = (512u >> 4) | (1u << 14) | (4u << 29);
      constexpr uint32_t hi_a = C == 16 ? ((1024u >> 4) | (1u << 14) | (2u << 29)) : hi;
      constexpr uint32_t kAStep = C == 16 ? 128u : 64u;     // 16 pixel rows of A in 16-byte units
      int sa = 0; uint32_t pa = 0; int sb = 0; uint32_t pb = 0;
      bool first = true;
      for (int it = blockIdx.x; it < samples; it += gridDim.x) {
        mbar_wait(fullB(sb), pb);
        const uint32_t b_lo = ((b_smem + sb * kW2BBytes) >> 4) | ((64u >> 4) << 16);
#pragma unroll 1
        for (int st = 0; st < 4; ++st) {
          mbar_wait(fullA(sa), pa);
          fence_after_sync();
          const uint32_t a_lo = ((a_smem + sa * kW2ABytes) >> 4) | (((uint32_t)kW2ABytes >> 4) << 16);
#pragma unroll
          for (int ks = 0; ks < 6; ++ks)
            mma_f16_lohi(tmem_base + (uint32_t)(st * 32), a_lo + (uint32_t)ks * kAStep, hi_a, b_lo + (uint32_t)(ks * 64), hi, idesc,
                         (first && ks == 0) ? 0u : 1u);
          mma_commit(emptyA(sa));
          if (++sa == kW2AStages) { sa = 0; pa ^= 1u; }
        }
        first = false;
        mma_commit(emptyB(sb));
        if (++sb == kW2BStages) { sb = 0; pb ^= 1u; }
      }
      mma_commit(done_bar);
    }
    __syncwarp();
  }
  {
    // ===== final epilogue: accumulator ky, row m = (kx,c) of a 64-row accumulator in TMEM lane 32*(m/16) + m%16
    // (16 rows in each of the four warps' sub-partitions), column o -> dW2 in HWIO order [ky][(kx,c)][o] =====
    mbar_wait(done_bar, 0);
    fence_after_sync();
    const int m = warp * 16 + lane;
#pragma unroll 1
    for (int st = 0; st < 4; ++st) {
      uint32_t v[32];
      tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(st * 32), v);
      tmem_ld_wait();
      float* o = dw + (st * (4 * C) + m) * 32;
      if (lane < 16 && m < 4 * C) {
        // 128-bit reductions: 296 CTAs add their 32 KB of partial filters to the same 8192 addresses, and 32 scalar atomics per
        // thread kept the LSU queue full (ncu: lg_throttle 5.7 stalled warps per issue at the end of the kernel)
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          red_add_v4(o + j, __uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
      }
    }
  }
  __syncwarp();
  fence_before_sync();
  __syncthreads();
  if (warp == 2) {
    fence_after_sync();
    tmem_dealloc<256>(tmem_base);
  }
}


// ---- conv2 input gradient (transposed convolution), fused -----------------------------------------
// dh1[y, x, c] = sum over taps of dY2[(y-ky)/2, (x-kx)/2, :] . W2[ky, kx, c, :].  In the space-to-depth
// view (y = 2Y+dy, ky = 2by+dy ...) this is again a 2x2 tap sum over a 10x10 grid:
//     dh1'[(Y,X), (dy,dx,c)] = sum_{by,bx} dY2pad[(Y-by, X-bx), :] . Wd[(by,bx)][(dy,dx,c), :]
// and the zero padding is free: a 4-D TMA box {32 o, 10 X, 10 Y, 1} over dY2 [S,9,9,32] at the SIGNED
// coordinates (0, -bx, -by, s) zero-fills everything outside the 9x9 image.  Each box lands as a
// 100-row K-major SW64 tile (K = 32 outputs), the four [64 x 32] tap filters stay resident, and the
// epilogue writes the [100 x 64] tile straight into the dense [S,20,20,16] gradient (each thread owns
// a 2x2 pixel block = two contiguous 64-byte runs).  Replaces the GEMM that materialised
// [S*81, 256] columns (41 KB per sample) plus unreal_col2im.
constexpr int kDgStages = 8;      // two CTAs per SM
constexpr int kDgAcc = 4;                          // 64 TMEM columns each
constexpr int kDgABytes = 128 * 64;
constexpr int kDgWBytes = 4 * 64 * 64;             // four tap filters [64 rows x 64 B]
constexpr int kDgSmem = kDgWBytes + kDgStages * kDgABytes + 1024 + 1024;

// CO = 16: conv2's input gradient, bf16 out.  CO = 8: the pixel-control head's merged deconv FORWARD
// (model.py:418-430: the same 4x4 stride-2 VALID transposed convolution [S,9,9,32] -> [S,20,20,8], filter
// [kh,kw,out,in] = conv2's HWIO with c = out): N = 32 accumulator columns, epilogue adds the bias, applies
// ReLU and writes f32 -- replaces a GEMM into 41 KB/sample of f32 columns + col2im.
// CO = 8 with `pl.target` set: the pixel-control head's loss FUSED into the deconv's epilogue (model.py:431-441 dueling
// combine + Q(a) gather, :531-546 lambda * 0.5 * sum (R - Q_a)^2).  A thread holds all 8 channels of its 2x2 pixels, so
// it finishes the loss and writes d loss / d (pre-ReLU output) straight as conv2-geometry input [S,400,16] bf16
// (channels 8..15 zero; un-scaled by the upstream gradient, which the backward convolutions apply) plus the bias
// gradient -- the f32 head output [S,20,20,8] (2.1 GB at 8192 envs x 20) is never written, nor read back twice.
struct PcLossArgs {
  const int32_t* act;     // [S]
  const float* target;    // [S,20,20]
  const float* mask;      // [S]
  double* loss;           // += lam * 0.5 * sum mask (target - Q[act])^2
  int a;                  // number of actions
  float lam;
  float* qmax;            // set (with target == NULL): write only max_a Q [S,20,20] (run_pc_q_max, model.py:707-712)
  int c8;                 // loss gradient as [S,400,8] (the real channels only) instead of conv2's [S,400,16] with zero padding;
                          // 2: as four parity planes [S][4 (dy,dx)][100 (Y,X)][8] (pc_planes_*_tcgen05_kernel's tile)
};

// PC (CO = 16 only): the same loss (or the q-max map) for the 16-channel head of 8..15 actions -- channel 0 the value,
// 1..A the advantages.  The thread holds all 16 channels of its pixels and writes the loss gradient as [S,400,16] with
// every channel real; the bias gradient is db [16].
// EPI = 8 (CO = 8, or PC): two epilogue warps per TMEM lane quarter, one per output-row parity dy (16 accumulator columns
// each; 32 with PC).  The loss epilogue is a chain of dependent instructions per pixel on ONE warp per scheduler (ncu of the 4-warp
// build, profiles/r2_conv2_bwd_20480samples_ncu_summary.txt: issue slots 39 % active, DRAM 29 %, tensor pipe 7 %, nothing
// saturated); twice the warps hide twice the latency.
template <int CO, int EPI = 4, int NA = 0, bool PC = false>   // NA: the pixel-control loss's action count when known at compile time (0: run time)
__global__ void __launch_bounds__(64 + 32 * EPI, 2)
conv2_dgrad_tcgen05_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_w,
                           void* __restrict__ out_raw, const float* __restrict__ bias, int samples,
                           const __nv_bfloat16* __restrict__ mask_y, float* __restrict__ db, int pitch21,
                           const PcLossArgs pl) {
  constexpr int kN = 4 * CO;                         // (dy, dx, c) accumulator columns
  constexpr int kTapBytes = kN * 64;                 // one resident tap filter [kN rows x 64 B]
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t w_smem = smem_base;
  const uint32_t a_smem = smem_base + kDgWBytes;
  const uint32_t bar_base = a_smem + kDgStages * kDgABytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kDgStages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * kDgStages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * kDgStages + kDgAcc + a); };
  const uint32_t w_bar = bar_base + 8u * (2 * kDgStages + 2 * kDgAcc);
  const uint32_t tmem_slot = w_bar + 8u;
  // PC: the 16 bias values in the barrier block's spare bytes (in registers they push the EPI = 8 epilogue into spills)
  float* s_bias = reinterpret_cast<float*>(smem_raw + (bar_base + 512u - smem_u32(smem_raw)));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tma_a); prefetch_tensormap(&tma_w);
    for (int s = 0; s < kDgStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < kDgAcc; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), EPI); }
    mbar_init(w_bar, 1);
    fence_mbar_init();
  } else if (warp == 2) {
    tmem_alloc<kDgAcc * 64>(tmem_slot);
  } else if (PC && warp == 3 && lane < 16) {
    s_bias[lane] = __ldg(bias + lane);
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = tmem_base_at(tmem_slot);

  if (warp == 0) {
    if (lane == 0) {
      mbar_arrive_expect_tx(w_bar, 4 * kTapBytes);
#pragma unroll
      for (int t = 0; t < 4; ++t) tma_load_2d(w_smem + t * kTapBytes, &tma_w, w_bar, 0, t * kN);
      int stage = 0; uint32_t phase = 0;
      for (int it = blockIdx.x; it < samples; it += gridDim.x) {
#pragma unroll 1
        for (int tap = 0; tap < 4; ++tap) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          mbar_arrive_expect_tx(full_bar(stage), 32 * 10 * 10 * 2);
          tma_load_4d(a_smem + stage * kDgABytes, &tma_a, full_bar(stage), 0, -(tap & 1), -(tap >> 1), it);
          if (++stage == kDgStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = idesc_bf16_f32(128, kN, false, false);
      constexpr uint32_t hi = (512u >> 4) | (1u << 14) | (4u << 29);     // K-major SW64
      mbar_wait(w_bar, 0);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int it = blockIdx.x; it < samples; it += gridDim.x) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        fence_after_sync();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * 64);
#pragma unroll
        for (int tap = 0; tap < 4; ++tap) {
          mbar_wait(full_bar(stage), phase);
          fence_after_sync();
          const uint32_t a_lo = ((a_smem + stage * kDgABytes) >> 4) | (1u << 16);
          const uint32_t b_lo = ((w_smem + tap * kTapBytes) >> 4) | (1u << 16);
#pragma unroll
          for (int k = 0; k < 2; ++k)
            mma_f16_lohi(tmem_d, a_lo + 2u * k, hi, b_lo + 2u * k, hi, idesc, (tap > 0 || k > 0) ? 1u : 0u);
          mma_commit(empty_bar(stage));
          if (++stage == kDgStages) { stage = 0; phase ^= 1u; }
        }
        mma_commit(tfull_bar(acc));
        if (++acc == kDgAcc) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else {
    // ===== epilogue: row m' = Y*10 + X holds the 2x2 pixel block (2Y+dy, 2X+dx), 16 channels each =====
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const int Y = r / 10, X = r - Y * 10;
    int acc = 0; uint32_t acc_phase = 0;
    float b8[8];
    if constexpr (CO == 8) {
#pragma unroll
      for (int c = 0; c < 8; ++c) b8[c] = bias ? __ldg(bias + c) : 0.f;
    }
    float dbacc[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) dbacc[c] = 0.f;
    const float* b16 = s_bias;
    float loss_part = 0.f;
    constexpr int kDyPre = ((CO == 8 || PC) && EPI == 8) ? 1 : 2;
    float2 tg_next[kDyPre];
    float m_next = 0.f;
    int a_next = 0;
#pragma unroll
    for (int d = 0; d < kDyPre; ++d) tg_next[d] = make_float2(0.f, 0.f);
    if ((CO == 8 || PC) && pl.target != nullptr && r < 100 && (int)blockIdx.x < samples) {
      const int dyb = EPI == 8 ? ((warp - 2) >> 2) : 0;
      m_next = __ldg(pl.mask + blockIdx.x);
      a_next = __ldg(pl.act + blockIdx.x);
#pragma unroll
      for (int d = 0; d < kDyPre; ++d)
        tg_next[d] = __ldcs(reinterpret_cast<const float2*>(pl.target + ((int64_t)blockIdx.x * 20 + 2 * Y + dyb + d) * 20 + 2 * X));
    }
    for (int it = blockIdx.x; it < samples; it += gridDim.x) {
      mbar_wait(tfull_bar(acc), acc_phase);
      fence_after_sync();
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * 64);
      if constexpr (CO == 8) {
        // column (dy, dx, c) = dy*16 + dx*8 + c; each dy is 16 contiguous floats (pixels 2X, 2X+1).  EPI = 4: one load of
        // both parities; EPI = 8: this warp's parity only
        constexpr int kDy = EPI == 8 ? 1 : 2;
        const int dy_base = EPI == 8 ? ((warp - 2) >> 2) : 0;
        uint32_t v[16 * kDy];
        if constexpr (EPI == 8) tmem_ld16(taddr + (uint32_t)(16 * dy_base), v);
        else tmem_ld32(taddr, v);
        tmem_ld_wait();
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(acc));
        if (pl.qmax != nullptr) {
          // bootstrap path: the dueling combine and max over actions in the epilogue, 1.6 KB out per sample instead of 12.8
          if (r < 100) {
            const float inv_a = 1.0f / (float)pl.a;
#pragma unroll
            for (int d = 0; d < kDy; ++d) {
              const int dy = dy_base + d;
              float q2[2];
#pragma unroll
              for (int dx = 0; dx < 2; ++dx) {
                float y[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) y[c] = fmaxf(__uint_as_float(v[d * 16 + dx * 8 + c]) + b8[c], 0.f);
                float sum = 0.f, best = -3.4e38f;
#pragma unroll
                for (int k = 0; k < 7; ++k) {
                  if (k < pl.a) { sum += y[1 + k]; best = fmaxf(best, y[1 + k]); }
                }
                q2[dx] = y[0] + best - sum * inv_a;          // max_a (V + A_a - mean A) = V + max_a A_a - mean A
              }
              *reinterpret_cast<float2*>(pl.qmax + ((int64_t)it * 20 + 2 * Y + dy) * 20 + 2 * X) = make_float2(q2[0], q2[1]);
            }
          }
          if (++acc == kDgAcc) { acc = 0; acc_phase ^= 1u; }
          continue;
        }
        if (pl.target != nullptr) {
          // this sample's targets / mask / action were requested one sample ago (their HBM latency would otherwise be
          // exposed once per sample and warp); request the next sample's now
          float2 tgs[kDy];
#pragma unroll
          for (int d = 0; d < kDy; ++d) tgs[d] = tg_next[d];
          const float m = m_next;
          const int a = a_next;
          if (r < 100 && it + (int)gridDim.x < samples) {
            const int nx = it + (int)gridDim.x;
            m_next = __ldg(pl.mask + nx);
            a_next = __ldg(pl.act + nx);
#pragma unroll
            for (int d = 0; d < kDy; ++d)
              tg_next[d] = __ldcs(reinterpret_cast<const float2*>(pl.target + ((int64_t)nx * 20 + 2 * Y + dy_base + d) * 20 + 2 * X));
          }
          if (r < 100) {
            // NA > 0: the action count as a compile-time constant (the epilogue was ALU-bound on the per-channel predicates:
            // ncu 71 % of the ALU pipe, issue slots 66 % busy, profiles/r2_pc_planes_ncu_summary.txt)
            constexpr int kA = NA > 0 ? NA : 7;
            const float inv_a = 1.0f / (float)pl.a;
            float ck[kA];                                    // (k == a) - 1/A: d Q_a / d Adv_k
#pragma unroll
            for (int k = 0; k < kA; ++k) ck[k] = (k == a ? 1.f : 0.f) - inv_a;
            __nv_bfloat16* out16 = reinterpret_cast<__nv_bfloat16*>(out_raw);
#pragma unroll
            for (int d = 0; d < kDy; ++d) {
              const int dy = dy_base + d;
              const int64_t pix = ((int64_t)it * 20 + 2 * Y + dy) * 20 + 2 * X;
              const float2 tg = tgs[d];
              uint4* dst = reinterpret_cast<uint4*>(out16 + pix * (pl.c8 ? 8 : 16));
#pragma unroll
              for (int dx = 0; dx < 2; ++dx) {
                float y[1 + kA];
#pragma unroll
                for (int c = 0; c <= kA; ++c) y[c] = fmaxf(__uint_as_float(v[d * 16 + dx * 8 + c]) + b8[c], 0.f);
                float sum = 0.f, qa = 0.f;
#pragma unroll
                for (int k = 0; k < kA; ++k) {
                  if (NA > 0 || k < pl.a) { sum += y[1 + k]; if (k == a) qa = y[1 + k]; }
                }
                qa = y[0] + qa - sum * inv_a;
                const float diff = qa - (dx ? tg.y : tg.x);
                loss_part += m * diff * diff;
                const float g = pl.lam * m * diff;
                float dd[8];
                dd[0] = y[0] > 0.f ? g : 0.f;
#pragma unroll
                for (int k = 0; k < 7; ++k)
                  dd[1 + k] = (k < kA && (NA > 0 || k < pl.a) && y[k < kA ? 1 + k : 0] > 0.f) ? g * ck[k < kA ? k : 0] : 0.f;
                uint32_t pk[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  if (2 * j > kA) { pk[j] = 0u; continue; }       // channels beyond 1 + A: zero
                  __nv_bfloat162 p = __floats2bfloat162_rn(dd[2 * j], dd[2 * j + 1]);
                  pk[j] = *reinterpret_cast<uint32_t*>(&p);
                  const float2 f = __bfloat1622float2(p);      // the bias gradient sums the ROUNDED values
                  dbacc[2 * j] += f.x;
                  if (2 * j + 1 <= kA) dbacc[2 * j + 1] += f.y;
                }
                if (pl.c8 == 2) {        // consecutive lanes = consecutive 16-byte rows of one plane
                  __stcs(reinterpret_cast<uint4*>(out16) + ((int64_t)it * 4 + dy * 2 + dx) * 100 + r, make_uint4(pk[0], pk[1], pk[2], pk[3]));
                } else if (pl.c8) {
                  __stcs(dst + dx, make_uint4(pk[0], pk[1], pk[2], pk[3]));
                } else {
                  __stcs(dst + 2 * dx, make_uint4(pk[0], pk[1], pk[2], pk[3]));
                  __stcs(dst + 2 * dx + 1, make_uint4(0u, 0u, 0u, 0u));
                }
              }
            }
          }
          if (++acc == kDgAcc) { acc = 0; acc_phase ^= 1u; }
          continue;
        }
        if (r < 100) {
          float* base = reinterpret_cast<float*>(out_raw) + (((int64_t)it * 20 + 2 * Y) * 20 + 2 * X) * 8;
#pragma unroll
          for (int d = 0; d < kDy; ++d) {
            const int dy = dy_base + d;
            float4* dst = reinterpret_cast<float4*>(base + dy * 160);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              float4 o;
              o.x = fmaxf(__uint_as_float(v[d * 16 + 4 * q + 0]) + b8[(4 * q + 0) & 7], 0.f);
              o.y = fmaxf(__uint_as_float(v[d * 16 + 4 * q + 1]) + b8[(4 * q + 1) & 7], 0.f);
              o.z = fmaxf(__uint_as_float(v[d * 16 + 4 * q + 2]) + b8[(4 * q + 2) & 7], 0.f);
              o.w = fmaxf(__uint_as_float(v[d * 16 + 4 * q + 3]) + b8[(4 * q + 3) & 7], 0.f);
              dst[q] = o;
            }
          }
        }
        if (++acc == kDgAcc) { acc = 0; acc_phase ^= 1u; }
        continue;
      }
      if constexpr (PC) {
        // column (dy, dx, c) = dy*32 + dx*16 + c.  EPI = 4: both parities; EPI = 8: this warp's parity only
        constexpr int kDy = EPI == 8 ? 1 : 2;
        const int dy_base = EPI == 8 ? ((warp - 2) >> 2) : 0;
        uint32_t v[kDy][32];
#pragma unroll
        for (int d = 0; d < kDy; ++d) tmem_ld32(taddr + (uint32_t)(32 * (dy_base + d)), v[d]);
        tmem_ld_wait();
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(acc));
        const float inv_a = 1.0f / (float)pl.a;
        if (pl.qmax != nullptr) {
          if (r < 100) {
#pragma unroll
            for (int d = 0; d < kDy; ++d) {
              float q2[2];
#pragma unroll
              for (int dx = 0; dx < 2; ++dx) {
                const uint32_t* vv = v[d] + dx * 16;
                float sum = 0.f, best = -3.4e38f;
#pragma unroll
                for (int k = 0; k < 15; ++k) {
                  if (k < pl.a) {
                    const float y = fmaxf(__uint_as_float(vv[1 + k]) + b16[1 + k], 0.f);
                    sum += y; best = fmaxf(best, y);
                  }
                }
                q2[dx] = fmaxf(__uint_as_float(vv[0]) + b16[0], 0.f) + best - sum * inv_a;
              }
              *reinterpret_cast<float2*>(pl.qmax + ((int64_t)it * 20 + 2 * Y + dy_base + d) * 20 + 2 * X) = make_float2(q2[0], q2[1]);
            }
          }
          if (++acc == kDgAcc) { acc = 0; acc_phase ^= 1u; }
          continue;
        }
        float2 tgs[kDy];
#pragma unroll
        for (int d = 0; d < kDy; ++d) tgs[d] = tg_next[d];
        const float m = m_next;
        const int a = a_next;
        if (r < 100 && it + (int)gridDim.x < samples) {
          const int nx = it + (int)gridDim.x;
          m_next = __ldg(pl.mask + nx);
          a_next = __ldg(pl.act + nx);
#pragma unroll
          for (int d = 0; d < kDy; ++d)
            tg_next[d] = __ldcs(reinterpret_cast<const float2*>(pl.target + ((int64_t)nx * 20 + 2 * Y + dy_base + d) * 20 + 2 * X));
        }
        if (r < 100) {
          uint4* out16 = reinterpret_cast<uint4*>(out_raw);
#pragma unroll
          for (int d = 0; d < kDy; ++d) {
            const int64_t pix = ((int64_t)it * 20 + 2 * Y + dy_base + d) * 20 + 2 * X;
#pragma unroll
            for (int dx = 0; dx < 2; ++dx) {
              const uint32_t* vv = v[d] + dx * 16;
              float y[16];
#pragma unroll
              for (int c = 0; c < 16; ++c) y[c] = fmaxf(__uint_as_float(vv[c]) + b16[c], 0.f);
              float sum = 0.f, qa = 0.f;
#pragma unroll
              for (int k = 0; k < 15; ++k) {
                if (k < pl.a) { sum += y[1 + k]; if (k == a) qa = y[1 + k]; }
              }
              qa = y[0] + qa - sum * inv_a;
              const float diff = qa - (dx ? tgs[d].y : tgs[d].x);
              loss_part += m * diff * diff;
              const float g = pl.lam * m * diff;
              uint32_t pk[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                float dd[2];
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                  const int c = 2 * j + e, k = c - 1;
                  dd[e] = c == 0 ? (y[0] > 0.f ? g : 0.f)
                                 : ((k < pl.a && y[c] > 0.f) ? g * ((k == a ? 1.f : 0.f) - inv_a) : 0.f);
                }
                __nv_bfloat162 p = __floats2bfloat162_rn(dd[0], dd[1]);
                pk[j] = *reinterpret_cast<uint32_t*>(&p);
                const float2 f = __bfloat1622float2(p);      // the bias gradient sums the ROUNDED values
                dbacc[2 * j] += f.x; dbacc[2 * j + 1] += f.y;
              }
              __stcs(out16 + pix * 2 + 2 * dx, make_uint4(pk[0], pk[1], pk[2], pk[3]));
              __stcs(out16 + pix * 2 + 2 * dx + 1, make_uint4(pk[4], pk[5], pk[6], pk[7]));
            }
          }
        }
        if (++acc == kDgAcc) { acc = 0; acc_phase ^= 1u; }
        continue;
      }
      __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(out_raw);
      uint32_t v0[32], v1[32];
      tmem_ld32(taddr, v0);            // dy = 0: (dx, c) = 32 values = pixels (2Y, 2X) and (2Y, 2X+1)
      tmem_ld32(taddr + 32, v1);       // dy = 1
      tmem_ld_wait();
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
      if (mask_y != nullptr) {
        // fused ReLU gradient of the layer below (conv1): mask by h1 > 0, round to bf16, write the two
        // 8-channel PLANES conv1's tensor-core wgrad consumes ([2][S*400][8]) and accumulate the bias
        // gradient -- the dense gradient is never written and no separate relu_grad pass reads it back
        if (r < 100) {
          const int64_t pix = ((int64_t)it * 20 + 2 * Y) * 20 + 2 * X;
          // output pixel index: dense [S*400], or on conv1-wgrad's 21-pixel row pitch [S*420] (column 20 zero)
          const int rowp = pitch21 ? 21 : 20;
          const int64_t opix = ((int64_t)it * 20 + 2 * Y) * rowp + 2 * X;
          const int64_t plane = (int64_t)samples * 20 * rowp;
#pragma unroll
          for (int dy = 0; dy < 2; ++dy) {
            const uint32_t* v = dy ? v1 : v0;
            const uint4* ysrc = reinterpret_cast<const uint4*>(mask_y + (pix + dy * 20) * 16);
#pragma unroll
            for (int q = 0; q < 4; ++q) {          // q = dx*2 + plane half: 8 channels of pixel (2Y+dy, 2X+dx)
              const uint4 yu = __ldg(ysrc + q);
              const __nv_bfloat162* yh = reinterpret_cast<const __nv_bfloat162*>(&yu);
              uint32_t pk[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float2 yf = __bfloat1622float2(yh[j]);
                const float a = yf.x > 0.f ? __uint_as_float(v[8 * q + 2 * j]) : 0.f;
                const float b = yf.y > 0.f ? __uint_as_float(v[8 * q + 2 * j + 1]) : 0.f;
                __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
                pk[j] = *reinterpret_cast<uint32_t*>(&p);
                const float2 f = __bfloat1622float2(p);      // the bias gradient sums the ROUNDED values
                dbacc[(q & 1) * 8 + 2 * j] += f.x; dbacc[(q & 1) * 8 + 2 * j + 1] += f.y;
              }
              __nv_bfloat16* dst = out + ((q & 1) * plane + opix + dy * rowp + (q >> 1)) * 8;
              *reinterpret_cast<uint4*>(dst) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            }
            if (pitch21 && X == 9) {           // the zero column ox = 20 of both planes
              *reinterpret_cast<uint4*>(out + (opix + dy * 21 + 2) * 8) = make_uint4(0u, 0u, 0u, 0u);
              *reinterpret_cast<uint4*>(out + (plane + opix + dy * 21 + 2) * 8) = make_uint4(0u, 0u, 0u, 0u);
            }
          }
        }
        if (++acc == kDgAcc) { acc = 0; acc_phase ^= 1u; }
        continue;
      }
      if (r < 100) {
        __nv_bfloat16* base = out + (((int64_t)it * 20 + 2 * Y) * 20 + 2 * X) * 16;
#pragma unroll
        for (int dy = 0; dy < 2; ++dy) {
          const uint32_t* v = dy ? v1 : v0;
          uint4* dst = reinterpret_cast<uint4*>(base + dy * 320);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            uint32_t pk[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              __nv_bfloat162 p = __floats2bfloat162_rn(__uint_as_float(v[8 * q + 2 * j]), __uint_as_float(v[8 * q + 2 * j + 1]));
              pk[j] = *reinterpret_cast<uint32_t*>(&p);
            }
            dst[q] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          }
        }
      }
      if (++acc == kDgAcc) { acc = 0; acc_phase ^= 1u; }
    }
    if (CO == 16 && mask_y != nullptr && db != nullptr) {
#pragma unroll
      for (int c = 0; c < 16; ++c) {
        float x = dbacc[c];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (lane == 0) atomicAdd(db + c, x);
      }
    }
    if ((CO == 8 || PC) && pl.target != nullptr) {
      if (db != nullptr) {
#pragma unroll
        for (int c = 0; c < (PC ? 16 : 8); ++c) {
          float x = dbacc[c];
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
          if (lane == 0) atomicAdd(db + c, x);
        }
      }
      if (pl.loss != nullptr) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) loss_part += __shfl_xor_sync(0xffffffffu, loss_part, o);
        if (lane == 0) atomicAdd(pl.loss, 0.5 * (double)pl.lam * (double)loss_part);
      }
    }
  }
  __syncwarp();
  fence_before_sync();
  __syncthreads();
  if (warp == 2) {
    fence_after_sync();
    tmem_dealloc<kDgAcc * 64>(tmem_base);
  }
}


// ---- pixel-control head: the backward pass on the PLANE-MAJOR loss gradient ----------------------------------------
// The two kernels above spend their time in the TMA engine, not in HBM or the tensor core: a sample is four boxes of 81
// rows (each filter row ky re-fetches the image rows it overlaps with, 3.2x the tensor's bytes), ~420 row requests, and
// halving the row width (16 -> 8 channels) changed nothing (scripts/pc_head_bench.py: wgrad 796 us at 163 840 samples
// either way).  conv1's remedy applies: the fused deconv + loss kernel owns the layout of its gradient, so it writes the
// space-to-depth view directly -- four parity planes (dy,dx) of the 10 x 10 grid, [S][4][100][8 channels] bf16, 6400
// contiguous bytes per sample = the un-swizzled UMMA layout with a 16-byte row pitch.  ONE bulk copy lands a sample;
// tap (by,bx) of the 2x2 stride-1 convolution over that view is the same tile with the descriptor start address advanced
// by (by*10 + bx) rows.  GEMM rows follow the 10-wide grid (m' = oy*10 + ox; ox = 9, oy = 9 and rows >= 100 are
// accumulator rows nobody stores).
constexpr int kPpPlaneBytes = 100 * 16;
constexpr int kPpTileBytes = 4 * kPpPlaneBytes;          // 6400
constexpr int kPpStages = 8;
constexpr int kPpAcc = 4;                                // TMEM accumulators of 32 columns
constexpr int kPpWBytes = 4 * 2 * 2 * 32 * 16;           // [tap][dy][dx][32 out rows][8 ch] bf16
constexpr int kPpSmem = kPpWBytes + kPpStages * kPpTileBytes + 1024 /*tail reads*/ + 1024 /*barriers*/ + 1024 /*align*/;

// d(pc_fc1 output) [S,9,9,32] = conv 4x4 stride 2 of the gradient with the merged deconv filter, times *scale, zeroed where
// the pc_fc1 output mask_y <= 0, rounded to bf16; db [81*32] += the rounded values summed over samples.
__global__ void __launch_bounds__(kConvThreads, 2)
pc_planes_conv_tcgen05_kernel(const __nv_bfloat16* __restrict__ dyp, const __nv_bfloat16* __restrict__ w_planes,
                              const float* __restrict__ scale, const __nv_bfloat16* __restrict__ mask_y,
                              __nv_bfloat16* __restrict__ out, float* __restrict__ db, int samples) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t w_smem = smem_base;
  const uint32_t a_smem = smem_base + kPpWBytes;
  const uint32_t bar_base = a_smem + kPpStages * kPpTileBytes + 1024;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kPpStages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * kPpStages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * kPpStages + kPpAcc + a); };
  const uint32_t w_bar = bar_base + 8u * (2 * kPpStages + 2 * kPpAcc);
  const uint32_t tmem_slot = w_bar + 8u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < kPpStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < kPpAcc; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4); }
    mbar_init(w_bar, 1);
    fence_mbar_init();
  } else if (warp == 2) {
    tmem_alloc<kPpAcc * 32>(tmem_slot);
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = tmem_base_at(tmem_slot);

  if (warp == 0) {
    if (lane == 0) {
      // ===== producer: resident filters (one bulk copy), then ONE 6400-byte bulk copy per sample =====
      mbar_arrive_expect_tx(w_bar, kPpWBytes);
      bulk_load(w_smem, w_planes, kPpWBytes, w_bar);
      int stage = 0; uint32_t phase = 0;
      for (int it = blockIdx.x; it < samples; it += gridDim.x) {
        mbar_wait(empty_bar(stage), phase ^ 1u);
        mbar_arrive_expect_tx(full_bar(stage), kPpTileBytes);
        bulk_load(a_smem + stage * kPpTileBytes, reinterpret_cast<const uint8_t*>(dyp) + (int64_t)it * kPpTileBytes, kPpTileBytes,
                  full_bar(stage));
        if (++stage == kPpStages) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===== MMA issuer: 4 taps x 2 UMMA (128 x 32 x 16: the two dx planes of one dy) on the one resident tile =====
      constexpr uint32_t idesc = idesc_bf16_f32(128, 32, false, false);
      constexpr uint32_t desc_hi = (128u >> 4) | (1u << 14);        // SBO = 128 B (8 rows), descriptor version 1, no swizzle
      const uint32_t w_lo0 = (w_smem >> 4) | ((512u >> 4) << 16);   // filter tiles: LBO = 512 B (32 rows of one 8-channel chunk)
      mbar_wait(w_bar, 0);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int it = blockIdx.x; it < samples; it += gridDim.x) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        mbar_wait(full_bar(stage), phase);
        fence_after_sync();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * 32);
        const uint32_t a_lo0 = ((a_smem + stage * kPpTileBytes) >> 4) | ((uint32_t)(kPpPlaneBytes >> 4) << 16);   // LBO = plane stride
#pragma unroll
        for (int tap = 0; tap < 4; ++tap) {
          const uint32_t shift16 = (uint32_t)((tap >> 1) * 10 + (tap & 1));
#pragma unroll
          for (int j = 0; j < 2; ++j)
            mma_f16_lohi(tmem_d, a_lo0 + (uint32_t)(2 * j * kPpPlaneBytes >> 4) + shift16, desc_hi,
                         w_lo0 + (uint32_t)(((tap * 2 + j) * 1024) >> 4), desc_hi, idesc, (tap > 0 || j > 0) ? 1u : 0u);
        }
        mma_commit(empty_bar(stage));
        mma_commit(tfull_bar(acc));
        if (++stage == kPpStages) { stage = 0; phase ^= 1u; }
        if (++acc == kPpAcc) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else {
    // ===== epilogue: row m' = oy*10 + ox -> scale, pc_fc1's ReLU mask, bf16, bias-gradient partial sums =====
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const int oy = r / 10, ox = r - oy * 10;
    const bool valid = oy < 9 && ox < 9;
    const int orow = valid ? oy * 9 + ox : 0;
    int acc = 0; uint32_t acc_phase = 0;
    float dbacc[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) dbacc[j] = 0.f;
    const float sc = scale ? __ldg(scale) : 1.f;
    // the mask row of a sample is requested one sample ahead: with the accumulators ready long before the epilogue gets to
    // them, a load issued in the same iteration would expose its whole HBM latency once per sample
    uint4 yn[4];
    if (blockIdx.x < samples) {
      const uint4* ysrc = reinterpret_cast<const uint4*>(mask_y + ((int64_t)blockIdx.x * 81 + orow) * 32);
#pragma unroll
      for (int q = 0; q < 4; ++q) yn[q] = __ldg(ysrc + q);
    }
    for (int it = blockIdx.x; it < samples; it += gridDim.x) {
      const int64_t row0 = ((int64_t)it * 81 + orow) * 32;
      uint4 yv[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) yv[q] = yn[q];
      if (it + (int)gridDim.x < samples) {
        const uint4* ysrc = reinterpret_cast<const uint4*>(mask_y + ((int64_t)(it + gridDim.x) * 81 + orow) * 32);
#pragma unroll
        for (int q = 0; q < 4; ++q) yn[q] = __ldg(ysrc + q);
      }
      mbar_wait(tfull_bar(acc), acc_phase);
      fence_after_sync();
      uint32_t v[32];
      tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * 32), v);
      tmem_ld_wait();
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
      if (valid) {
        uint4* dst = reinterpret_cast<uint4*>(out + row0);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint32_t pk[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint32_t yw = j == 0 ? yv[q].x : (j == 1 ? yv[q].y : (j == 2 ? yv[q].z : yv[q].w));
            const float2 yf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&yw));
            const float v0 = yf.x > 0.f ? __uint_as_float(v[8 * q + 2 * j]) * sc : 0.f;
            const float v1 = yf.y > 0.f ? __uint_as_float(v[8 * q + 2 * j + 1]) * sc : 0.f;
            __nv_bfloat162 p2 = __floats2bfloat162_rn(v0, v1);
            pk[j] = *reinterpret_cast<uint32_t*>(&p2);
            const float2 f = __bfloat1622float2(p2);      // the bias gradient sums the ROUNDED values (as unreal_relu_grad does)
            dbacc[8 * q + 2 * j] += f.x; dbacc[8 * q + 2 * j + 1] += f.y;
          }
          __stcs(dst + q, make_uint4(pk[0], pk[1], pk[2], pk[3]));
        }
      }
      if (++acc == kPpAcc) { acc = 0; acc_phase ^= 1u; }
    }
    if (valid && db != nullptr) {
#pragma unroll
      for (int j = 0; j < 32; ++j) atomicAdd(db + orow * 32 + j, dbacc[j]);
    }
  }
  __syncwarp();
  fence_before_sync();
  __syncthreads();
  if (warp == 2) {
    fence_after_sync();
    tmem_dealloc<kPpAcc * 32>(tmem_base);
  }
}

// The merged deconv filter's gradient dW8[ky][kx][c][o] = sum over samples and (oy,ox) of dy[2oy+ky, 2ox+kx, c] . hp[oy,ox,o]:
// the reduction runs over pixels, so both operands are MN-major -- the gradient planes as they lie (A: M = (dy,dx,c) = 4 real
// 8-channel chunks of the 8 a 64-row UMMA reads, K = grid rows at a 16-byte pitch, tap = start address shift), the sample's
// pc_fc1 output hp [9,9,32] through a 4-D box {32, 10, 9, 1} (column ox = 9 is out of bounds = TMA zero fill) as a
// 64-byte-swizzled B tile on the same 10-wide grid.  K = 96 rows: rows 90..95 of the B tile are zero (zeroed once, never
// written), so the finite gradient values A holds there contribute nothing.  Four [32 x 32] accumulators (one per
// tap) live in TMEM across all samples of a CTA and are added to global once, in HWIO order.
constexpr int kPwAStages = 10;
constexpr int kPwBStages = 6;
constexpr int kPwBBytes = 6144;                    // 90 landed rows x 64 B (+ 6 zero rows), 1024-aligned
constexpr int kPwTail = 8192;                      // the four garbage chunks of the last A stage read here
constexpr int kPwSmem = kPwBStages * kPwBBytes + kPwAStages * kPpTileBytes + kPwTail + 1024 + 1024;

__global__ void __launch_bounds__(128, 2)
pc_planes_wgrad_tcgen05_kernel(const __nv_bfloat16* __restrict__ dyp, const __grid_constant__ CUtensorMap tma_hp,
                               float* __restrict__ dw, int samples) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t b_smem = smem_base;
  const uint32_t a_smem = b_smem + kPwBStages * kPwBBytes;
  const uint32_t bar_base = a_smem + kPwAStages * kPpTileBytes + kPwTail;
  auto fullA = [&](int s) { return bar_base + 8u * s; };
  auto emptyA = [&](int s) { return bar_base + 8u * (kPwAStages + s); };
  auto fullB = [&](int s) { return bar_base + 8u * (2 * kPwAStages + s); };
  auto emptyB = [&](int s) { return bar_base + 8u * (2 * kPwAStages + kPwBStages + s); };
  const uint32_t done_bar = bar_base + 8u * (2 * kPwAStages + 2 * kPwBStages);
  const uint32_t tmem_slot = done_bar + 8u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // zero every tile byte once: the never-written rows of the B tiles, and whatever A reads before its first copies land
  for (uint32_t off = threadIdx.x * 16u; off < (uint32_t)(kPwBStages * kPwBBytes + kPwAStages * kPpTileBytes + kPwTail); off += 128u * 16u)
    st_shared_v4(smem_base + off, 0u, 0u, 0u, 0u);
  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tma_hp);
    for (int s = 0; s < kPwAStages; ++s) { mbar_init(fullA(s), 1); mbar_init(emptyA(s), 1); }
    for (int s = 0; s < kPwBStages; ++s) { mbar_init(fullB(s), 1); mbar_init(emptyB(s), 1); }
    mbar_init(done_bar, 1);
    fence_mbar_init();
  } else if (warp == 2) {
    tmem_alloc<128>(tmem_slot);
  }
  fence_proxy_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = tmem_base_at(tmem_slot);

  if (warp == 0) {
    if (lane == 0) {
      int sa = 0; uint32_t pa = 0; int sb = 0; uint32_t pb = 0;
      for (int it = blockIdx.x; it < samples; it += gridDim.x) {
        mbar_wait(emptyB(sb), pb ^ 1u);
        mbar_arrive_expect_tx(fullB(sb), 90 * 64);
        tma_load_4d(b_smem + sb * kPwBBytes, &tma_hp, fullB(sb), 0, 0, 0, it);
        if (++sb == kPwBStages) { sb = 0; pb ^= 1u; }
        mbar_wait(emptyA(sa), pa ^ 1u);
        mbar_arrive_expect_tx(fullA(sa), kPpTileBytes);
        bulk_load(a_smem + sa * kPpTileBytes, reinterpret_cast<const uint8_t*>(dyp) + (int64_t)it * kPpTileBytes, kPpTileBytes, fullA(sa));
        if (++sa == kPwAStages) { sa = 0; pa ^= 1u; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = idesc_bf16_f32(64, 32, true, true);
      // A: MN-major un-swizzled -- LBO = 128 B (next 8 grid rows), SBO = plane stride (next 8-channel chunk)
      // B: MN-major, 64-byte rows, 64-byte swizzle -- SBO = 512 B (next 8 grid rows)
      constexpr uint32_t a_hi = ((uint32_t)kPpPlaneBytes >> 4) | (1u << 14);
      constexpr uint32_t b_hi = (512u >> 4) | (1u << 14) | (4u << 29);
      int sa = 0; uint32_t pa = 0; int sb = 0; uint32_t pb = 0;
      bool first = true;
      for (int it = blockIdx.x; it < samples; it += gridDim.x) {
        mbar_wait(fullB(sb), pb);
        mbar_wait(fullA(sa), pa);
        fence_after_sync();
        const uint32_t a_lo0 = ((a_smem + sa * kPpTileBytes) >> 4) | ((128u >> 4) << 16);
        const uint32_t b_lo0 = ((b_smem + sb * kPwBBytes) >> 4) | ((64u >> 4) << 16);
#pragma unroll
        for (int tap = 0; tap < 4; ++tap) {
          const uint32_t shift16 = (uint32_t)((tap >> 1) * 10 + (tap & 1));
#pragma unroll
          for (int ks = 0; ks < 6; ++ks)
            mma_f16_lohi(tmem_base + (uint32_t)(tap * 32), a_lo0 + shift16 + (uint32_t)(ks * 16), a_hi, b_lo0 + (uint32_t)(ks * 64), b_hi,
                         idesc, (first && ks == 0) ? 0u : 1u);
        }
        first = false;
        mma_commit(emptyA(sa));
        mma_commit(emptyB(sb));
        if (++sa == kPwAStages) { sa = 0; pa ^= 1u; }
        if (++sb == kPwBStages) { sb = 0; pb ^= 1u; }
      }
      mma_commit(done_bar);
    }
    __syncwarp();
  }
  {
    // ===== final epilogue: a 64-row accumulator keeps row m = (dy,dx,c) in lane 32*(m/16) + m%16 (warps 0, 1: the 32 real
    // rows), accumulator `tap` in columns tap*32 + o -> dW8 in HWIO order [ky = 2by+dy][kx = 2bx+dx][c][o] =====
    mbar_wait(done_bar, 0);
    fence_after_sync();
    const int m = warp * 16 + lane;
    const int pdy = (m >> 4) & 1, pdx = (m >> 3) & 1, c = m & 7;
#pragma unroll 1
    for (int tap = 0; tap < 4; ++tap) {
      uint32_t v[32];
      tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(tap * 32), v);
      tmem_ld_wait();
      const int ky = 2 * (tap >> 1) + pdy, kx = 2 * (tap & 1) + pdx;
      float* o = dw + ((ky * 4 + kx) * 8 + c) * 32;
      if (lane < 16 && m < 32) {
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          red_add_v4(o + j, __uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
      }
    }
  }
  __syncwarp();
  fence_before_sync();
  __syncthreads();
  if (warp == 2) {
    fence_after_sync();
    tmem_dealloc<128>(tmem_base);
  }
}

template <int N, int MODE, bool MASKED = false, int C = 16, bool SPLIT = false>
static int launch_conv(const CUtensorMap& ta, const CUtensorMap& ta2, const CUtensorMap& tw, const CUtensorMap& tc,
                       const ConvArgs& g, cudaStream_t st, const CUtensorMap& talo, const CUtensorMap& talo2,
                       const CUtensorMap& twlo) {
  using Cfg = ConvCfg<MODE, C>;
  constexpr int kWBytes = (SPLIT ? 2 : 1) * ((Cfg::kSteps * N * Cfg::kRowBytes + 1023) / 1024 * 1024);
  // + 5 KB: the last stage's 128-row UMMA read runs 40 rows past its 88-row stage into barriers / epilogue buffers
  constexpr int kSmem = kWBytes + (SPLIT ? 2 * 2 * Cfg::kStageBytes : Cfg::kStages * Cfg::kStageBytes) + 1024 +
                        Cfg::kEpiWarps * 2 * 4096 + 1024;
  auto kern = conv_fwd_tcgen05_kernel<N, MODE, MASKED, C, SPLIT>;
  const int rc = allow_dynamic_smem((const void*)kern, kSmem);
  if (rc != UNREAL_OK) return rc;
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  const int grid = g.items < 2 * sms ? g.items : 2 * sms;
  kern<<<grid, kConvThreads, kSmem, st>>>(ta, ta2, tw, tc, g, talo, talo2, twlo);
  UNREAL_LAUNCH_CHECK("conv_fwd_tcgen05_kernel");
  return UNREAL_OK;
}

}  // namespace unreal

using namespace unreal;

static int s2d_frames_impl(const void* frames, int dtype, void* out_bf16, void* out_lo_bf16, int s, void* stream) {
  UNREAL_REQUIRE(frames && out_bf16 && s > 0, "unreal_s2d_frames: null buffer or s <= 0");
  UNREAL_REQUIRE(dtype == UNREAL_F32 || dtype == UNREAL_U8, "unreal_s2d_frames: frames must be f32 or u8");
  UNREAL_REQUIRE(aligned16(frames) && aligned16(out_bf16), "unreal_s2d_frames: buffers must be 16-byte aligned");
  const int64_t total = (int64_t)s * 441;
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  int64_t want = (total + 255) / 256;
  const int grid = (int)(want < (int64_t)sms * 16 ? want : (int64_t)sms * 16);
  auto* hi = reinterpret_cast<__nv_bfloat16*>(out_bf16);
  auto* lo = reinterpret_cast<__nv_bfloat16*>(out_lo_bf16);
  if (dtype == UNREAL_F32 && lo)
    s2d_frames_kernel<float, true><<<grid, 256, 0, as_stream(stream)>>>(reinterpret_cast<const float*>(frames), hi, total, 0x4B000000u, lo);
  else if (dtype == UNREAL_F32)
    s2d_frames_kernel<float><<<grid, 256, 0, as_stream(stream)>>>(reinterpret_cast<const float*>(frames), hi, total, 0x4B000000u, nullptr);
  else if (lo)
    s2d_frames_kernel<uint8_t, true><<<grid, 256, 0, as_stream(stream)>>>(reinterpret_cast<const uint8_t*>(frames), hi, total, 0x4B000000u, lo);
  else
    s2d_frames_kernel<uint8_t><<<grid, 256, 0, as_stream(stream)>>>(reinterpret_cast<const uint8_t*>(frames), hi, total, 0x4B000000u, nullptr);
  UNREAL_LAUNCH_CHECK("s2d_frames_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_s2d_frames(const void* frames, int dtype, void* out_bf16, int s, void* stream) {
  return s2d_frames_impl(frames, dtype, out_bf16, nullptr, s, stream);
}

extern "C" int unreal_s2d_frames_split(const void* frames, int dtype, void* out_hi_bf16, void* out_lo_bf16, int s, void* stream) {
  UNREAL_REQUIRE(out_lo_bf16 && aligned16(out_lo_bf16), "unreal_s2d_frames_split: null or unaligned lo planes");
  return s2d_frames_impl(frames, dtype, out_hi_bf16, out_lo_bf16, s, stream);
}

// conv1 forward over x'' planes (pos == NULL) or render-fused over maze cells; SPLIT: w_lo / out_lo non-null, xpp_lo nullable
template <bool SPLIT>
static int conv1_fwd_launch(const void* xpp, const int32_t* pos, const void* w_taps, const float* bias, void* out, int s,
                            void* stream, const void* xpp_lo = nullptr, const void* w_lo = nullptr, void* out_lo = nullptr) {
  const uint64_t walls = pos != nullptr ? maze_walls49() : 0;
  constexpr int kSmem = SPLIT ? kC1SplitSmem : kC1Smem;
  const int rc = allow_dynamic_smem((const void*)conv1_fwd_tcgen05_kernel<SPLIT>, kSmem);
  if (rc != UNREAL_OK) return rc;
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  const int items = s * 4;
  const int ctas = 2 * sms;
  using bf = __nv_bfloat16;
  conv1_fwd_tcgen05_kernel<SPLIT><<<items < ctas ? items : ctas, kConvThreads, kSmem, as_stream(stream)>>>(
      reinterpret_cast<const bf*>(xpp), reinterpret_cast<const bf*>(w_taps), bias, reinterpret_cast<bf*>(out), items, pos, walls,
      reinterpret_cast<const bf*>(xpp_lo), reinterpret_cast<const bf*>(w_lo), reinterpret_cast<bf*>(out_lo));
  UNREAL_LAUNCH_CHECK(pos ? "conv1_fwd_tcgen05_kernel(maze)" : "conv1_fwd_tcgen05_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_conv1_fwd_maze(const int32_t* pos, const void* w_taps_bf16, const float* bias, void* out_bf16, int s,
                                     void* stream) {
  UNREAL_REQUIRE(pos && w_taps_bf16 && out_bf16 && s > 0, "unreal_conv1_fwd_maze: null buffer or s <= 0");
  UNREAL_REQUIRE(aligned16(w_taps_bf16) && aligned16(out_bf16) && (reinterpret_cast<uintptr_t>(pos) & 7u) == 0,
                 "unreal_conv1_fwd_maze: alignment (pos 8, buffers 16 bytes)");
  return conv1_fwd_launch<false>(nullptr, pos, w_taps_bf16, bias, out_bf16, s, stream);
}

extern "C" int unreal_conv1_fwd_maze_split(const int32_t* pos, const void* w_hi_bf16, const void* w_lo_bf16, const float* bias,
                                           void* out_hi_bf16, void* out_lo_bf16, int s, void* stream) {
  UNREAL_REQUIRE(pos && w_hi_bf16 && w_lo_bf16 && out_hi_bf16 && out_lo_bf16 && s > 0,
                 "unreal_conv1_fwd_maze_split: null buffer or s <= 0");
  UNREAL_REQUIRE(aligned16(w_hi_bf16) && aligned16(w_lo_bf16) && aligned16(out_hi_bf16) && aligned16(out_lo_bf16) &&
                 (reinterpret_cast<uintptr_t>(pos) & 7u) == 0, "unreal_conv1_fwd_maze_split: alignment (pos 8, buffers 16 bytes)");
  return conv1_fwd_launch<true>(nullptr, pos, w_hi_bf16, bias, out_hi_bf16, s, stream, nullptr, w_lo_bf16, out_lo_bf16);
}

extern "C" int unreal_conv1_fwd_split(const void* xpp_hi_bf16, const void* xpp_lo_bf16, const void* w_hi_bf16,
                                      const void* w_lo_bf16, const float* bias, void* out_hi_bf16, void* out_lo_bf16, int s,
                                      void* stream) {
  UNREAL_REQUIRE(xpp_hi_bf16 && w_hi_bf16 && w_lo_bf16 && out_hi_bf16 && out_lo_bf16 && s > 0,
                 "unreal_conv1_fwd_split: null buffer or s <= 0");
  UNREAL_REQUIRE(aligned16(xpp_hi_bf16) && (xpp_lo_bf16 == nullptr || aligned16(xpp_lo_bf16)) && aligned16(w_hi_bf16) &&
                 aligned16(w_lo_bf16) && aligned16(out_hi_bf16) && aligned16(out_lo_bf16),
                 "unreal_conv1_fwd_split: buffers must be 16-byte aligned");
  return conv1_fwd_launch<true>(xpp_hi_bf16, nullptr, w_hi_bf16, bias, out_hi_bf16, s, stream, xpp_lo_bf16, w_lo_bf16,
                                out_lo_bf16);
}

static int conv_fwd_impl(const void* in_bf16, int layer, const void* w_taps_bf16, const float* bias, void* out_bf16, int s,
                         int relu, void* stream, const float* scale = nullptr, const void* mask_y = nullptr,
                         float* db = nullptr, int c_in = 16, const void* in_lo_bf16 = nullptr, const void* w_lo_bf16 = nullptr) {
  UNREAL_REQUIRE(in_bf16 && w_taps_bf16 && out_bf16 && s > 0, "unreal_conv_fwd: null buffer or s <= 0");
  UNREAL_REQUIRE(mask_y == nullptr || (layer == 2 && bias == nullptr && !relu && aligned16(mask_y)),
                 "unreal_conv2_fwd_linear_masked: conv2 geometry, no bias / ReLU, 16-byte aligned mask");
  UNREAL_REQUIRE(c_in == 16 || (c_in == 8 && mask_y != nullptr), "unreal_conv_fwd: 8 input channels only in the masked conv2 build");
  UNREAL_REQUIRE(layer == 1 || layer == 2, "unreal_conv_fwd: layer must be 1 (conv1 over x') or 2 (conv2 over h1)");
  UNREAL_REQUIRE(aligned16(in_bf16) && aligned16(w_taps_bf16) && aligned16(out_bf16),
                 "unreal_conv_fwd: buffers must be 16-byte aligned");
  const bool split = in_lo_bf16 != nullptr;     // conv2 only (the split conv1 has its own entry point)
  CUtensorMap ta, ta2, tw, tc, talo, talo2, twlo;
  ConvArgs g;
  g.bias = bias;
  g.mode = layer;
  g.relu = relu;
  g.scale = scale;
  g.mask_y = reinterpret_cast<const __nv_bfloat16*>(mask_y);
  g.db = db;
  int rc;
  const int n = layer == 1 ? 16 : 32;
  if (layer == 1) {
    // x'' [S*6 planes][441 pixels][8 ch] bf16: the kernel bulk-copies 126-pixel plane slices
    return conv1_fwd_launch<false>(in_bf16, nullptr, w_taps_bf16, bias, out_bf16, s, stream);
  } else {
    // h1 [S][20][20][16]: image rows y = 2Y' + dy as {64 (4 pixels x 16 c), 9 X (stride 2 pixels: rows overlap),
    // 10 Y', S}, one map per dy; the box at Y' = by is filter row ky = 2by+dy for all 81 outputs
    // (c_in = 8: the same boxes at half the widths -- 64-byte rows, 64-byte swizzle)
    const uint64_t c4 = 4 * (uint64_t)c_in;                       // elements of a box row: 4 pixels x c_in channels
    const uint64_t dims[4] = {c4, 9, 10, (uint64_t)s};
    const uint64_t strides[3] = {c4, 20 * c4, 200 * c4};          // bytes: 2 pixels, 2 image rows, one sample
    const uint32_t box[4] = {(uint32_t)c4, 9, 9, 1};
    rc = make_tma_nd_bf16(&ta, in_bf16, 4, dims, strides, box, 2 * (int)c4);
    if (rc != UNREAL_OK) return rc;
    rc = make_tma_nd_bf16(&ta2, reinterpret_cast<const uint8_t*>(in_bf16) + 10 * c4, 4, dims, strides, box, 2 * (int)c4);
    if (rc == UNREAL_OK && split) {
      rc = make_tma_nd_bf16(&talo, in_lo_bf16, 4, dims, strides, box, 2 * (int)c4);
      if (rc == UNREAL_OK)
        rc = make_tma_nd_bf16(&talo2, reinterpret_cast<const uint8_t*>(in_lo_bf16) + 10 * c4, 4, dims, strides, box, 2 * (int)c4);
    }
    g.items = s; g.rows = 81; g.box_bytes = (int)c4 * 9 * 9 * 2;
  }
  if (rc != UNREAL_OK) return rc;
  {
    const uint64_t k_row = layer == 1 ? 64 : 4 * (uint64_t)c_in;  // [o][(ky,kx,c)]: one k_row-column slice per filter row
    const uint64_t dims[2] = {4 * k_row, (uint64_t)n};
    const uint64_t strides[1] = {8 * k_row};
    const uint32_t box[2] = {(uint32_t)k_row, (uint32_t)n};
    rc = make_tma_nd_bf16(&tw, w_taps_bf16, 2, dims, strides, box, 2 * (int)k_row);
    if (rc == UNREAL_OK && split) rc = make_tma_nd_bf16(&twlo, w_lo_bf16, 2, dims, strides, box, 2 * (int)k_row);
    if (rc != UNREAL_OK) return rc;
  }
  {
    // out [items][rows][n] bf16: the row bound clips the tile's unused rows
    const uint64_t dims[3] = {(uint64_t)n, (uint64_t)g.rows, (uint64_t)g.items};
    const uint64_t strides[2] = {(uint64_t)n * 2, (uint64_t)n * 2 * g.rows};
    const uint32_t box[3] = {64, 32, 1};
    rc = make_tma_nd_bf16(&tc, out_bf16, 3, dims, strides, box, 128);
    if (rc != UNREAL_OK) return rc;
  }
  cudaStream_t st = as_stream(stream);
  if (split) return launch_conv<32, 2, false, 16, true>(ta, ta2, tw, tc, g, st, talo, talo2, twlo);
  if (mask_y != nullptr && c_in == 8) return launch_conv<32, 2, true, 8>(ta, ta2, tw, tc, g, st, ta, ta2, tw);
  if (mask_y != nullptr) return launch_conv<32, 2, true>(ta, ta2, tw, tc, g, st, ta, ta2, tw);
  return launch_conv<32, 2>(ta, ta2, tw, tc, g, st, ta, ta2, tw);
}

extern "C" int unreal_conv_fwd(const void* in_bf16, int layer, const void* w_taps_bf16, const float* bias,
                               void* out_bf16, int s, void* stream) {
  return conv_fwd_impl(in_bf16, layer, w_taps_bf16, bias, out_bf16, s, 1, stream);
}

extern "C" int unreal_conv2_fwd_split(const void* h1_hi_bf16, const void* h1_lo_bf16, const void* w_hi_bf16,
                                      const void* w_lo_bf16, const float* bias, void* out_bf16, int s, void* stream) {
  UNREAL_REQUIRE(h1_lo_bf16 && w_lo_bf16 && aligned16(h1_lo_bf16) && aligned16(w_lo_bf16),
                 "unreal_conv2_fwd_split: null or unaligned lo operand");
  return conv_fwd_impl(h1_hi_bf16, 2, w_hi_bf16, bias, out_bf16, s, 1, stream, nullptr, nullptr, nullptr, 16, h1_lo_bf16,
                       w_lo_bf16);
}

extern "C" int unreal_conv2_fwd_linear(const void* in_bf16, const void* w_taps_bf16, void* out_bf16, int s, void* stream) {
  return conv_fwd_impl(in_bf16, 2, w_taps_bf16, nullptr, out_bf16, s, 0, stream);
}

extern "C" int unreal_conv2_fwd_linear_scaled(const void* in_bf16, const void* w_taps_bf16, const float* scale, void* out_bf16,
                                              int s, void* stream) {
  return conv_fwd_impl(in_bf16, 2, w_taps_bf16, nullptr, out_bf16, s, 0, stream, scale);
}

extern "C" int unreal_conv2_fwd_linear_masked(const void* in_bf16, int c_in, const void* w_taps_bf16, const float* scale,
                                              const void* mask_y_bf16, void* out_bf16, float* db, int s, void* stream) {
  UNREAL_REQUIRE(mask_y_bf16 != nullptr, "unreal_conv2_fwd_linear_masked: null mask");
  UNREAL_REQUIRE(c_in == 16 || c_in == 8, "unreal_conv2_fwd_linear_masked: c_in must be 16 or 8");
  return conv_fwd_impl(in_bf16, 2, w_taps_bf16, nullptr, out_bf16, s, 0, stream, scale, mask_y_bf16, db, c_in);
}

static int conv1_wgrad_launch(const void* xpp_bf16, const void* dy_planes_bf16, float* dw_taps, int s, int pitch21,
                              void* stream, const int32_t* maze_pos = nullptr) {
  UNREAL_REQUIRE(xpp_bf16 && dy_planes_bf16 && dw_taps && s > 0, "unreal_conv1_wgrad: null buffer or s <= 0");
  UNREAL_REQUIRE(aligned16(xpp_bf16) && aligned16(dy_planes_bf16) && aligned16(dw_taps),
                 "unreal_conv1_wgrad: buffers must be 16-byte aligned");
  const int rc = allow_dynamic_smem((const void*)conv1_wgrad_tcgen05_kernel, kWgSmem);
  if (rc != UNREAL_OK) return rc;
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  const uint64_t walls = maze_pos != nullptr ? maze_walls49() : 0;
  const int items = s * 4;
  conv1_wgrad_tcgen05_kernel<<<items < 3 * sms ? items : 3 * sms, 96, kWgSmem, as_stream(stream)>>>(
      reinterpret_cast<const __nv_bfloat16*>(xpp_bf16), reinterpret_cast<const __nv_bfloat16*>(dy_planes_bf16), dw_taps,
      items, (int64_t)s * (pitch21 ? 420 : 400) * 8, pitch21, maze_pos, walls);
  UNREAL_LAUNCH_CHECK("conv1_wgrad_tcgen05_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_conv1_wgrad(const void* xpp_bf16, const void* dy_planes_bf16, float* dw_taps, int s, void* stream) {
  return conv1_wgrad_launch(xpp_bf16, dy_planes_bf16, dw_taps, s, 0, stream);
}

extern "C" int unreal_conv1_wgrad_maze(const int32_t* pos, const void* dy_planes21_bf16, float* dw_taps, int s, void* stream) {
  UNREAL_REQUIRE(pos != nullptr && (reinterpret_cast<uintptr_t>(pos) & 7u) == 0, "unreal_conv1_wgrad_maze: pos null or not 8-byte aligned");
  return conv1_wgrad_launch(dy_planes21_bf16 /* x'' is synthesised; any aligned non-null pointer */, dy_planes21_bf16, dw_taps, s, 1,
                            stream, pos);
}

extern "C" int unreal_conv1_wgrad_p21(const void* xpp_bf16, const void* dy_planes21_bf16, float* dw_taps, int s,
                                      void* stream) {
  return conv1_wgrad_launch(xpp_bf16, dy_planes21_bf16, dw_taps, s, 1, stream);
}

template <int C>
static int conv2_wgrad_launch(const void* h1_bf16, const void* dy_bf16, float* dw_taps, int s, void* stream) {
  UNREAL_REQUIRE(h1_bf16 && dy_bf16 && dw_taps && s > 0, "unreal_conv2_wgrad: null buffer or s <= 0");
  UNREAL_REQUIRE(aligned16(h1_bf16) && aligned16(dy_bf16) && aligned16(dw_taps), "unreal_conv2_wgrad: 16-byte alignment");
  CUtensorMap ta, ta2, td;
  {
    constexpr uint64_t c4 = 4 * C;                              // the forward's overlapping rows of 4 pixels x C channels
    const uint64_t dims[4] = {c4, 9, 10, (uint64_t)s};
    const uint64_t strides[3] = {c4, 20 * c4, 200 * c4};
    const uint32_t box[4] = {(uint32_t)c4, 9, 9, 1};
    int rc = make_tma_nd_bf16(&ta, h1_bf16, 4, dims, strides, box, 2 * (int)c4);
    if (rc != UNREAL_OK) return rc;
    rc = make_tma_nd_bf16(&ta2, reinterpret_cast<const uint8_t*>(h1_bf16) + 10 * c4, 4, dims, strides, box, 2 * (int)c4);
    if (rc != UNREAL_OK) return rc;
  }
  {
    const uint64_t dims[3] = {32, 81, (uint64_t)s};
    const uint64_t strides[2] = {64, 64 * 81};
    const uint32_t box[3] = {32, 96, 1};
    int rc = make_tma_nd_bf16(&td, dy_bf16, 3, dims, strides, box, 64);
    if (rc != UNREAL_OK) return rc;
  }
  const int rc = allow_dynamic_smem((const void*)conv2_wgrad_tcgen05_kernel<C>, W2Cfg<C>::kSmem);
  if (rc != UNREAL_OK) return rc;
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  conv2_wgrad_tcgen05_kernel<C><<<s < 2 * sms ? s : 2 * sms, 128, W2Cfg<C>::kSmem, as_stream(stream)>>>(ta, ta2, td, dw_taps, s);
  UNREAL_LAUNCH_CHECK("conv2_wgrad_tcgen05_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_conv2_wgrad(const void* h1_bf16, const void* dy_bf16, float* dw_taps, int s, void* stream) {
  return conv2_wgrad_launch<16>(h1_bf16, dy_bf16, dw_taps, s, stream);
}

extern "C" int unreal_conv2_wgrad_c8(const void* x8_bf16, const void* dy_bf16, float* dw_taps, int s, void* stream) {
  return conv2_wgrad_launch<8>(x8_bf16, dy_bf16, dw_taps, s, stream);
}

template <int CO, int EPI = 4, int NA = 0, bool PC = false>
static int launch_deconv(const void* dy_bf16, const void* w_dtaps_bf16, void* out, const float* bias, int s, void* stream,
                         const void* mask_y = nullptr, float* db = nullptr, int pitch21 = 0,
                         PcLossArgs pl = PcLossArgs{nullptr, nullptr, nullptr, nullptr, 0, 0.f, nullptr, 0}) {
  CUtensorMap ta, tw;
  {
    const uint64_t dims[4] = {32, 9, 9, (uint64_t)s};           // dY2 [S][9 Y][9 X][32 o]
    const uint64_t strides[3] = {64, 64 * 9, 64 * 81};
    const uint32_t box[4] = {32, 10, 10, 1};                   // one row / column of zero fill around the image
    int rc = make_tma_nd_bf16(&ta, dy_bf16, 4, dims, strides, box, 64);
    if (rc != UNREAL_OK) return rc;
  }
  {
    const uint64_t dims[2] = {32, 16 * CO};                      // [4 taps x 4*CO (dy,dx,c) rows][32 o]
    const uint64_t strides[1] = {64};
    const uint32_t box[2] = {32, 4 * CO};
    int rc = make_tma_nd_bf16(&tw, w_dtaps_bf16, 2, dims, strides, box, 64);
    if (rc != UNREAL_OK) return rc;
  }
  const int rc = allow_dynamic_smem((const void*)conv2_dgrad_tcgen05_kernel<CO, EPI, NA, PC>, kDgSmem);
  if (rc != UNREAL_OK) return rc;
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  conv2_dgrad_tcgen05_kernel<CO, EPI, NA, PC><<<s < 2 * sms ? s : 2 * sms, 64 + 32 * EPI, kDgSmem, as_stream(stream)>>>(
      ta, tw, out, bias, s, reinterpret_cast<const __nv_bfloat16*>(mask_y), db, pitch21, pl);
  UNREAL_LAUNCH_CHECK("conv2_dgrad_tcgen05_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_conv2_dgrad(const void* dy_bf16, const void* w_dtaps_bf16, void* dh1_bf16, int s, void* stream) {
  UNREAL_REQUIRE(dy_bf16 && w_dtaps_bf16 && dh1_bf16 && s > 0, "unreal_conv2_dgrad: null buffer or s <= 0");
  UNREAL_REQUIRE(aligned16(dy_bf16) && aligned16(w_dtaps_bf16) && aligned16(dh1_bf16), "unreal_conv2_dgrad: 16-byte alignment");
  return launch_deconv<16>(dy_bf16, w_dtaps_bf16, dh1_bf16, nullptr, s, stream);
}

extern "C" int unreal_conv2_dgrad_relu(const void* dy_bf16, const void* w_dtaps_bf16, const void* h1_bf16,
                                       void* dy1_planes_bf16, float* db1, int s, int pitch21, void* stream) {
  UNREAL_REQUIRE(dy_bf16 && w_dtaps_bf16 && h1_bf16 && dy1_planes_bf16 && s > 0, "unreal_conv2_dgrad_relu: null buffer or s <= 0");
  UNREAL_REQUIRE(aligned16(dy_bf16) && aligned16(w_dtaps_bf16) && aligned16(h1_bf16) && aligned16(dy1_planes_bf16),
                 "unreal_conv2_dgrad_relu: 16-byte alignment");
  return launch_deconv<16>(dy_bf16, w_dtaps_bf16, dy1_planes_bf16, nullptr, s, stream, h1_bf16, db1, pitch21 ? 1 : 0);
}

extern "C" int unreal_pc_deconv_fwd(const void* h_bf16, const void* w_dtaps_bf16, const float* bias8, float* y8, int s,
                                    void* stream) {
  UNREAL_REQUIRE(h_bf16 && w_dtaps_bf16 && y8 && s > 0, "unreal_pc_deconv_fwd: null buffer or s <= 0");
  UNREAL_REQUIRE(aligned16(h_bf16) && aligned16(w_dtaps_bf16) && aligned16(y8), "unreal_pc_deconv_fwd: 16-byte alignment");
  return launch_deconv<8>(h_bf16, w_dtaps_bf16, y8, bias8, s, stream);
}

static int pc_deconv_loss_impl(const void* h_bf16, const void* w_dtaps_bf16, const float* bias8, const int32_t* act,
                               const float* target, const float* mask, int a, float lam, int s, double* loss,
                               void* dy_bf16, float* db8, int c8, void* stream) {
  UNREAL_REQUIRE(h_bf16 && w_dtaps_bf16 && act && target && mask && dy_bf16 && s > 0,
                 "unreal_pc_deconv_loss: null buffer or s <= 0");
  UNREAL_REQUIRE(a >= 1 && a <= 7, "unreal_pc_deconv_loss: action count %d not in 1..7 (8-channel padded head)", a);
  UNREAL_REQUIRE(aligned16(h_bf16) && aligned16(w_dtaps_bf16) && aligned16(dy_bf16) && aligned16(target),
                 "unreal_pc_deconv_loss: 16-byte alignment");
  const PcLossArgs pl{act, target, mask, loss, a, lam, nullptr, c8};
  if (get_tunable("pc_loss_epi8", 1) != 0) {   // eight epilogue warps (A/B switch for the benchmark scripts)
    // the two action counts of the reference's environments (maze: 4; indoor pointgoal: 3) as compile-time constants
    if (a == 4 && get_tunable("pc_loss_static_a", 1) != 0) return launch_deconv<8, 8, 4>(h_bf16, w_dtaps_bf16, dy_bf16, bias8, s, stream, nullptr, db8, 0, pl);
    if (a == 3 && get_tunable("pc_loss_static_a", 1) != 0) return launch_deconv<8, 8, 3>(h_bf16, w_dtaps_bf16, dy_bf16, bias8, s, stream, nullptr, db8, 0, pl);
    return launch_deconv<8, 8>(h_bf16, w_dtaps_bf16, dy_bf16, bias8, s, stream, nullptr, db8, 0, pl);
  }
  return launch_deconv<8>(h_bf16, w_dtaps_bf16, dy_bf16, bias8, s, stream, nullptr, db8, 0, pl);
}

extern "C" int unreal_pc_deconv_loss(const void* h_bf16, const void* w_dtaps_bf16, const float* bias8, const int32_t* act,
                                     const float* target, const float* mask, int a, float lam, int s, double* loss,
                                     void* dy16_bf16, float* db8, void* stream) {
  return pc_deconv_loss_impl(h_bf16, w_dtaps_bf16, bias8, act, target, mask, a, lam, s, loss, dy16_bf16, db8, 0, stream);
}

extern "C" int unreal_pc_deconv_loss_c8(const void* h_bf16, const void* w_dtaps_bf16, const float* bias8, const int32_t* act,
                                        const float* target, const float* mask, int a, float lam, int s, double* loss,
                                        void* dy8_bf16, float* db8, void* stream) {
  return pc_deconv_loss_impl(h_bf16, w_dtaps_bf16, bias8, act, target, mask, a, lam, s, loss, dy8_bf16, db8, 1, stream);
}

extern "C" int unreal_pc_deconv_loss_planes(const void* h_bf16, const void* w_dtaps_bf16, const float* bias8, const int32_t* act,
                                            const float* target, const float* mask, int a, float lam, int s, double* loss,
                                            void* dy_planes_bf16, float* db8, void* stream) {
  return pc_deconv_loss_impl(h_bf16, w_dtaps_bf16, bias8, act, target, mask, a, lam, s, loss, dy_planes_bf16, db8, 2, stream);
}

extern "C" int unreal_pc_planes_conv(const void* dy_planes_bf16, const void* w_planes_bf16, const float* scale,
                                     const void* mask_y_bf16, void* out_bf16, float* db, int s, void* stream) {
  UNREAL_REQUIRE(dy_planes_bf16 && w_planes_bf16 && mask_y_bf16 && out_bf16 && s > 0, "unreal_pc_planes_conv: null buffer or s <= 0");
  UNREAL_REQUIRE(aligned16(dy_planes_bf16) && aligned16(w_planes_bf16) && aligned16(mask_y_bf16) && aligned16(out_bf16),
                 "unreal_pc_planes_conv: 16-byte alignment");
  const int rc = allow_dynamic_smem((const void*)pc_planes_conv_tcgen05_kernel, kPpSmem);
  if (rc != UNREAL_OK) return rc;
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  pc_planes_conv_tcgen05_kernel<<<s < 2 * sms ? s : 2 * sms, kConvThreads, kPpSmem, as_stream(stream)>>>(
      reinterpret_cast<const __nv_bfloat16*>(dy_planes_bf16), reinterpret_cast<const __nv_bfloat16*>(w_planes_bf16), scale,
      reinterpret_cast<const __nv_bfloat16*>(mask_y_bf16), reinterpret_cast<__nv_bfloat16*>(out_bf16), db, s);
  UNREAL_LAUNCH_CHECK("pc_planes_conv_tcgen05_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_pc_planes_wgrad(const void* dy_planes_bf16, const void* hp_bf16, float* dw8, int s, void* stream) {
  UNREAL_REQUIRE(dy_planes_bf16 && hp_bf16 && dw8 && s > 0, "unreal_pc_planes_wgrad: null buffer or s <= 0");
  UNREAL_REQUIRE(aligned16(dy_planes_bf16) && aligned16(hp_bf16) && aligned16(dw8), "unreal_pc_planes_wgrad: 16-byte alignment");
  CUtensorMap th;
  {
    const uint64_t dims[4] = {32, 9, 9, (uint64_t)s};           // hp [S][9 oy][9 ox][32 o]
    const uint64_t strides[3] = {64, 64 * 9, 64 * 81};
    const uint32_t box[4] = {32, 10, 9, 1};                    // one zero column: the gradient planes' 10-wide grid
    int rc = make_tma_nd_bf16(&th, hp_bf16, 4, dims, strides, box, 64);
    if (rc != UNREAL_OK) return rc;
  }
  const int rc = allow_dynamic_smem((const void*)pc_planes_wgrad_tcgen05_kernel, kPwSmem);
  if (rc != UNREAL_OK) return rc;
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  pc_planes_wgrad_tcgen05_kernel<<<s < 2 * sms ? s : 2 * sms, 128, kPwSmem, as_stream(stream)>>>(
      reinterpret_cast<const __nv_bfloat16*>(dy_planes_bf16), th, dw8, s);
  UNREAL_LAUNCH_CHECK("pc_planes_wgrad_tcgen05_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_pc_deconv_qmax(const void* h_bf16, const void* w_dtaps_bf16, const float* bias8, int a, int s, float* qmax,
                                     void* stream) {
  UNREAL_REQUIRE(h_bf16 && w_dtaps_bf16 && qmax && s > 0, "unreal_pc_deconv_qmax: null buffer or s <= 0");
  UNREAL_REQUIRE(a >= 1 && a <= 7, "unreal_pc_deconv_qmax: action count %d not in 1..7 (8-channel padded head)", a);
  UNREAL_REQUIRE(aligned16(h_bf16) && aligned16(w_dtaps_bf16) && aligned16(qmax), "unreal_pc_deconv_qmax: 16-byte alignment");
  return launch_deconv<8>(h_bf16, w_dtaps_bf16, qmax, bias8, s, stream, nullptr, nullptr, 0,
                          PcLossArgs{nullptr, nullptr, nullptr, nullptr, a, 0.f, qmax, 0});
}

// The 16-channel pixel-control head (8..15 actions): channel 0 the value, 1..A the advantages, no padding channel in the
// loss gradient, which goes to conv2's own backward kernels (unreal_conv2_fwd_linear_masked with c_in 16, unreal_conv2_wgrad).
constexpr int kPc16Epi = 8;

extern "C" int unreal_pc_deconv_loss16(const void* h_bf16, const void* w_dtaps_bf16, const float* bias16, const int32_t* act,
                                       const float* target, const float* mask, int a, float lam, int s, double* loss,
                                       void* dy16_bf16, float* db16, void* stream) {
  UNREAL_REQUIRE(h_bf16 && w_dtaps_bf16 && bias16 && act && target && mask && dy16_bf16 && s > 0,
                 "unreal_pc_deconv_loss16: null buffer or s <= 0");
  UNREAL_REQUIRE(a >= 8 && a <= 15, "unreal_pc_deconv_loss16: action count %d not in 8..15 (16-channel head)", a);
  UNREAL_REQUIRE(aligned16(h_bf16) && aligned16(w_dtaps_bf16) && aligned16(dy16_bf16) && aligned16(target),
                 "unreal_pc_deconv_loss16: 16-byte alignment");
  return launch_deconv<16, kPc16Epi, 0, true>(h_bf16, w_dtaps_bf16, dy16_bf16, bias16, s, stream, nullptr, db16, 0,
                                              PcLossArgs{act, target, mask, loss, a, lam, nullptr, 0});
}

extern "C" int unreal_pc_deconv_qmax16(const void* h_bf16, const void* w_dtaps_bf16, const float* bias16, int a, int s,
                                       float* qmax, void* stream) {
  UNREAL_REQUIRE(h_bf16 && w_dtaps_bf16 && bias16 && qmax && s > 0, "unreal_pc_deconv_qmax16: null buffer or s <= 0");
  UNREAL_REQUIRE(a >= 8 && a <= 15, "unreal_pc_deconv_qmax16: action count %d not in 8..15 (16-channel head)", a);
  UNREAL_REQUIRE(aligned16(h_bf16) && aligned16(w_dtaps_bf16) && aligned16(qmax), "unreal_pc_deconv_qmax16: 16-byte alignment");
  return launch_deconv<16, kPc16Epi, 0, true>(h_bf16, w_dtaps_bf16, qmax, bias16, s, stream, nullptr, nullptr, 0,
                                              PcLossArgs{nullptr, nullptr, nullptr, nullptr, a, 0.f, qmax, 0});
}
