// K2 fast path: Environment._calc_pixel_change (environment/environment.py:88-99) for 84x84x3
// frames (the lab / indoor / gym observation shape), u8 (/255) or f32, pair or stream form.
//
// HBM-bound design: every frame is read from HBM exactly once, as ONE 16-byte-aligned TMA bulk copy
// of its 2-pixel-cropped rows into a 3-deep ring of shared-memory buffers (prefetch of frame k+2
// overlaps the reduction of frames k-1 / k); a frame serves as `cur` and then as `prev` from shared
// memory.  One thread per 4x4 output cell reads its 4 x 12 values of both frames (word loads at a
// 12-byte stride: bank-conflict free), and reduces in exactly numpy's order and roundings:
//   pixel:  ((|a0-b0| + |a1-b1|) + |a2-b2|) / 3      (abs-diff, mean over channels)
//   cell row: (((m0+m1)+m2)+m3) * 0.25                (mean over the 4 columns first, :90-91)
//   cell:   (((r0+r1)+r2)+r3) * 0.25                  (then over the 4 rows)
// so fp32 results are bit-identical to the generic kernel and to the reference's float32 evaluation.
// u8 frames (`pixel_change84_u8_kernel`): a byte becomes the float32 `v / 255` of lab_environment.py:99-102 in four
// ALU instructions and no memory access -- PRMT drops it into the mantissa of 2^23 (0x4B000000 | v), one FADD
// removes the 2^23, and v / 255 correctly rounded is  fma(v, hi, RN(v * lo))  with hi = RN(1/255),
// lo = RN(1/255 - hi): equal to __fdiv_rn(v, 255) for all 256 byte values (checked exhaustively here on the host at
// library load and by tests/test_gpu_pixel_change.py on the device).  A thread owns one 4x4 cell for a whole
// sequence and keeps the previous frame's 48 converted values in REGISTERS, so every byte is converted once and
// the only shared-memory traffic is 16 word loads per cell and frame.  (Round 1 pushed every byte of both frames
// through a bank-replicated shared-memory table: 192 dependent LDS per cell, LSU-bound at 0.31 of HBM.)
#include "common.cuh"
#include "tc05.cuh"

namespace unreal {
using namespace tc05;

constexpr int kRowElems84 = 84 * 3;   // 252

template <typename T, int PR> struct Pc84 {
  static constexpr int kFrameBytes = 84 * 84 * 3 * (int)sizeof(T);
  static constexpr int kRowBytes = kRowElems84 * (int)sizeof(T);
  static constexpr int kRegionBytes = 4 * PR * kRowBytes;          // the cropped rows of one part
  static constexpr int kParts = 20 / PR;
  static constexpr int kCells = PR * 20;
  static constexpr int kThreads = (kCells + 31) / 32 * 32;
  // the region starts at row 2 + 4*PR*part; copy from the 16-byte boundary below it
  static constexpr int kLead = (2 * kRowBytes) % 16;               // same for every part (4*PR*kRowBytes % 16 == 0)
  static constexpr int kCopyBytes = (kLead + kRegionBytes + 15) / 16 * 16;
  static constexpr int kBufBytes = (kCopyBytes + 127) / 128 * 128;
  static constexpr int kLutBytes = sizeof(T) == 1 ? 256 * 32 * 4 : 0;
  static constexpr int kSmem = 3 * kBufBytes + kLutBytes + 64 /*barriers*/ + 128;
  static_assert((4 * PR * kRowBytes) % 16 == 0, "part stride must keep the 16-byte phase");
};

struct Pc84Args {
  const uint8_t* p0; int64_t stride0;   // frame 0 of sequence s:   p0 + s*stride0
  const uint8_t* p1; int64_t stride1;   // frame f >= 1:            p1 + s*stride1 + (f-1)*frame_bytes
  float* pc;
  int sequences, l;
  uint32_t magic;   // 0x4B000000, passed as a kernel parameter so that it stays an OPERAND (constant bank) of the u8
                    // kernel's PRMTs and their selectors can be immediates
};

__device__ __forceinline__ float pc84_pixel(float a0, float a1, float a2, float b0, float b1, float b2) {
  float s = fabsf(__fsub_rn(a0, b0));
  s = __fadd_rn(s, fabsf(__fsub_rn(a1, b1)));
  s = __fadd_rn(s, fabsf(__fsub_rn(a2, b2)));
  // s / 3, correctly rounded, in three FMA-pipe instructions instead of the ~25 of __fdiv_rn:
  // q = s*RN(1/3) corrected by one exact-remainder step.  Checked against __fdiv_rn for EVERY
  // non-negative finite float on the B200 (scripts/probes/div3_probe.cu: 0 mismatches of 2^31-2^23).
  // (The u8 kernel, which is instruction-bound, uses the two-instruction div3_exact below.)
  const float r = 1.0f / 3.0f;
  const float q = __fmul_rn(s, r);
  return __fmaf_rn(__fmaf_rn(-3.0f, q, s), r, q);
}

template <typename T> struct CellRow;
template <> struct CellRow<uint8_t> {
  // 12 bytes at byte offset `off` (off % 4 == 2) of a shared buffer -> 12 floats through the table
  static __device__ __forceinline__ void load(const uint8_t* buf, int off, const float* lut, float (&v)[12]) {
    const uint32_t* wp = reinterpret_cast<const uint32_t*>(buf + (off - 2));
    uint32_t w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) w[k] = wp[k];
#pragma unroll
    for (int e = 0; e < 12; ++e) {
      const int byte = e + 2;
      v[e] = lut[((w[byte >> 2] >> (8 * (byte & 3))) & 255u) << 5];   // lut already points at this lane's bank
    }
  }
};
template <> struct CellRow<float> {
  static __device__ __forceinline__ void load(const uint8_t* buf, int off, const float*, float (&v)[12]) {
    const float2* fp = reinterpret_cast<const float2*>(buf + off);
#pragma unroll
    for (int k = 0; k < 6; ++k) { const float2 t = fp[k]; v[2 * k] = t.x; v[2 * k + 1] = t.y; }
  }
};

template <typename T, int PR>
__global__ void __launch_bounds__(Pc84<T, PR>::kThreads) pixel_change84_kernel(const Pc84Args g) {
  using P = Pc84<T, PR>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 127u) & ~127u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  float* lut_all = reinterpret_cast<float*>(gen + 3 * P::kBufBytes);
  const uint32_t bar0 = base + 3 * P::kBufBytes + P::kLutBytes;
  const int tid = threadIdx.x;
  if (sizeof(T) == 1) {
    for (int e = tid; e < 256 * 32; e += P::kThreads) lut_all[e] = __fdiv_rn((float)(e >> 5), 255.0f);
  }
  const float* lut = lut_all + (tid & 31);
  if (tid == 0) {
    for (int b = 0; b < 3; ++b) mbar_init(bar0 + 8u * b, 1);
    fence_mbar_init();
  }
  __syncthreads();

  const int items = g.sequences * P::kParts;
  const int nitems = (items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int per = g.l + 1;
  const int total = nitems * per;
  auto issue = [&](int k) {
    const int itn = k / per, f = k - itn * per;
    const int item = (int)blockIdx.x + itn * (int)gridDim.x;
    const int s = item / P::kParts, part = item - s * P::kParts;
    const uint8_t* frame = f == 0 ? g.p0 + (int64_t)s * g.stride0 : g.p1 + (int64_t)s * g.stride1 + (int64_t)(f - 1) * P::kFrameBytes;
    const uint8_t* src = frame + (2 + 4 * PR * part) * P::kRowBytes - P::kLead;
    const uint32_t bar = bar0 + 8u * (k % 3);
    mbar_arrive_expect_tx(bar, P::kCopyBytes);
    bulk_load(base + (uint32_t)(k % 3) * P::kBufBytes, src, P::kCopyBytes, bar);
  };
  if (tid == 0) {
    if (total > 0) issue(0);
    if (total > 1) issue(1);
  }
  const int ci = tid / 20, cj = tid - ci * 20;          // this thread's cell inside the part
  for (int k = 0; k < total; ++k) {
    const int b = k % 3;
    mbar_wait(bar0 + 8u * b, (uint32_t)(k / 3) & 1u);
    const int itn = k / per, f = k - itn * per;
    if (f > 0 && tid < P::kCells) {
      const uint8_t* cur = gen + b * P::kBufBytes;
      const uint8_t* prv = gen + ((k + 2) % 3) * P::kBufBytes;
      float rows[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int off = P::kLead + (4 * ci + r) * P::kRowBytes + (6 + 12 * cj) * (int)sizeof(T);
        float a[12], p[12];
        CellRow<T>::load(cur, off, lut, a);
        CellRow<T>::load(prv, off, lut, p);
        const float m0 = pc84_pixel(a[0], a[1], a[2], p[0], p[1], p[2]);
        const float m1 = pc84_pixel(a[3], a[4], a[5], p[3], p[4], p[5]);
        const float m2 = pc84_pixel(a[6], a[7], a[8], p[6], p[7], p[8]);
        const float m3 = pc84_pixel(a[9], a[10], a[11], p[9], p[10], p[11]);
        rows[r] = __fmul_rn(__fadd_rn(__fadd_rn(__fadd_rn(m0, m1), m2), m3), 0.25f);
      }
      const float cell = __fmul_rn(__fadd_rn(__fadd_rn(__fadd_rn(rows[0], rows[1]), rows[2]), rows[3]), 0.25f);
      const int item = (int)blockIdx.x + itn * (int)gridDim.x;
      const int s = item / P::kParts, part = item - s * P::kParts;
      __stcs(g.pc + ((int64_t)s * g.l + (f - 1)) * 400 + part * P::kCells + tid, cell);
    }
    __syncthreads();                     // frame k-1's buffer is free: prefetch frame k+2 into it
    if (tid == 0 && k + 2 < total) issue(k + 2);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// u8 frames: conversion in registers, previous frame kept in registers (see the header comment)
// ---------------------------------------------------------------------------------------------------------------
// byte `byte` of `word` -> float32 v / 255, correctly rounded: I2F.U8 with the byte selector (one instruction on the
// conversion pipe), then fma(v, hi, RN(v * lo)) with hi = RN(1/255), lo = RN(1/255 - hi).  Equal to __fdiv_rn(v, 255)
// for all 256 values (unreal_selfcheck_arith, tests/test_gpu_pixel_change.py).
__device__ __forceinline__ float u8_over_255(uint32_t word, int byte) {
  const float v = (float)((word >> (8 * byte)) & 0xffu);
  const float hi = 0x1.010102p-8f;
  const float lo = -0x1.fdfdfep-33f;
  return __fmaf_rn(v, hi, __fmul_rn(v, lo));
}

// s / 3 correctly rounded in TWO instructions: fma(s, hi, RN(s * lo)), hi = RN(1/3), lo = RN(1/3 - hi) -- the
// double-word-constant multiplication.  Equal to __fdiv_rn(s, 3) for every float in [2^-100, 2^100] and for 0
// (unreal_selfcheck_arith runs all 2^31 of them on the device; the sums here lie in {0} U [2^-9, 3]).
__device__ __forceinline__ float div3_exact(float s) {
  const float hi = 0x1.555556p-2f;
  const float lo = -0x1.555556p-27f;
  return __fmaf_rn(s, hi, __fmul_rn(s, lo));
}

__device__ __forceinline__ float pc84_pixel2(float a0, float a1, float a2, float b0, float b1, float b2) {
  float s = fabsf(__fsub_rn(a0, b0));
  s = __fadd_rn(s, fabsf(__fsub_rn(a1, b1)));
  s = __fadd_rn(s, fabsf(__fsub_rn(a2, b2)));
  return div3_exact(s);
}

struct Pc84U8 {
  static constexpr int kRowBytes = kRowElems84;                    // 252
  static constexpr int kRegionBytes = 80 * kRowBytes;              // rows 2..81
  static constexpr int kLead = (2 * kRowBytes) % 16;               // 8
  static constexpr int kCopyBytes = (kLead + kRegionBytes + 15) / 16 * 16;
  static constexpr int kBufBytes = (kCopyBytes + 127) / 128 * 128;
  static constexpr int kBufs = 4;
  static constexpr int kComputeWarps = 13;                         // 400 cells + 16 idle lanes
  static constexpr int kThreads = (kComputeWarps + 1) * 32;        // + the TMA producer warp
  static constexpr int kSmem = kBufs * kBufBytes + 128 + 128;
  static constexpr int kFrameBytes = 84 * 84 * 3;
};

// ---- packed fp32x2 arithmetic (Blackwell FADD2 / FMUL2 / FFMA2: two IEEE-rounded fp32 operations per issue slot; the
// kernel is issue-bound, not lane-bound).  A pair holds the SAME byte position of two consecutive pixel rows.
__device__ __forceinline__ float2 f2(float v) { return make_float2(v, v); }
__device__ __forceinline__ float2 neg2(float2 a) { return make_float2(-a.x, -a.y); }       // folds into the -R operand modifier
__device__ __forceinline__ float2 abs2(float2 a) { return make_float2(fabsf(a.x), fabsf(a.y)); }   // |R| operand modifier

// byte `byte` of the two rows' words -> (v0 / 255, v1 / 255), each correctly rounded: PRMT drops the byte into the
// mantissa of 2^23 (0x4B000000 | v), one FADD2 removes the 2^23 from both, then fma(v, hi, RN(v * lo)) with
// hi = RN(1/255), lo = RN(1/255 - hi): 2 + 3 issue slots for two bytes.  kXu: convert through I2F.U8 instead (one slot
// per byte, but on the 16-lane conversion pipe) -- used for a few byte positions to balance the pipes.
// `magic` = 0x4B000000 arrives as a kernel parameter (PRMT takes a single immediate: with the constant folded into it
// the compiler re-materialises a selector register per PRMT -- 40 extra MOVs per frame)

template <bool kXu>
__device__ __forceinline__ float2 u8pair_over_255(uint32_t w0, uint32_t w1, int byte, uint32_t magic) {
  float2 v;
  if (kXu) {
    v.x = (float)((w0 >> (8 * byte)) & 0xffu);
    v.y = (float)((w1 >> (8 * byte)) & 0xffu);
  } else {
    float2 m;
    m.x = __uint_as_float(__byte_perm(w0, magic, 0x7540u | (uint32_t)byte));
    m.y = __uint_as_float(__byte_perm(w1, magic, 0x7540u | (uint32_t)byte));
    v = __fadd2_rn(m, f2(-8388608.0f));
  }
  return __ffma2_rn(v, f2(0x1.010102p-8f), __fmul2_rn(v, f2(-0x1.fdfdfep-33f)));
}

// ((|a0-b0| + |a1-b1|) + |a2-b2|) / 3 for two pixels at once
__device__ __forceinline__ float2 pc84_pixel_pair(float2 a0, float2 a1, float2 a2, float2 b0, float2 b1, float2 b2) {
  const float2 d0 = __fadd2_rn(a0, neg2(b0)), d1 = __fadd2_rn(a1, neg2(b1)), d2 = __fadd2_rn(a2, neg2(b2));
  float2 s = __fadd2_rn(abs2(d0), abs2(d1));
  s = __fadd2_rn(s, abs2(d2));
  return __ffma2_rn(s, f2(0x1.555556p-2f), __fmul2_rn(s, f2(-0x1.555556p-27f)));       // div3_exact, both lanes
}

// one frame of one cell: 4 x 4 word loads, 48 conversions into cur[] (pairs of rows), the 16 pixel means against prev[]
template <int kXuBytes>
__device__ __forceinline__ float pc84_u8_cell(const uint8_t* cellp, float2 (&cur)[24], const float2 (&prev)[24], uint32_t magic) {
  float2 rows[2];
#pragma unroll
  for (int rp = 0; rp < 2; ++rp) {
    const uint32_t* wa = reinterpret_cast<const uint32_t*>(cellp + (2 * rp) * Pc84U8::kRowBytes);
    const uint32_t* wb = reinterpret_cast<const uint32_t*>(cellp + (2 * rp + 1) * Pc84U8::kRowBytes);
    const uint32_t a4[4] = {wa[0], wa[1], wa[2], wa[3]};
    const uint32_t b4[4] = {wb[0], wb[1], wb[2], wb[3]};
    float2* a = cur + rp * 12;
    const float2* p = prev + rp * 12;
#pragma unroll
    for (int e = 0; e < 12; ++e) {
      if (e < kXuBytes) a[e] = u8pair_over_255<true>(a4[(e + 2) >> 2], b4[(e + 2) >> 2], (e + 2) & 3, magic);
      else a[e] = u8pair_over_255<false>(a4[(e + 2) >> 2], b4[(e + 2) >> 2], (e + 2) & 3, magic);
    }
    const float2 m0 = pc84_pixel_pair(a[0], a[1], a[2], p[0], p[1], p[2]);
    const float2 m1 = pc84_pixel_pair(a[3], a[4], a[5], p[3], p[4], p[5]);
    const float2 m2 = pc84_pixel_pair(a[6], a[7], a[8], p[6], p[7], p[8]);
    const float2 m3 = pc84_pixel_pair(a[9], a[10], a[11], p[9], p[10], p[11]);
    rows[rp] = __fmul2_rn(__fadd2_rn(__fadd2_rn(__fadd2_rn(m0, m1), m2), m3), f2(0.25f));    // mean over the 4 columns
  }
  return __fmul_rn(__fadd_rn(__fadd_rn(__fadd_rn(rows[0].x, rows[0].y), rows[1].x), rows[1].y), 0.25f);   // then the 4 rows
}

// Warp-specialised: warp 13 is the TMA producer (one bulk copy per frame into a 4-deep ring, gated by per-buffer `empty`
// barriers), warps 0..12 own one cell per thread and run free of each other -- a warp waits on `full[b]`, reduces its
// cells and arrives on `empty[b]`; there is no CTA-wide barrier in the loop.  The previous frame's 48 values ping-pong
// between two register arrays (frame k in A against B, frame k+1 in B against A: no copies).
template <int kXuBytes>
__global__ void __launch_bounds__(Pc84U8::kThreads, 1) pixel_change84_u8_kernel(const Pc84Args g) {
  using P = Pc84U8;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 127u) & ~127u;
  const uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t full0 = base + P::kBufs * P::kBufBytes;
  const uint32_t empty0 = full0 + 8u * P::kBufs;
  const int tid = threadIdx.x;
  if (tid == 0) {
    for (int b = 0; b < P::kBufs; ++b) { mbar_init(full0 + 8u * b, 1); mbar_init(empty0 + 8u * b, P::kComputeWarps); }
    fence_mbar_init();
  }
  __syncthreads();
  const int items = g.sequences;
  const int nitems = (items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int per = g.l + 1;
  const int total = nitems * per;
  const int warp = tid >> 5, lane = tid & 31;

  if (warp == P::kComputeWarps) {                      // ---- producer
    if (lane == 0) {
      for (int k = 0; k < total; ++k) {
        const int b = k % P::kBufs;
        if (k >= P::kBufs) mbar_wait(empty0 + 8u * b, (uint32_t)(k / P::kBufs - 1) & 1u);
        const int itn = k / per, f = k - itn * per;
        const int s = (int)blockIdx.x + itn * (int)gridDim.x;
        const uint8_t* frame = f == 0 ? g.p0 + (int64_t)s * g.stride0 : g.p1 + (int64_t)s * g.stride1 + (int64_t)(f - 1) * P::kFrameBytes;
        const uint8_t* src = frame + 2 * P::kRowBytes - P::kLead;
        const uint32_t bar = full0 + 8u * b;
        mbar_arrive_expect_tx(bar, P::kCopyBytes);
        bulk_load(base + (uint32_t)b * P::kBufBytes, src, P::kCopyBytes, bar);
      }
    }
    return;
  }

  const bool live = tid < 400;                         // ---- consumers
  const int cell = live ? tid : 0;
  const int ci = cell / 20, cj = cell - ci * 20;
  // byte offset of the word holding the cell's first byte (the cell starts 2 bytes into it: (6 + 12 cj) % 4 == 2)
  const int off0 = P::kLead + 4 * ci * P::kRowBytes + (6 + 12 * cj) - 2;
  const uint32_t magic = g.magic;
  float2 A[24], B[24];
#pragma unroll
  for (int e = 0; e < 24; ++e) A[e] = B[e] = make_float2(0.f, 0.f);
  auto step = [&](int k, float2 (&cur)[24], const float2 (&prev)[24]) {
    const int b = k % P::kBufs;
    mbar_wait(full0 + 8u * b, (uint32_t)(k / P::kBufs) & 1u);
    const float v = pc84_u8_cell<kXuBytes>(gen + b * P::kBufBytes + off0, cur, prev, magic);
    __syncwarp();
    if (lane == 0) mbar_arrive(empty0 + 8u * b);       // this warp is done with buffer b
    const int itn = k / per, f = k - itn * per;
    if (f > 0 && live) {
      const int s = (int)blockIdx.x + itn * (int)gridDim.x;
      __stcs(g.pc + ((int64_t)s * g.l + (f - 1)) * 400 + tid, v);
    }
  };
  for (int k = 0; k < total; k += 2) {
    step(k, A, B);
    if (k + 1 < total) step(k + 1, B, A);
  }
}

template <int kXuBytes>
static int launch84_u8(const Pc84Args& g, cudaStream_t st) {
  using P = Pc84U8;
  auto kern = pixel_change84_u8_kernel<kXuBytes>;
  const int rc = allow_dynamic_smem((const void*)kern, P::kSmem);
  if (rc != UNREAL_OK) return rc;
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  const int grid = g.sequences < sms ? g.sequences : sms;
  kern<<<grid, P::kThreads, P::kSmem, st>>>(g);
  UNREAL_LAUNCH_CHECK("pixel_change84_u8_kernel");
  return UNREAL_OK;
}

// Exhaustive device check of the two division-free roundings above against __fdiv_rn.
__global__ void selfcheck_arith_kernel(unsigned long long* out, uint32_t mg) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  const uint64_t id = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long bad3 = 0, bad255 = 0;
  // every float in [2^-100, 2^100): exponent fields 27 .. 226
  for (uint64_t i = (27ull << 23) + id; i < (227ull << 23); i += stride) {
    const float s = __uint_as_float((uint32_t)i);
    if (__float_as_uint(div3_exact(s)) != __float_as_uint(__fdiv_rn(s, 3.0f))) ++bad3;
  }
  if (id == 0 && __float_as_uint(div3_exact(0.f)) != 0u) ++bad3;
  if (id < 256 * 4) {                                   // every byte value in every byte lane of a word
    const uint32_t v = (uint32_t)(id >> 2), lane_b = (uint32_t)(id & 3);
    const uint32_t word = (v << (8 * lane_b)) | (0xA5A5A5A5u & ~(0xffu << (8 * lane_b)));
    float2 g0, g1;                                      // both conversion paths, both lanes of the packed pair
    switch (lane_b) {
      case 0: g0 = u8pair_over_255<false>(word, ~word, 0, mg); g1 = u8pair_over_255<true>(~word, word, 0, mg); break;
      case 1: g0 = u8pair_over_255<false>(word, ~word, 1, mg); g1 = u8pair_over_255<true>(~word, word, 1, mg); break;
      case 2: g0 = u8pair_over_255<false>(word, ~word, 2, mg); g1 = u8pair_over_255<true>(~word, word, 2, mg); break;
      default: g0 = u8pair_over_255<false>(word, ~word, 3, mg); g1 = u8pair_over_255<true>(~word, word, 3, mg); break;
    }
    const uint32_t want = __float_as_uint(__fdiv_rn((float)v, 255.0f));
    const uint32_t wantn = __float_as_uint(__fdiv_rn((float)(255u - v), 255.0f));
    if (__float_as_uint(g0.x) != want || __float_as_uint(g0.y) != wantn) ++bad255;
    if (__float_as_uint(g1.x) != wantn || __float_as_uint(g1.y) != want) ++bad255;
    if (__float_as_uint(u8_over_255(word, (int)lane_b)) != want) ++bad255;
    const float2 t3 = pc84_pixel_pair(f2(0.f), f2(0.f), f2(0.f), make_float2((float)v, 0.f), f2(0.f), make_float2(0.f, (float)v * 0.5f));
    if (__float_as_uint(t3.x) != __float_as_uint(__fdiv_rn((float)v, 3.0f)) ||
        __float_as_uint(t3.y) != __float_as_uint(__fdiv_rn((float)v * 0.5f, 3.0f))) ++bad255;
  }
  if (bad3) atomicAdd(out, bad3);
  if (bad255) atomicAdd(out + 1, bad255);
}

template <typename T, int PR>
static int launch84(const Pc84Args& g, cudaStream_t st) {
  using P = Pc84<T, PR>;
  auto kern = pixel_change84_kernel<T, PR>;
  const int rc = allow_dynamic_smem((const void*)kern, P::kSmem);
  if (rc != UNREAL_OK) return rc;
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  const int per_sm = (227 * 1024) / (P::kSmem + 1024);
  const int64_t items = (int64_t)g.sequences * P::kParts;
  const int64_t cap = (int64_t)sms * (per_sm < 1 ? 1 : per_sm);
  const int grid = (int)(items < cap ? items : cap);
  kern<<<grid, P::kThreads, P::kSmem, st>>>(g);
  UNREAL_LAUNCH_CHECK("pixel_change84_kernel");
  return UNREAL_OK;
}

// p0/p1 as in Pc84Args; returns UNREAL_OK after enqueueing, or -100 when the fast path does not apply
int pixel_change84(const void* p0, int64_t stride0, const void* p1, int64_t stride1, int dtype, float* pc,
                   int sequences, int l, cudaStream_t st) {
  if (!aligned16(p0) || !aligned16(p1)) return -100;
  Pc84Args g{reinterpret_cast<const uint8_t*>(p0), stride0, reinterpret_cast<const uint8_t*>(p1), stride1, pc,
             sequences, l, 0x4B000000u};
  if (dtype == UNREAL_U8) {
    if (get_tunable("pc84_u8_lut", 0) != 0) return launch84<uint8_t, 20>(g, st);   // round-1 table kernel (A/B)
    switch (get_tunable("pc84_u8_xu_bytes", 0)) {     // byte positions (of 12 per row) converted on the I2F pipe
      case 2: return launch84_u8<2>(g, st);
      case 4: return launch84_u8<4>(g, st);
      default: return launch84_u8<0>(g, st);
    }
  }
  return launch84<float, 10>(g, st);
}

}  // namespace unreal

// mismatches[0]: floats s in [2^-100, 2^100] (and 0) where the two-instruction s/3 differs from __fdiv_rn(s, 3);
// mismatches[1]: (byte value, byte lane) pairs where the three-instruction v/255 differs from __fdiv_rn(v, 255).
extern "C" int unreal_selfcheck_arith(unsigned long long* mismatches, void* stream) {
  UNREAL_REQUIRE(mismatches != nullptr, "unreal_selfcheck_arith: null output");
  cudaStream_t st = unreal::as_stream(stream);
  UNREAL_CUDA(cudaMemsetAsync(mismatches, 0, 2 * sizeof(unsigned long long), st));
  unreal::selfcheck_arith_kernel<<<148 * 8, 256, 0, st>>>(mismatches, 0x4B000000u);
  UNREAL_LAUNCH_CHECK("selfcheck_arith_kernel");
  return UNREAL_OK;
}
