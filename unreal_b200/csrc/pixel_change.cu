// K2: generic pixel change, Environment._calc_pixel_change + _subsample
// (environment/environment.py:88-99) for frames that have no closed form (lab / indoor /
// gym / synthetic):  d = |cur - prev| on the 2-pixel-cropped frame, mean over channels,
// then 4x4 mean (columns first, then rows).
//
// One CTA per (frame, pool row): 4 pixel rows x (W-4) pixels, one thread per pixel, so a warp
// reads consecutive pixels of one row (coalesced).  The three reductions are done in exactly
// numpy's order and roundings -- (d0+d1+d2)/C per pixel, ((m0+m1)+m2)+m3)/4 across a cell row
// (warp shuffles), ((c0+c1)+c2)+c3)/4 down the four rows (shared memory) -- so float32
// frames give bit-identical maps to the reference's float32 evaluation.
// The stream form walks L+1 consecutive frames of a sequence with the previous frame's pixel
// held in registers: every frame is read from HBM exactly once.
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

// grid: (frames-or-sequences x pool rows, column tiles); block: 4 rows x 4*cells pixels, rounded
// up to whole warps (the padding threads only take part in the shuffles)
template <typename T, int C, bool kStream>
__global__ void __launch_bounds__(1024) pixel_change_kernel(const T* __restrict__ cur_or_frames,
                                                            const T* __restrict__ prev, float* __restrict__ pc,
                                                            int H, int W, int ph, int pw, int L) {
  __shared__ float s_rows[4][kMaxCellsPerCta];
  const size_t m = blockIdx.x / ph;               // frame (or sequence)
  const int i = blockIdx.x - (int)m * ph;         // pool row
  const int j0 = blockIdx.y * kMaxCellsPerCta;    // first cell of this tile
  const int cells = min(kMaxCellsPerCta, pw - j0);
  const int tile_px = cells * 4;
  const bool live = threadIdx.x < 4 * tile_px;
  const int r = live ? threadIdx.x / tile_px : 0;  // pixel row inside the pool row, 0..3
  const int p = threadIdx.x - r * tile_px;        // pixel inside the tile
  const size_t frame_elems = (size_t)H * W * C;
  const size_t off = ((size_t)(4 * i + 2 + r) * W + (size_t)(4 * j0 + 2 + p)) * C;
  float a[C], b[C];
#pragma unroll
  for (int c = 0; c < C; ++c) a[c] = b[c] = 0.f;
  if (!kStream) {
    if (live) {
#pragma unroll
      for (int c = 0; c < C; ++c) {
        a[c] = Px<T>::load(cur_or_frames + m * frame_elems + off + c);
        b[c] = Px<T>::load(prev + m * frame_elems + off + c);
      }
    }
    float row = cell_row_mean(pixel_mean<C>(a, b));
    if (live && (p & 3) == 0) s_rows[r][p >> 2] = row;
    __syncthreads();
    if (threadIdx.x < cells) {
      const int j = threadIdx.x;
      float v = __fadd_rn(__fadd_rn(__fadd_rn(s_rows[0][j], s_rows[1][j]), s_rows[2][j]), s_rows[3][j]);
      pc[(m * ph + i) * pw + j0 + j] = __fmul_rn(v, 0.25f);
    }
  } else {
    const T* seq = cur_or_frames + m * (size_t)(L + 1) * frame_elems + off;
    float nx[C];
#pragma unroll
    for (int c = 0; c < C; ++c) nx[c] = 0.f;
    if (live) {
#pragma unroll
      for (int c = 0; c < C; ++c) b[c] = Px<T>::load(seq + c);
#pragma unroll
      for (int c = 0; c < C; ++c) nx[c] = Px<T>::load(seq + frame_elems + c);
    }
    for (int f = 0; f < L; ++f) {
#pragma unroll
      for (int c = 0; c < C; ++c) a[c] = nx[c];
      if (live && f + 1 < L) {  // prefetch the frame after next while this one is reduced
#pragma unroll
        for (int c = 0; c < C; ++c) nx[c] = Px<T>::load(seq + (size_t)(f + 2) * frame_elems + c);
      }
      float row = cell_row_mean(pixel_mean<C>(a, b));
      if (live && (p & 3) == 0) s_rows[r][p >> 2] = row;
      __syncthreads();
      if (threadIdx.x < cells) {
        const int j = threadIdx.x;
        float v = __fadd_rn(__fadd_rn(__fadd_rn(s_rows[0][j], s_rows[1][j]), s_rows[2][j]), s_rows[3][j]);
        pc[((m * L + f) * ph + i) * pw + j0 + j] = __fmul_rn(v, 0.25f);
      }
      __syncthreads();
#pragma unroll
      for (int c = 0; c < C; ++c) b[c] = a[c];
    }
  }
}

template <typename T, bool kStream>
static int launch_c(const void* x, const void* y, float* pc, int m, int l, int h, int w, int c, cudaStream_t st) {
  const int ph = (h - 4) / 4, pw = (w - 4) / 4;
  const int tiles = (pw + kMaxCellsPerCta - 1) / kMaxCellsPerCta;
  const int cells = pw < kMaxCellsPerCta ? pw : kMaxCellsPerCta;
  // every tile but the last is full; the last may be narrower: size the block for the widest
  dim3 grid((unsigned)((size_t)m * ph), tiles), block((16 * cells + 31) / 32 * 32);
  UNREAL_REQUIRE(tiles == 1 || pw % kMaxCellsPerCta == 0,
                 "unreal_pixel_change: frames wider than 260 px need (W-4)/4 to be a multiple of 64");
  const T* a = static_cast<const T*>(x);
  const T* b = static_cast<const T*>(y);
  switch (c) {
    case 1: pixel_change_kernel<T, 1, kStream><<<grid, block, 0, st>>>(a, b, pc, h, w, ph, pw, l); break;
    case 3: pixel_change_kernel<T, 3, kStream><<<grid, block, 0, st>>>(a, b, pc, h, w, ph, pw, l); break;
    case 4: pixel_change_kernel<T, 4, kStream><<<grid, block, 0, st>>>(a, b, pc, h, w, ph, pw, l); break;
    default: UNREAL_REQUIRE(false, "unreal_pixel_change: %d channels not supported (1, 3, 4)", c);
  }
  UNREAL_LAUNCH_CHECK("pixel_change_kernel");
  return UNREAL_OK;
}

// _subsample alone (environment.py:88-91): one thread per output cell, numpy's order of operations
__global__ void subsample_kernel(const float* __restrict__ a, float* __restrict__ out, int H, int W, int width, int oh,
                                 int ow, size_t total) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int j = (int)(idx % ow);
  const int i = (int)((idx / ow) % oh);
  const size_t m = idx / ((size_t)ow * oh);
  const float* base = a + (m * H + (size_t)i * width) * W + (size_t)j * width;
  const float wf = (float)width;
  float acc = 0.f;
  for (int r = 0; r < width; ++r) {
    float s = base[(size_t)r * W];
    for (int c = 1; c < width; ++c) s = __fadd_rn(s, base[(size_t)r * W + c]);
    const float row = __fdiv_rn(s, wf);                 // .mean(-1)
    acc = r == 0 ? row : __fadd_rn(acc, row);
  }
  out[idx] = __fdiv_rn(acc, wf);                        // .mean(1)
}

static int check_shape(const char* fn, int m, int h, int w, int dtype) {
  UNREAL_REQUIRE(m >= 0, "%s: negative batch", fn);
  UNREAL_REQUIRE(h >= 8 && w >= 8 && (h - 4) % 4 == 0 && (w - 4) % 4 == 0,
                 "%s: H-4 and W-4 must be positive multiples of 4 (got %dx%d), as _subsample requires", fn, h, w);
  UNREAL_REQUIRE(dtype == UNREAL_F32 || dtype == UNREAL_U8, "%s: bad dtype %d", fn, dtype);
  UNREAL_REQUIRE((long long)m * ((h - 4) / 4) < 2147483647LL, "%s: batch too large for one launch", fn);
  return UNREAL_OK;
}

}  // namespace unreal

using namespace unreal;

extern "C" int unreal_pixel_change(const void* cur, const void* prev, int dtype, float* pc, int m, int h, int w,
                                   int c, void* stream) {
  int rc = check_shape("unreal_pixel_change", m, h, w, dtype);
  if (rc) return rc;
  if (m == 0) return UNREAL_OK;
  UNREAL_REQUIRE(cur && prev && pc, "unreal_pixel_change: null buffer");
  if (h == 84 && w == 84 && c == 3 && get_tunable("pc84", 1) != 0) {
    const int64_t fb = 84 * 84 * 3 * (dtype == UNREAL_F32 ? 4 : 1);
    rc = pixel_change84(prev, fb, cur, fb, dtype, pc, m, 1, as_stream(stream));
    if (rc != -100) return rc;
  }
  if (dtype == UNREAL_F32) return launch_c<float, false>(cur, prev, pc, m, 0, h, w, c, as_stream(stream));
  return launch_c<uint8_t, false>(cur, prev, pc, m, 0, h, w, c, as_stream(stream));
}

extern "C" int unreal_pixel_change_stream(const void* frames, int dtype, float* pc, int s, int l, int h, int w,
                                          int c, void* stream) {
  int rc = check_shape("unreal_pixel_change_stream", s, h, w, dtype);
  if (rc) return rc;
  UNREAL_REQUIRE(l >= 0, "unreal_pixel_change_stream: negative sequence length");
  if (s == 0 || l == 0) return UNREAL_OK;
  UNREAL_REQUIRE(frames && pc, "unreal_pixel_change_stream: null buffer");
  if (h == 84 && w == 84 && c == 3 && get_tunable("pc84", 1) != 0) {
    const int64_t fb = 84 * 84 * 3 * (dtype == UNREAL_F32 ? 4 : 1);
    rc = pixel_change84(frames, (l + 1) * fb, reinterpret_cast<const uint8_t*>(frames) + fb, (l + 1) * fb, dtype, pc,
                        s, l, as_stream(stream));
    if (rc != -100) return rc;
  }
  if (dtype == UNREAL_F32) return launch_c<float, true>(frames, nullptr, pc, s, l, h, w, c, as_stream(stream));
  return launch_c<uint8_t, true>(frames, nullptr, pc, s, l, h, w, c, as_stream(stream));
}

extern "C" int unreal_subsample(const float* a, float* out, int m, int h, int w, int width, void* stream) {
  UNREAL_REQUIRE(m >= 0 && h > 0 && w > 0 && width > 0, "unreal_subsample: bad sizes");
  UNREAL_REQUIRE(h % width == 0 && w % width == 0, "unreal_subsample: %dx%d is not a multiple of the block width %d", h, w,
                 width);
  if (m == 0) return UNREAL_OK;
  UNREAL_REQUIRE(a && out, "unreal_subsample: null buffer");
  const size_t total = (size_t)m * (h / width) * (w / width);
  subsample_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(a, out, h, w, width, h / width, w / width,
                                                                                 total);
  UNREAL_LAUNCH_CHECK("subsample_kernel");
  return UNREAL_OK;
}
