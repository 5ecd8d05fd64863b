// K7 support kernels around the tcgen05 GEMM: the non-GEMM pieces of UnrealModel's dense layers
// (model/model.py:281-443).  All are HBM-bound data movement / pointwise work.
//
//   im2col / col2im   tf.nn.conv2d (:786-787) and tf.nn.conv2d_transpose (:803-820) with VALID
//                     padding on NHWC tensors, expressed around a GEMM: patches are rows of a
//                     [S*OH*OW, KH*KW*C] matrix whose column index is (ky*KW + kx)*C + c -- the
//                     row-major order of TF's HWIO filter, so weights are used where they lie.
//   lstm cell         contrib.rnn.BasicLSTMCell (:110): gates i, j, f, o, forget_bias 1.0.
#include <cuda_bf16.h>

#include "common.cuh"

namespace unreal {

struct ConvGeom {
  int s, h, w, c, kh, kw, stride, oh, ow;
};

template <typename T> struct In;
template <> struct In<float> { static __device__ __forceinline__ float ld(const float* p) { return *p; } };
template <> struct In<uint8_t> {
  // frames stored as uint8 are scaled by 1/255 on load (lab_environment.py:99-102)
  static __device__ __forceinline__ float ld(const uint8_t* p) { return __fdiv_rn((float)*p, 255.0f); }
};
template <> struct In<__nv_bfloat16> {
  static __device__ __forceinline__ float ld(const __nv_bfloat16* p) { return __bfloat162float(*p); }
};

// One thread per chunk of V consecutive elements inside one patch-row segment (KW*C contiguous
// input elements).  Consecutive threads walk one output row, so stores are fully coalesced.
template <typename T, int V>
__global__ void __launch_bounds__(256) im2col_kernel(const T* __restrict__ in, __nv_bfloat16* __restrict__ out,
                                                     ConvGeom g, int64_t total_chunks) {
  const int seg = g.kw * g.c;            // contiguous input run
  const int chunks_per_seg = seg / V;
  const int k = g.kh * seg;              // output row length
  for (int64_t id = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; id < total_chunks;
       id += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = id;
    const int ch = (int)(r % chunks_per_seg); r /= chunks_per_seg;
    const int ky = (int)(r % g.kh); r /= g.kh;
    const int ox = (int)(r % g.ow); r /= g.ow;
    const int oy = (int)(r % g.oh); r /= g.oh;
    const int64_t s = r;
    const T* src = in + (((s * g.h + (oy * g.stride + ky)) * g.w + ox * g.stride) * (int64_t)g.c) + ch * V;
    __nv_bfloat16* dst = out + (((s * g.oh + oy) * g.ow + ox) * (int64_t)k) + ky * seg + ch * V;
    if (V == 8) {
      float v[8];
      if (sizeof(T) == 4) {
        const float4 a = *reinterpret_cast<const float4*>(src);
        const float4 b = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(src) + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
      } else if (sizeof(T) == 2) {
        const uint4 u = *reinterpret_cast<const uint4*>(src);
        *reinterpret_cast<uint4*>(dst) = u;  // bf16 -> bf16: plain 16-byte move
        continue;
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = In<T>::ld(src + j);
      }
      __nv_bfloat162 p0 = __floats2bfloat162_rn(v[0], v[1]), p1 = __floats2bfloat162_rn(v[2], v[3]);
      __nv_bfloat162 p2 = __floats2bfloat162_rn(v[4], v[5]), p3 = __floats2bfloat162_rn(v[6], v[7]);
      uint4 u;
      u.x = *reinterpret_cast<uint32_t*>(&p0); u.y = *reinterpret_cast<uint32_t*>(&p1);
      u.z = *reinterpret_cast<uint32_t*>(&p2); u.w = *reinterpret_cast<uint32_t*>(&p3);
      *reinterpret_cast<uint4*>(dst) = u;
    } else {
      dst[0] = __float2bfloat16_rn(In<T>::ld(src));
    }
  }
}

// Gather form of col2im: out[s,y,x,c] = act(bias[c] + sum over taps (ky,kx) with
// y = oy*stride + ky, x = ox*stride + kx of cols[(s,oy,ox), (ky*KW+kx)*C + c]).
template <typename TC, typename TO>
__global__ void __launch_bounds__(256) col2im_kernel(const TC* __restrict__ cols, TO* __restrict__ out,
                                                     const float* __restrict__ bias, int relu, ConvGeom g,
                                                     int64_t total) {
  const int k = g.kh * g.kw * g.c;
  for (int64_t id = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; id < total; id += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = id;
    const int c = (int)(r % g.c); r /= g.c;
    const int x = (int)(r % g.w); r /= g.w;
    const int y = (int)(r % g.h); r /= g.h;
    const int64_t s = r;
    float acc = bias ? bias[c] : 0.f;
    for (int ky = y % g.stride; ky < g.kh; ky += g.stride) {
      const int oy = (y - ky) / g.stride;
      if (y - ky < 0 || oy >= g.oh) continue;
      for (int kx = x % g.stride; kx < g.kw; kx += g.stride) {
        const int ox = (x - kx) / g.stride;
        if (x - kx < 0 || ox >= g.ow) continue;
        acc += In<TC>::ld(cols + ((s * g.oh + oy) * g.ow + ox) * (int64_t)k + (ky * g.kw + kx) * g.c + c);
      }
    }
    if (relu) acc = fmaxf(acc, 0.f);
    if (sizeof(TO) == 2) reinterpret_cast<__nv_bfloat16*>(out)[id] = __float2bfloat16_rn(acc);
    else reinterpret_cast<float*>(out)[id] = acc;
  }
}

// 8 channels per thread (one 16-byte load per tap): the conv2 dgrad case, C = 16, bf16 in / out.
template <typename TO>
__global__ void __launch_bounds__(256) col2im_vec8_kernel(const __nv_bfloat16* __restrict__ cols, TO* __restrict__ out,
                                                          const float* __restrict__ bias, int relu, ConvGeom g,
                                                          int64_t total8) {
  const int k = g.kh * g.kw * g.c;
  const int c8n = g.c >> 3;
  for (int64_t id = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; id < total8; id += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = id;
    const int c = (int)(r % c8n) * 8; r /= c8n;
    const int x = (int)(r % g.w); r /= g.w;
    const int y = (int)(r % g.h); r /= g.h;
    const int64_t s = r;
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = bias ? bias[c + j] : 0.f;
    for (int ky = y % g.stride; ky < g.kh; ky += g.stride) {
      const int oy = (y - ky) / g.stride;
      if (y - ky < 0 || oy >= g.oh) continue;
      for (int kx = x % g.stride; kx < g.kw; kx += g.stride) {
        const int ox = (x - kx) / g.stride;
        if (x - kx < 0 || ox >= g.ow) continue;
        const uint4 u = *reinterpret_cast<const uint4*>(cols + ((s * g.oh + oy) * g.ow + ox) * (int64_t)k +
                                                        (ky * g.kw + kx) * g.c + c);
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = __bfloat1622float2(h[j]);
          acc[2 * j] += f.x; acc[2 * j + 1] += f.y;
        }
      }
    }
    if (relu) {
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = fmaxf(acc[j], 0.f);
    }
    if (sizeof(TO) == 2) {
      __nv_bfloat162 p0 = __floats2bfloat162_rn(acc[0], acc[1]), p1 = __floats2bfloat162_rn(acc[2], acc[3]);
      __nv_bfloat162 p2 = __floats2bfloat162_rn(acc[4], acc[5]), p3 = __floats2bfloat162_rn(acc[6], acc[7]);
      uint4 o;
      o.x = *reinterpret_cast<uint32_t*>(&p0); o.y = *reinterpret_cast<uint32_t*>(&p1);
      o.z = *reinterpret_cast<uint32_t*>(&p2); o.w = *reinterpret_cast<uint32_t*>(&p3);
      reinterpret_cast<uint4*>(out)[id] = o;
    } else {
      float4* o = reinterpret_cast<float4*>(out) + id * 2;
      o[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
      o[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
    }
  }
}

// ---- BasicLSTMCell pointwise -----------------------------------------------------------
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + __expf(-x)); }

// Gate storage type: float, or bf16 (UnrealModel.lstm_gates_bf16: the step GEMM writes the pre-activations as bf16 and
// the activations kept for the backward pass are bf16 as well -- the cell kernels are HBM-bound on exactly that buffer:
// 95 MB per step at 8192 envs in f32, 61 MB in bf16; the rounding is that of every other activation between layers).
template <typename TG> struct Gate;
template <> struct Gate<float> {
  static __device__ __forceinline__ float ld(const float* p) { return *p; }
  static __device__ __forceinline__ void st(float* p, float v) { *p = v; }
};
template <> struct Gate<__nv_bfloat16> {
  static __device__ __forceinline__ float ld(const __nv_bfloat16* p) { return __bfloat162float(*p); }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
};

// gates [N,1024] pre-activations (i | j | f | o blocks of 256) are replaced by their activations
template <typename TG>
__global__ void __launch_bounds__(256) lstm_cell_fwd_kernel(TG* __restrict__ gates, const float* __restrict__ c_prev,
                                                            float* __restrict__ c_out, float* __restrict__ h_out,
                                                            __nv_bfloat16* __restrict__ h16_out, int n, int h16_ld) {
  const int id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= n * 256) return;
  const int e = id >> 8, u = id & 255;
  TG* gr = gates + (size_t)e * 1024;
  const float i = sigmoidf_(Gate<TG>::ld(gr + u));
  const float j = tanhf(Gate<TG>::ld(gr + 256 + u));
  const float f = sigmoidf_(Gate<TG>::ld(gr + 512 + u) + 1.0f);   // forget_bias = 1.0
  const float o = sigmoidf_(Gate<TG>::ld(gr + 768 + u));
  const float c = c_prev[id] * f + i * j;
  const float h = tanhf(c) * o;
  Gate<TG>::st(gr + u, i); Gate<TG>::st(gr + 256 + u, j); Gate<TG>::st(gr + 512 + u, f); Gate<TG>::st(gr + 768 + u, o);
  c_out[id] = c;
  h_out[id] = h;
  h16_out[(size_t)e * h16_ld + u] = __float2bfloat16_rn(h);     // h16_ld > 256: straight into the next step's [x, h] GEMM operand
}

// Acting step: the cell applied IN PLACE to the persistent state of the envs with active[e] != 0 (the others keep
// their state and report their old h): replaces cell + two masked selects + two copies per env step.
template <typename TG>
__global__ void __launch_bounds__(256) lstm_cell_act_kernel(const TG* __restrict__ gates, float* __restrict__ c_state,
                                                            float* __restrict__ h_state, float* __restrict__ h_out,
                                                            const uint8_t* __restrict__ active, int n) {
  const int id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= n * 256) return;
  const int e = id >> 8, u = id & 255;
  if (active != nullptr && active[e] == 0) {
    if (h_out != nullptr) h_out[id] = h_state[id];
    return;
  }
  const TG* gr = gates + (size_t)e * 1024;
  const float i = sigmoidf_(Gate<TG>::ld(gr + u));
  const float j = tanhf(Gate<TG>::ld(gr + 256 + u));
  const float f = sigmoidf_(Gate<TG>::ld(gr + 512 + u) + 1.0f);   // forget_bias = 1.0
  const float o = sigmoidf_(Gate<TG>::ld(gr + 768 + u));
  const float c = c_state[id] * f + i * j;
  const float h = tanhf(c) * o;
  c_state[id] = c;
  h_state[id] = h;
  if (h_out != nullptr) h_out[id] = h;
}

// bf16 gate storage, 8 units per thread (16-byte accesses): the scalar form above issues 13 two- and four-byte memory
// instructions per unit and was LSU-instruction-bound (14.6 us for 61 MB at 8192 envs)
struct __align__(16) Bf8 { __nv_bfloat162 v[4]; };
__device__ __forceinline__ void bf8_unpack(const Bf8& b, float (&f)[8]) {
#pragma unroll
  for (int k = 0; k < 4; ++k) { const float2 t = __bfloat1622float2(b.v[k]); f[2 * k] = t.x; f[2 * k + 1] = t.y; }
}
__device__ __forceinline__ Bf8 bf8_pack(const float (&f)[8]) {
  Bf8 b;
#pragma unroll
  for (int k = 0; k < 4; ++k) b.v[k] = __floats2bfloat162_rn(f[2 * k], f[2 * k + 1]);
  return b;
}

__device__ __forceinline__ void lstm_cell8(const __nv_bfloat16* gr, const float* cp_ptr, float (&zi)[8], float (&zj)[8],
                                           float (&zf)[8], float (&zo)[8], float (&c)[8], float (&h)[8]) {
  float cp[8];
  bf8_unpack(*reinterpret_cast<const Bf8*>(gr), zi);
  bf8_unpack(*reinterpret_cast<const Bf8*>(gr + 256), zj);
  bf8_unpack(*reinterpret_cast<const Bf8*>(gr + 512), zf);
  bf8_unpack(*reinterpret_cast<const Bf8*>(gr + 768), zo);
  *reinterpret_cast<float4*>(cp) = reinterpret_cast<const float4*>(cp_ptr)[0];
  *reinterpret_cast<float4*>(cp + 4) = reinterpret_cast<const float4*>(cp_ptr)[1];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    zi[k] = sigmoidf_(zi[k]);
    zj[k] = tanhf(zj[k]);
    zf[k] = sigmoidf_(zf[k] + 1.0f);   // forget_bias = 1.0
    zo[k] = sigmoidf_(zo[k]);
    c[k] = cp[k] * zf[k] + zi[k] * zj[k];
    h[k] = tanhf(c[k]) * zo[k];
  }
}
__device__ __forceinline__ void st8(float* p, const float (&v)[8]) {
  reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
  reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
}

// training step: activations written back over the pre-activations, c / h / h16 out
__global__ void __launch_bounds__(256) lstm_cell_fwd8_kernel(__nv_bfloat16* __restrict__ gates, const float* __restrict__ c_prev,
                                                             float* __restrict__ c_out, float* __restrict__ h_out,
                                                             __nv_bfloat16* __restrict__ h16_out, int n, int h16_ld) {
  const int id = blockIdx.x * blockDim.x + threadIdx.x;     // one thread per 8 units
  if (id >= n * 32) return;
  const int e = id >> 5, u = (id & 31) * 8;
  const size_t so = (size_t)e * 256 + u;
  __nv_bfloat16* gr = gates + (size_t)e * 1024 + u;
  float zi[8], zj[8], zf[8], zo[8], c[8], h[8];
  lstm_cell8(gr, c_prev + so, zi, zj, zf, zo, c, h);
  *reinterpret_cast<Bf8*>(gr) = bf8_pack(zi);
  *reinterpret_cast<Bf8*>(gr + 256) = bf8_pack(zj);
  *reinterpret_cast<Bf8*>(gr + 512) = bf8_pack(zf);
  *reinterpret_cast<Bf8*>(gr + 768) = bf8_pack(zo);
  st8(c_out + so, c);
  st8(h_out + so, h);
  *reinterpret_cast<Bf8*>(h16_out + (size_t)e * h16_ld + u) = bf8_pack(h);
}

// acting step, in place on the persistent state of the envs with active[e] != 0 (the others report their old h)
__global__ void __launch_bounds__(256) lstm_cell_act8_kernel(const __nv_bfloat16* __restrict__ gates, float* __restrict__ c_state,
                                                             float* __restrict__ h_state, float* __restrict__ h_out,
                                                             const uint8_t* __restrict__ active, int n) {
  const int id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= n * 32) return;
  const int e = id >> 5, u = (id & 31) * 8;
  const size_t so = (size_t)e * 256 + u;
  if (active != nullptr && active[e] == 0) {
    if (h_out != nullptr) {
      reinterpret_cast<float4*>(h_out + so)[0] = reinterpret_cast<const float4*>(h_state + so)[0];
      reinterpret_cast<float4*>(h_out + so)[1] = reinterpret_cast<const float4*>(h_state + so)[1];
    }
    return;
  }
  float zi[8], zj[8], zf[8], zo[8], c[8], h[8];
  lstm_cell8(gates + (size_t)e * 1024 + u, c_state + so, zi, zj, zf, zo, c, h);
  st8(c_state + so, c);
  st8(h_state + so, h);
  if (h_out != nullptr) st8(h_out + so, h);
}

// dh: total gradient wrt h_t (heads + recurrent); dc: in = gradient wrt c_t from step t+1,
// out = gradient wrt c_{t-1}.  dgates are the gradients wrt the PRE-activations, as bf16 (the
// operand dtype of the dgrad / wgrad GEMMs that consume them).
template <typename TG>
__global__ void __launch_bounds__(256) lstm_cell_bwd_kernel(const TG* __restrict__ gates_act,
                                                            const float* __restrict__ c_prev, const float* __restrict__ c,
                                                            const float* __restrict__ dh, float* __restrict__ dc,
                                                            __nv_bfloat16* __restrict__ dgates, int n,
                                                            const float* __restrict__ dh2) {
  const int id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= n * 256) return;
  const int e = id >> 8, u = id & 255;
  const TG* gr = gates_act + (size_t)e * 1024;
  const float i = Gate<TG>::ld(gr + u), j = Gate<TG>::ld(gr + 256 + u), f = Gate<TG>::ld(gr + 512 + u), o = Gate<TG>::ld(gr + 768 + u);
  const float tc = tanhf(c[id]);
  const float dhv = dh[id] + (dh2 ? dh2[id] : 0.f);     // heads' gradient (+ the recurrent one from step t+1)
  const float d_o = dhv * tc;
  const float dcv = dc[id] + dhv * o * (1.0f - tc * tc);
  __nv_bfloat16* dg = dgates + (size_t)e * 1024;
  dg[u] = __float2bfloat16_rn(dcv * j * i * (1.0f - i));
  dg[256 + u] = __float2bfloat16_rn(dcv * i * (1.0f - j * j));
  dg[512 + u] = __float2bfloat16_rn(dcv * c_prev[id] * f * (1.0f - f));
  dg[768 + u] = __float2bfloat16_rn(d_o * o * (1.0f - o));
  dc[id] = dcv * f;
}


// ---- ReLU backward + bias gradient, fused ---------------------------------------------------------
// out = dy * (y > 0) as bf16 (the operand of the dgrad / wgrad GEMMs) and db[c] += sum over rows of
// out[:, c] in one pass; y == nullptr: no mask (plain bf16 copy / column sum).  Replaces the
// compare / multiply / cast / float / sum chain of element-wise launches.
// One thread per 8-column group of a row, threads laid over (row, group) in memory order; the grid
// size is a multiple of the groups per row, so a thread keeps its column group while striding rows
// and sums it in registers; block partials go through shared-memory atomics, one global atomic per
// column per block.
template <typename TD>
__global__ void __launch_bounds__(256) relu_grad_kernel(const TD* __restrict__ dy, const __nv_bfloat16* __restrict__ y,
                                                        __nv_bfloat16* __restrict__ out, float* __restrict__ db,
                                                        int64_t rows, int cols, int planes) {
  extern __shared__ float s_db[];
  const int groups = cols >> 3;
  if (db != nullptr) {
    for (int c = threadIdx.x; c < cols; c += blockDim.x) s_db[c] = 0.f;
    __syncthreads();
  }
  const int64_t total = rows * groups;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;          // multiple of `groups`
  const int64_t id0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int c0 = (int)(id0 % groups) * 8;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  for (int64_t id = id0; id < total; id += stride) {
    const int64_t off = id * 8;
    float v[8];
    if (sizeof(TD) == 2) {
      const uint4 u = __ldcs(reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(dy) + off));
      const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
      for (int j = 0; j < 4; ++j) { const float2 f = __bfloat1622float2(h[j]); v[2 * j] = f.x; v[2 * j + 1] = f.y; }
    } else {
      const float4 a = __ldcs(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(dy) + off));
      const float4 b = __ldcs(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(dy) + off + 4));
      v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    }
    if (y != nullptr) {
      const uint4 u = *reinterpret_cast<const uint4*>(y + off);
      const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = __bfloat1622float2(h[j]);
        if (!(f.x > 0.f)) v[2 * j] = 0.f;
        if (!(f.y > 0.f)) v[2 * j + 1] = 0.f;
      }
    }
    uint32_t pk[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      __nv_bfloat162 p = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
      pk[j] = *reinterpret_cast<uint32_t*>(&p);
      const float2 f = __bfloat1622float2(p);          // the bias gradient sums the ROUNDED values,
      acc[2 * j] += f.x; acc[2 * j + 1] += f.y;        // like dy16.float().sum(0)
    }
    if (out != nullptr) {
      // planes: out[cols/8][rows][8] (8-column chunks as separate planes, the tensor-core wgrad layout)
      const int64_t o = planes ? ((int64_t)(c0 >> 3) * rows + id / groups) * 8 : off;
      *reinterpret_cast<uint4*>(out + o) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
  }
  if (db == nullptr) return;
#pragma unroll
  for (int j = 0; j < 8; ++j) atomicAdd(&s_db[c0 + j], acc[j]);
  __syncthreads();
  for (int c = threadIdx.x; c < cols; c += blockDim.x) atomicAdd(db + c, s_db[c]);
}


// ---- pixel-control head: dueling combine + Q(a) gather + L2 loss, fused (model.py:431-441, :531-546) ----
// y [rows, 8] f32: the merged deconv output after ReLU, channel 0 = V, channels 1..A = advantages
// (channels A+1..7 are padding).  q = V + Adv - mean_a Adv;  loss = lam * 0.5 * sum mask * (R - q[act])^2.
// With dy != nullptr the same pass writes d loss / d (pre-ReLU deconv output), scaled by *go:
//   g = go * lam * mask * (q[act] - R);  dV = g;  dAdv_k = g * ([k == act] - 1/A);  masked by y > 0.
__global__ void __launch_bounds__(256) pc_loss_kernel(const float* __restrict__ y, const int32_t* __restrict__ act,
                                                      const float* __restrict__ target, const float* __restrict__ mask,
                                                      int A, float lam, int64_t rows, int px_per_sample,
                                                      double* __restrict__ loss, float* __restrict__ dy,
                                                      const float* __restrict__ go, __nv_bfloat16* __restrict__ dy16,
                                                      float* __restrict__ db8) {
  float part = 0.f;
  float dbacc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  const float gscale = ((dy != nullptr || dy16 != nullptr) && go != nullptr) ? *go : 1.f;
  const float inv_a = 1.0f / (float)A;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x) {
    const int64_t smp = r / px_per_sample;
    const float m = mask[smp];
    const int a = act[smp];
    const float4 lo = __ldcs(reinterpret_cast<const float4*>(y + r * 8));
    const float4 hi = __ldcs(reinterpret_cast<const float4*>(y + r * 8 + 4));
    const float v[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
    float sum = 0.f, qa = 0.f;
#pragma unroll
    for (int k = 0; k < 7; ++k) {
      if (k < A) { sum += v[1 + k]; if (k == a) qa = v[1 + k]; }
    }
    qa = v[0] + qa - sum * inv_a;
    const float diff = qa - __ldcs(target + r);
    part += m * diff * diff;
    if (dy != nullptr || dy16 != nullptr) {
      const float g = gscale * lam * m * diff;
      float d[8];
      d[0] = v[0] > 0.f ? g : 0.f;
#pragma unroll
      for (int k = 0; k < 7; ++k) d[1 + k] = (k < A && v[1 + k] > 0.f) ? g * ((k == a ? 1.f : 0.f) - inv_a) : 0.f;
      if (dy != nullptr) {
        __stcs(reinterpret_cast<float4*>(dy + r * 8), make_float4(d[0], d[1], d[2], d[3]));
        __stcs(reinterpret_cast<float4*>(dy + r * 8 + 4), make_float4(d[4], d[5], d[6], d[7]));
      }
      if (dy16 != nullptr) {
        // the gradient as conv2-geometry input [rows, 16] bf16 (channels 8..15 zero): the deconv's backward runs on
        // the encoder's conv2 kernels; the bias gradient sums the ROUNDED values (as unreal_relu_grad does)
        uint32_t pk[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          __nv_bfloat162 p = __floats2bfloat162_rn(d[2 * j], d[2 * j + 1]);
          pk[j] = *reinterpret_cast<uint32_t*>(&p);
          const float2 f = __bfloat1622float2(p);
          dbacc[2 * j] += f.x; dbacc[2 * j + 1] += f.y;
        }
        uint4* o = reinterpret_cast<uint4*>(dy16 + r * 16);
        o[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        o[1] = make_uint4(0u, 0u, 0u, 0u);
      }
    }
  }
  if (dy16 != nullptr && db8 != nullptr) {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float x = dbacc[c];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
      if ((threadIdx.x & 31) == 0) atomicAdd(db8 + c, x);
    }
  }
  if (loss == nullptr) return;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
  __shared__ float s_part[8];
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = part;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += (double)s_part[w];
    atomicAdd(loss, 0.5 * (double)lam * t);
  }
}

// ---- policy / value heads + A3C losses, fused (model.py:358-377 heads; :499-527 base loss; :556-565 VR loss) ----
// h [M,256] f32 (LSTM output), Wp [256,A], bp [A], Wv [256], bv [1] (TF [in,out] layouts).  One warp per row; the
// warp keeps its 8 x (A+1) weight slice in registers and walks rows persistently.
//   logits = h Wp + bp;  pi = softmax(logits);  v = h Wv + bv
//   policy = -sum mask * (log pi[a] * adv + beta * H),  H = -sum_k pi_k log pi_k   (pi clamped to [1e-20, 1] like :499-514)
//   value  = coef * sum mask * (R - v)^2        (coef 0.25 base :527, 0.5 value replay :565)
// The same pass writes d policy / d logits (dz) and d value / d v (dv) for the backward kernel:
//   dz_j = mask * (-adv * ([j == a] - pi_j) + beta * pi_j * (log pi_j + H)),   dv = -2 coef mask (R - v).
// The loss and backward kernels are built for up to MAXA = 7 actions (8 outputs, four lanes each) and 15 (16 outputs, two
// lanes each); a launch takes the narrowest build that holds A.
constexpr int kHeadMaxA = 7;
constexpr int kHeadMaxAWide = 15;

template <int MAXA>
struct HeadW {
  float wp[8][MAXA];
  float wv[8];
};

// [Wp | Wv] of the heads, transposed into shared memory once per CTA (s_w[j][k]; row kHeadMaxA = Wv), then each lane's
// eight rows k = lane + 32 i into registers.  (Every warp used to fetch its 64 weights with scalar global loads of
// stride A: at acting batch sizes -- one or two rows of work per warp -- that set-up WAS the kernel, 21 us for an
// 8 MB read.)  Block size 256.
template <int MAXA>
__device__ __forceinline__ void head_load_w(HeadW<MAXA>& w, const float* __restrict__ Wp, const float* __restrict__ Wv, int A,
                                            int lane, float* s_w) {
  for (int i = threadIdx.x; i < 256 * A; i += blockDim.x) {
    const int k = i / A, j = i - k * A;
    s_w[j * 256 + k] = Wp[i];
  }
  for (int k = threadIdx.x; k < 256; k += blockDim.x) s_w[MAXA * 256 + k] = Wv ? Wv[k] : 0.f;
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int k = lane + 32 * i;
#pragma unroll
    for (int j = 0; j < MAXA; ++j) w.wp[i][j] = (j < A) ? s_w[j * 256 + k] : 0.f;
    w.wv[i] = s_w[MAXA * 256 + k];
  }
}

__device__ __forceinline__ float warp_sum(float x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}

// One row of the heads on one warp.  x[i] = h[r, lane + 32 i].  The MAXA + 1 dot products (policy logits + the value) are
// reduced with a TRANSPOSING butterfly.  MAXA = 7: at distance 16 a lane keeps four of its eight partial sums and trades
// the other four, at distance 8 two of four, at distance 4 one of two, then two plain steps -- 9 shuffles instead of 40,
// and lane L ends up holding output j = L >> 2.  MAXA = 15: 16 partial sums halve at distances 16, 8, 4 and 2, then one
// plain step, and lane L holds output j = L >> 1.  Softmax, entropy and log-likelihood then run ACROSS the lanes (one
// shuffle per remaining distance), each output's exp / log computed once.
template <int MAXA> struct HeadLanes {
  static constexpr int kOut = MAXA + 1;                 // outputs per warp
  static constexpr int kPer = 32 / kOut;                // lanes per output (4 or 2)
  static constexpr int kShift = kPer == 4 ? 2 : 1;
  static_assert(kOut * kPer == 32 && (kPer == 4 || kPer == 2), "head builds: 8 or 16 outputs per warp");
};
struct HeadRow {
  float p, lp, H, v, z;      // this lane's (j = lane / lanes per output) probability and clamped log; entropy and value in every lane
};
template <int MAXA>
__device__ __forceinline__ HeadRow head_row(const HeadW<MAXA>& w, const float (&x)[8], int lane, int A, float bias_j) {
  using L = HeadLanes<MAXA>;
  float z[L::kOut];
#pragma unroll
  for (int j = 0; j < L::kOut; ++j) z[j] = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
#pragma unroll
    for (int j = 0; j < MAXA; ++j) z[j] = fmaf(x[i], w.wp[i][j], z[j]);
    z[MAXA] = fmaf(x[i], w.wv[i], z[MAXA]);
  }
#pragma unroll
  for (int n = L::kOut / 2, d = 16; d >= L::kPer; n >>= 1, d >>= 1) {
    const bool hi = lane & d;
#pragma unroll
    for (int t = 0; t < n; ++t) z[t] = (hi ? z[n + t] : z[t]) + __shfl_xor_sync(0xffffffffu, hi ? z[t] : z[n + t], d);
  }
  float s = z[0];
#pragma unroll
  for (int d = L::kPer / 2; d >= 1; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
  const int j = lane >> L::kShift;
  HeadRow o;
  o.z = s + bias_j;
  o.v = __shfl_sync(0xffffffffu, o.z, L::kPer * MAXA);
  float mx = (j < A) ? o.z : -3.0e38f;
#pragma unroll
  for (int d = L::kPer; d <= 16; d <<= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, d));
  const float e = (j < A) ? __expf(o.z - mx) : 0.f;
  float den = e;
#pragma unroll
  for (int d = L::kPer; d <= 16; d <<= 1) den += __shfl_xor_sync(0xffffffffu, den, d);
  o.p = e * (1.0f / den);
  o.lp = __logf(fminf(fmaxf(o.p, 1e-20f), 1.0f));
  float H = (j < A) ? -o.p * o.lp : 0.f;
#pragma unroll
  for (int d = L::kPer; d <= 16; d <<= 1) H += __shfl_xor_sync(0xffffffffu, H, d);
  o.H = H;
  return o;
}

// Acting step of the cell WITH the policy / value heads (model.py:343-377 for one step): 32 lanes x 8 units are one env's
// row of h, so the warp that has just computed the row reduces its five-to-eight dot products with [Wp | Wv] itself and lane 0
// finishes the softmax -- h never goes back to HBM for a separate head kernel (8.7 us per acting step at 8192 envs).
// Inactive envs keep c / h and report the heads of the h they hold.
__global__ void __launch_bounds__(256) lstm_cell_act_heads8_kernel(const __nv_bfloat16* __restrict__ gates, float* __restrict__ c_state,
                                                                   float* __restrict__ h_state, const uint8_t* __restrict__ active,
                                                                   int n, const float* __restrict__ Wp, const float* __restrict__ bp,
                                                                   const float* __restrict__ Wv, const float* __restrict__ bv, int A,
                                                                   float* __restrict__ pi_out, float* __restrict__ v_out) {
  // a lane owns units 8*lane .. 8*lane+7 of every row its warp processes: its 8 x (A+1) head weights are staged through shared
  // memory ONCE per CTA (s_w[j][k*32 + lane] = W_j[8*lane + k]: conflict-free reads).
  // (Reading them per row straight from global memory cost 32 L1 wavefronts per load -- the lanes' rows are 128 bytes apart --
  // and made the fused kernel 4x slower than the cell alone.)
  __shared__ float s_w[kHeadMaxA + 1][256];
  for (int i = threadIdx.x; i < (A + 1) * 256; i += blockDim.x) {
    const int j = i >> 8, uu = i & 255;
    s_w[j < A ? j : kHeadMaxA][(uu & 7) * 32 + (uu >> 3)] = (j < A) ? Wp[(size_t)uu * A + j] : Wv[uu];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, u = lane * 8;
  for (int e = blockIdx.x * 8 + warp; e < n; e += gridDim.x * 8) {     // a warp is one env's row
    const size_t so = (size_t)e * 256 + u;
    float h[8];
    if (active != nullptr && active[e] == 0) {
      *reinterpret_cast<float4*>(h) = reinterpret_cast<const float4*>(h_state + so)[0];
      *reinterpret_cast<float4*>(h + 4) = reinterpret_cast<const float4*>(h_state + so)[1];
    } else {
      float zi[8], zj[8], zf[8], zo[8], c[8];
      lstm_cell8(gates + (size_t)e * 1024 + u, c_state + so, zi, zj, zf, zo, c, h);
      st8(c_state + so, c);
      st8(h_state + so, h);
    }
    float z[kHeadMaxA + 1];
#pragma unroll
    for (int j = 0; j <= kHeadMaxA; ++j) z[j] = 0.f;
    // (the weights are read from shared memory per row, not kept in registers: 64 more registers halve the warps in
    // flight of what is otherwise a streaming kernel -- measured 20.9 us against 12.7 for the cell alone)
#pragma unroll
    for (int j = 0; j <= kHeadMaxA; ++j) {
      if (j < A || j == kHeadMaxA) {
#pragma unroll
        for (int k = 0; k < 8; ++k) z[j] = fmaf(h[k], s_w[j][k * 32 + lane], z[j]);
        z[j] = warp_sum(z[j]);
      }
    }
    if (lane == 0) {
      float mx = -3.0e38f;
#pragma unroll
      for (int j = 0; j < kHeadMaxA; ++j)
        if (j < A) { z[j] += bp[j]; mx = fmaxf(mx, z[j]); }
      float den = 0.f;
#pragma unroll
      for (int j = 0; j < kHeadMaxA; ++j)
        if (j < A) { z[j] = __expf(z[j] - mx); den += z[j]; }
      const float inv = 1.0f / den;
#pragma unroll
      for (int j = 0; j < kHeadMaxA; ++j)
        if (j < A) pi_out[(size_t)e * A + j] = z[j] * inv;
      v_out[e] = z[kHeadMaxA] + (bv ? bv[0] : 0.f);
    }
  }
}

template <int MAXA>
__global__ void __launch_bounds__(256) a3c_head_loss_kernel(const float* __restrict__ h, const float* __restrict__ Wp,
                                                            const float* __restrict__ bp, const float* __restrict__ Wv,
                                                            const float* __restrict__ bv, const int32_t* __restrict__ act,
                                                            const float* __restrict__ adv, const float* __restrict__ R,
                                                            const float* __restrict__ mask, int64_t M, int A, float beta,
                                                            float coef, float* __restrict__ pi_out, float* __restrict__ v_out,
                                                            double* __restrict__ sums, float* __restrict__ dz,
                                                            float* __restrict__ dv) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  using L = HeadLanes<MAXA>;
  constexpr int kVLane = L::kPer * MAXA;               // the lane that holds the value
  __shared__ float s_w[(MAXA + 1) * 256];
  HeadW<MAXA> w;
  head_load_w(w, Wp, Wv, A, lane, s_w);
  const int j = lane >> L::kShift;
  const bool writer = (lane & (L::kPer - 1)) == 0;     // one lane per output
  const float bias_j = (j < A) ? bp[j] : ((j == MAXA && bv) ? bv[0] : 0.f);
  float s_pol = 0.f, s_val = 0.f, s_ent = 0.f;         // lane 0 (policy, entropy) and lane kVLane (value) accumulate
  // two rows per iteration: both rows' loads are in flight before either row's arithmetic starts
  for (int64_t r0 = 2 * warp0; r0 < M; r0 += 2 * nwarps) {
    const int nrow = (r0 + 1 < M) ? 2 : 1;
    float x[2][8];
#pragma unroll
    for (int q = 0; q < 2; ++q)
#pragma unroll
      for (int i = 0; i < 8; ++i) x[q][i] = (q < nrow) ? h[(r0 + q) * 256 + lane + 32 * i] : 0.f;
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      if (q >= nrow) break;
      const int64_t r = r0 + q;
      const HeadRow o = head_row<MAXA>(w, x[q], lane, A, bias_j);
      const float m = mask ? mask[r] : 1.f;
      if (writer && j < A && pi_out) pi_out[r * A + j] = o.p;
      if (lane == kVLane && v_out) v_out[r] = o.v;
      if (act != nullptr) {
        const int a = act[r];
        const float ad = adv[r];
        const float lpa_any = __shfl_sync(0xffffffffu, o.lp, (L::kPer * a) & 31);
        const float lpa = (a >= 0 && a < A) ? lpa_any : 0.f;
        if (lane == 0) { s_pol -= m * (lpa * ad + beta * o.H); s_ent += m * o.H; }
        if (writer && j < A && dz) dz[r * A + j] = m * (-ad * ((j == a ? 1.f : 0.f) - o.p) + beta * o.p * (o.lp + o.H));
      }
      if (R != nullptr && lane == kVLane) {
        const float d = R[r] - o.v;
        s_val += coef * m * d * d;
        if (dv) dv[r] = -2.f * coef * m * d;
      }
    }
  }
  if (sums == nullptr) return;
  __shared__ float sp[8][3];
  if (lane == 0) { sp[threadIdx.x >> 5][0] = s_pol; sp[threadIdx.x >> 5][2] = s_ent; }
  if (lane == kVLane) sp[threadIdx.x >> 5][1] = s_val;
  __syncthreads();
  if (threadIdx.x < 3) {
    double t = 0.0;
    for (int q = 0; q < (int)(blockDim.x >> 5); ++q) t += (double)sp[q][threadIdx.x];
    atomicAdd(sums + threadIdx.x, t);
  }
}

// dh = go_p * dz Wp^T + go_v * dv Wv^T;  dWp += go_p * h^T dz;  dbp += go_p * sum dz;  dWv += go_v * h^T dv;  dbv += ...
// One thread per COLUMN k of h (256 per CTA), CTAs stride over chunks of 32 rows whose upstream gradients
// g[row][0..A) = go_p dz, g[row][MAXA] = go_v dv are staged in shared memory: per row a thread reads h[r,k], writes dh[r,k]
// (both coalesced) and does 16 FMAs against 8 broadcast values (32 against 16 in the 15-action build) -- ~40 registers, so the SM holds 32+ warps and the
// row-to-row load latency is hidden by other warps.  (The first form -- one warp per row, 64 weight + 64 accumulator
// registers per lane, 16 warps per SM, each row's loads waited for in turn -- ran at 244 us for 163 840 rows: 1.4 TB/s.)
constexpr int kHeadBwdRows = 32;
template <int MAXA>
__global__ void __launch_bounds__(256) a3c_head_bwd_kernel(const float* __restrict__ h, const float* __restrict__ Wp,
                                                           const float* __restrict__ Wv, const float* __restrict__ dz,
                                                           const float* __restrict__ dv, const float* __restrict__ go,
                                                           int64_t M, int A, float* __restrict__ dh, float* __restrict__ dWp,
                                                           float* __restrict__ dbp, float* __restrict__ dWv,
                                                           float* __restrict__ dbv) {
  constexpr int kOut = MAXA + 1;
  constexpr int kStageRows = 256 / kOut;               // chunk rows one pass of the 256 threads stages
  __shared__ __align__(16) float s_g[2][kHeadBwdRows][kOut];
  __shared__ float s_b[kOut];
  const int k = threadIdx.x;
  const float gp = dz ? go[0] : 0.f, gv = dv ? go[1] : 0.f;
  float w[kOut], acc[kOut];
#pragma unroll
  for (int j = 0; j < MAXA; ++j) { w[j] = (dz && j < A) ? Wp[k * A + j] : 0.f; acc[j] = 0.f; }
  w[MAXA] = (dv && Wv) ? Wv[k] : 0.f;
  acc[MAXA] = 0.f;
  if (k <= MAXA) s_b[k] = 0.f;
  // staging role of this thread: rows k / kOut (+ kStageRows) of a chunk, component k % kOut
  const int srow = k / kOut, sj = k % kOut;
  float bsum = 0.f;
  const int64_t chunks = (M + kHeadBwdRows - 1) / kHeadBwdRows;
  int buf = 0;
  for (int64_t c = blockIdx.x; c < chunks; c += gridDim.x, buf ^= 1) {
    const int64_t r0 = c * kHeadBwdRows;
#pragma unroll
    for (int p = 0; p < kHeadBwdRows / kStageRows; ++p) {
      const int64_t r = r0 + srow + p * kStageRows;
      float g = 0.f;
      if (r < M) {
        if (sj < MAXA) { if (dz && sj < A) g = gp * dz[r * A + sj]; }
        else if (dv) g = gv * dv[r];
      }
      s_g[buf][srow + p * kStageRows][sj] = g;
      bsum += g;
    }
    __syncthreads();            // one barrier per chunk: the other buffer is rewritten only after the next one
    const int rows = (int)((M - r0) < kHeadBwdRows ? (M - r0) : kHeadBwdRows);
    const float* hp = h + r0 * 256 + k;
    float* dp = dh + r0 * 256 + k;
#pragma unroll 8
    for (int i = 0; i < rows; ++i) {
      const float x = hp[(int64_t)i * 256];
      float g[kOut];
#pragma unroll
      for (int q = 0; q < kOut / 4; ++q) {
        const float4 g4 = *reinterpret_cast<const float4*>(&s_g[buf][i][4 * q]);
        g[4 * q] = g4.x; g[4 * q + 1] = g4.y; g[4 * q + 2] = g4.z; g[4 * q + 3] = g4.w;
      }
      float d = 0.f;
#pragma unroll
      for (int j = 0; j < kOut; ++j) { d = fmaf(g[j], w[j], d); acc[j] = fmaf(x, g[j], acc[j]); }
      dp[(int64_t)i * 256] = d;
    }
  }
  atomicAdd(&s_b[sj], bsum);
  __syncthreads();
#pragma unroll
  for (int j = 0; j < MAXA; ++j) if (j < A && dWp) atomicAdd(dWp + k * A + j, acc[j]);
  if (dWv) atomicAdd(dWv + k, acc[MAXA]);
  if (k < A && dbp) atomicAdd(dbp + k, s_b[k]);
  if (k == MAXA && dbv) atomicAdd(dbv, s_b[MAXA]);
}

// col2im for f32 columns with C a multiple of 4 (the merged, padded deconv: C = 8): float4 per tap
__global__ void __launch_bounds__(256) col2im_f32v4_kernel(const float* __restrict__ cols, float* __restrict__ out,
                                                           const float* __restrict__ bias, int relu, ConvGeom g,
                                                           int64_t total4) {
  const int k = g.kh * g.kw * g.c;
  const int c4n = g.c >> 2;
  for (int64_t id = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; id < total4; id += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = id;
    const int c = (int)(r % c4n) * 4; r /= c4n;
    const int x = (int)(r % g.w); r /= g.w;
    const int y = (int)(r % g.h); r /= g.h;
    const int64_t s = r;
    float4 acc = bias ? make_float4(bias[c], bias[c + 1], bias[c + 2], bias[c + 3]) : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int ky = y % g.stride; ky < g.kh; ky += g.stride) {
      const int oy = (y - ky) / g.stride;
      if (y - ky < 0 || oy >= g.oh) continue;
      for (int kx = x % g.stride; kx < g.kw; kx += g.stride) {
        const int ox = (x - kx) / g.stride;
        if (x - kx < 0 || ox >= g.ow) continue;
        const float4 t = __ldcs(reinterpret_cast<const float4*>(cols + ((s * g.oh + oy) * g.ow + ox) * (int64_t)k +
                                                                (ky * g.kw + kx) * g.c + c));
        acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
      }
    }
    if (relu) { acc.x = fmaxf(acc.x, 0.f); acc.y = fmaxf(acc.y, 0.f); acc.z = fmaxf(acc.z, 0.f); acc.w = fmaxf(acc.w, 0.f); }
    reinterpret_cast<float4*>(out)[id] = acc;
  }
}

static int grid_for_elems(int64_t total, int per_block = 256) {
  int sms = sm_count();
  if (sms <= 0) return 0;
  int64_t want = (total + per_block - 1) / per_block;
  int64_t cap = (int64_t)sms * 16;
  if (want < 1) want = 1;
  return (int)(want < cap ? want : cap);
}

static int check_geom(const char* fn, ConvGeom& g) {
  UNREAL_REQUIRE(g.s > 0 && g.h > 0 && g.w > 0 && g.c > 0 && g.kh > 0 && g.kw > 0 && g.stride > 0,
                 "%s: non-positive geometry", fn);
  UNREAL_REQUIRE(g.h >= g.kh && g.w >= g.kw, "%s: kernel larger than the image", fn);
  UNREAL_REQUIRE((g.h - g.kh) % g.stride == 0 && (g.w - g.kw) % g.stride == 0,
                 "%s: VALID windows must tile the image exactly (H-KH and W-KW multiples of the stride)", fn);
  g.oh = (g.h - g.kh) / g.stride + 1;
  g.ow = (g.w - g.kw) / g.stride + 1;
  return UNREAL_OK;
}

// Reward-prediction head after the fc GEMM (model.py:482-488, :571-575): logits8 [N,8] f32 hold h2 . W_rp in columns
// 0..2 (the bf16 tcgen05 GEMM on the weight shadow padded to 8 columns; no bias yet).  One thread per sample:
//   z = logits + b;  p = softmax(z);  loss += -sum_k c_k log(clip(p_k, 1e-20, 1));
//   dz_j = go * sum_k c_k [p_k >= 1e-20] (p_j - delta_kj)      -> dz16 bf16 [N,8] (columns 3..7 zero), db [3] += sum_n dz
__global__ void __launch_bounds__(256) rp_loss_kernel(const float* __restrict__ logits8, const float* __restrict__ bias,
                                                      const float* __restrict__ c, int64_t n, float* __restrict__ p_out,
                                                      double* __restrict__ loss, __nv_bfloat16* __restrict__ dz16,
                                                      float* __restrict__ db, const float* __restrict__ go) {
  const float b0 = bias[0], b1 = bias[1], b2 = bias[2];
  const float g = go ? *go : 1.f;
  double lsum = 0.0;
  float d0 = 0.f, d1 = 0.f, d2 = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 l = *reinterpret_cast<const float4*>(logits8 + i * 8);
    const float z0 = l.x + b0, z1 = l.y + b1, z2 = l.z + b2;
    const float m = fmaxf(z0, fmaxf(z1, z2));
    const float e0 = expf(z0 - m), e1 = expf(z1 - m), e2 = expf(z2 - m);
    const float inv = 1.f / (e0 + e1 + e2);
    const float p0 = e0 * inv, p1 = e1 * inv, p2 = e2 * inv;
    if (p_out) { p_out[i * 3] = p0; p_out[i * 3 + 1] = p1; p_out[i * 3 + 2] = p2; }
    if (c == nullptr) continue;
    const float c0 = c[i * 3], c1 = c[i * 3 + 1], c2 = c[i * 3 + 2];
    if (loss) {
      lsum -= (double)(c0 * logf(fminf(fmaxf(p0, 1e-20f), 1.f)) + c1 * logf(fminf(fmaxf(p1, 1e-20f), 1.f)) +
                       c2 * logf(fminf(fmaxf(p2, 1e-20f), 1.f)));
    }
    if (dz16) {
      const float k0 = p0 >= 1e-20f ? c0 : 0.f, k1 = p1 >= 1e-20f ? c1 : 0.f, k2 = p2 >= 1e-20f ? c2 : 0.f;
      const float ks = k0 + k1 + k2;
      const float g0 = g * (ks * p0 - k0), g1 = g * (ks * p1 - k1), g2 = g * (ks * p2 - k2);
      __align__(16) __nv_bfloat16 o[8];
      o[0] = __float2bfloat16(g0); o[1] = __float2bfloat16(g1); o[2] = __float2bfloat16(g2);
#pragma unroll
      for (int q = 3; q < 8; ++q) o[q] = __float2bfloat16(0.f);
      *reinterpret_cast<uint4*>(dz16 + i * 8) = *reinterpret_cast<const uint4*>(o);
      d0 += g0; d1 += g1; d2 += g2;
    }
  }
  // block reduction: loss (double) and the three bias-gradient sums
  __shared__ double s_l[8];
  __shared__ float s_d[8][3];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lsum += __shfl_down_sync(0xffffffffu, lsum, o);
    d0 += __shfl_down_sync(0xffffffffu, d0, o);
    d1 += __shfl_down_sync(0xffffffffu, d1, o);
    d2 += __shfl_down_sync(0xffffffffu, d2, o);
  }
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) { s_l[w] = lsum; s_d[w][0] = d0; s_d[w][1] = d1; s_d[w][2] = d2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double L = 0.0; float a0 = 0.f, a1 = 0.f, a2 = 0.f;
    for (int q = 0; q < (int)(blockDim.x >> 5); ++q) { L += s_l[q]; a0 += s_d[q][0]; a1 += s_d[q][1]; a2 += s_d[q][2]; }
    if (loss && c) atomicAdd(loss, L);
    if (db && dz16) { atomicAdd(db, a0); atomicAdd(db + 1, a1); atomicAdd(db + 2, a2); }
  }
}

// ---- maze-cell de-duplication of the encoder (UnrealModel.dedup_cells) -------------------------------------------------
// A maze frame is a pure function of the agent cell, so conv1 -> conv2 -> fc1 (model.py:281-289, :332-340) of ALL samples
// of an update is a lookup in a 49-row table evaluated once, and its backward pass is a segment sum of the per-sample
// gradient by cell followed by a 49-sample encoder backward.  Same values as the dense path up to summation order.
//
// gather: out[s, :] = table[cell(s), :]   (bf16, D columns; out rows ld_out elements apart: e.g. the LSTM step operand)
__global__ void __launch_bounds__(256) cell_gather_kernel(const __nv_bfloat16* __restrict__ table, const int32_t* __restrict__ pos,
                                                          __nv_bfloat16* __restrict__ out, int64_t ld_out, int64_t s, int d8) {
  const int64_t total = s * d8;     // one thread per 16-byte chunk
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / d8;
    const int c = (int)(i - r * d8);
    int x = pos[2 * r], y = pos[2 * r + 1];
    x = x < 0 ? 0 : (x > 6 ? 6 : x); y = y < 0 ? 0 : (y > 6 ? 6 : y);
    const uint4 v = reinterpret_cast<const uint4*>(table + (size_t)(y * 7 + x) * d8 * 8)[c];
    reinterpret_cast<uint4*>(out + r * ld_out)[c] = v;
  }
}

// segment sum: out[cell, :] += sum over the samples s with cell(s) == cell of dy[s, :]   (D = 256; out [49,256] f32).
// One thread per column: a thread owns column j of all 49 bins in shared memory, so rows are accumulated without atomics;
// the CTA's bins go to global memory with one atomicAdd per non-zero bin element at the end.
template <typename TD>
__global__ void __launch_bounds__(256) cell_segment_sum_kernel(const TD* __restrict__ dy, const int32_t* __restrict__ pos,
                                                               float* __restrict__ out, int64_t s, int64_t rows_per_cta) {
  extern __shared__ float s_bins[];      // [49][256]
  const int j = threadIdx.x;
  for (int b = 0; b < 49; ++b) s_bins[b * 256 + j] = 0.f;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_cta;
  const int64_t r1 = r0 + rows_per_cta < s ? r0 + rows_per_cta : s;
  int64_t r = r0;
  for (; r + 4 <= r1; r += 4) {
    float v[4]; int c[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      v[u] = In<TD>::ld(dy + (r + u) * 256 + j);
      int x = pos[2 * (r + u)], y = pos[2 * (r + u) + 1];
      x = x < 0 ? 0 : (x > 6 ? 6 : x); y = y < 0 ? 0 : (y > 6 ? 6 : y);
      c[u] = y * 7 + x;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) s_bins[c[u] * 256 + j] += v[u];
  }
  for (; r < r1; ++r) {
    int x = pos[2 * r], y = pos[2 * r + 1];
    x = x < 0 ? 0 : (x > 6 ? 6 : x); y = y < 0 ? 0 : (y > 6 ? 6 : y);
    s_bins[(y * 7 + x) * 256 + j] += In<TD>::ld(dy + r * 256 + j);
  }
  for (int b = 0; b < 49; ++b) {
    const float v = s_bins[b * 256 + j];
    if (v != 0.f) atomicAdd(out + b * 256 + j, v);
  }
}

}  // namespace unreal

using namespace unreal;

extern "C" int unreal_im2col(const void* in, int in_dtype, void* out_bf16, int s, int h, int w, int c, int kh, int kw,
                             int stride, void* stream) {
  UNREAL_REQUIRE(in && out_bf16, "unreal_im2col: null buffer");
  ConvGeom g{s, h, w, c, kh, kw, stride, 0, 0};
  int rc = check_geom("unreal_im2col", g);
  if (rc != UNREAL_OK) return rc;
  const int seg = kw * c;
  const int esz = in_dtype == UNREAL_F32 ? 4 : (in_dtype == UNREAL_U8 ? 1 : 2);
  UNREAL_REQUIRE(in_dtype == UNREAL_F32 || in_dtype == UNREAL_U8 || in_dtype == UNREAL_BF16, "unreal_im2col: bad dtype");
  // the 8-wide path needs every chunk 16-byte aligned on both sides (f32: 32 B reads)
  const bool v8 = (seg % 8 == 0) && ((stride * c * esz) % 16 == 0) && ((w * c * esz) % 16 == 0) && aligned16(in) &&
                  aligned16(out_bf16) && in_dtype != UNREAL_U8;
  const int64_t rows = (int64_t)s * g.oh * g.ow;
  const int64_t chunks = rows * kh * (v8 ? seg / 8 : seg);
  const int grid = grid_for_elems(chunks);
  if (grid <= 0) return UNREAL_ECUDA;
  cudaStream_t st = as_stream(stream);
  __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out_bf16);
  if (in_dtype == UNREAL_F32) {
    if (v8) im2col_kernel<float, 8><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(in), o, g, chunks);
    else im2col_kernel<float, 1><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(in), o, g, chunks);
  } else if (in_dtype == UNREAL_U8) {
    im2col_kernel<uint8_t, 1><<<grid, 256, 0, st>>>(reinterpret_cast<const uint8_t*>(in), o, g, chunks);
  } else {
    if (v8) im2col_kernel<__nv_bfloat16, 8><<<grid, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(in), o, g, chunks);
    else im2col_kernel<__nv_bfloat16, 1><<<grid, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(in), o, g, chunks);
  }
  UNREAL_LAUNCH_CHECK("im2col_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_col2im(const void* cols, int cols_dtype, void* out, int out_dtype, const float* bias, int relu,
                             int s, int h, int w, int c, int kh, int kw, int stride, void* stream) {
  UNREAL_REQUIRE(cols && out, "unreal_col2im: null buffer");
  UNREAL_REQUIRE((cols_dtype == UNREAL_F32 || cols_dtype == UNREAL_BF16) && (out_dtype == UNREAL_F32 || out_dtype == UNREAL_BF16),
                 "unreal_col2im: dtypes must be f32 or bf16");
  ConvGeom g{s, h, w, c, kh, kw, stride, 0, 0};
  int rc = check_geom("unreal_col2im", g);
  if (rc != UNREAL_OK) return rc;
  const int64_t total = (int64_t)s * h * w * c;
  const int grid = grid_for_elems(total);
  if (grid <= 0) return UNREAL_ECUDA;
  cudaStream_t st = as_stream(stream);
  if (cols_dtype == UNREAL_BF16 && (c & 7) == 0 && aligned16(cols) && aligned16(out)) {
    const int64_t total8 = total / 8;
    const int grid8 = grid_for_elems(total8);
    if (out_dtype == UNREAL_BF16)
      col2im_vec8_kernel<__nv_bfloat16><<<grid8, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(cols), reinterpret_cast<__nv_bfloat16*>(out), bias, relu, g, total8);
    else
      col2im_vec8_kernel<float><<<grid8, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(cols), reinterpret_cast<float*>(out), bias, relu, g, total8);
    UNREAL_LAUNCH_CHECK("col2im_vec8_kernel");
    return UNREAL_OK;
  }
  if (cols_dtype == UNREAL_F32 && out_dtype == UNREAL_F32 && (c & 3) == 0 && aligned16(cols) && aligned16(out)) {
    const int64_t total4 = total / 4;
    col2im_f32v4_kernel<<<grid_for_elems(total4), 256, 0, st>>>(reinterpret_cast<const float*>(cols), reinterpret_cast<float*>(out), bias, relu, g, total4);
    UNREAL_LAUNCH_CHECK("col2im_f32v4_kernel");
    return UNREAL_OK;
  }
  if (cols_dtype == UNREAL_F32 && out_dtype == UNREAL_F32)
    col2im_kernel<float, float><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(cols), reinterpret_cast<float*>(out), bias, relu, g, total);
  else if (cols_dtype == UNREAL_F32)
    col2im_kernel<float, __nv_bfloat16><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(cols), reinterpret_cast<__nv_bfloat16*>(out), bias, relu, g, total);
  else if (out_dtype == UNREAL_F32)
    col2im_kernel<__nv_bfloat16, float><<<grid, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(cols), reinterpret_cast<float*>(out), bias, relu, g, total);
  else
    col2im_kernel<__nv_bfloat16, __nv_bfloat16><<<grid, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(cols), reinterpret_cast<__nv_bfloat16*>(out), bias, relu, g, total);
  UNREAL_LAUNCH_CHECK("col2im_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_lstm_cell_fwd(float* gates, const float* c_prev, float* c_out, float* h_out, void* h16_out,
                                    int n, void* stream) {
  UNREAL_REQUIRE(gates && c_prev && c_out && h_out && h16_out && n > 0, "unreal_lstm_cell_fwd: null buffer or n <= 0");
  lstm_cell_fwd_kernel<float><<<(n * 256 + 255) / 256, 256, 0, as_stream(stream)>>>(
      gates, c_prev, c_out, h_out, reinterpret_cast<__nv_bfloat16*>(h16_out), n, 256);
  UNREAL_LAUNCH_CHECK("lstm_cell_fwd_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_lstm_cell_fwd_ld(float* gates, const float* c_prev, float* c_out, float* h_out, void* h16_out,
                                       int h16_ld, int n, void* stream) {
  UNREAL_REQUIRE(gates && c_prev && c_out && h_out && h16_out && n > 0, "unreal_lstm_cell_fwd_ld: null buffer or n <= 0");
  UNREAL_REQUIRE(h16_ld >= 256, "unreal_lstm_cell_fwd_ld: h16_ld %d < 256", h16_ld);
  lstm_cell_fwd_kernel<float><<<(n * 256 + 255) / 256, 256, 0, as_stream(stream)>>>(
      gates, c_prev, c_out, h_out, reinterpret_cast<__nv_bfloat16*>(h16_out), n, h16_ld);
  UNREAL_LAUNCH_CHECK("lstm_cell_fwd_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_lstm_cell_act(const float* gates, float* c_state, float* h_state, float* h_out, const uint8_t* active,
                                    int n, void* stream) {
  UNREAL_REQUIRE(gates && c_state && h_state && n > 0, "unreal_lstm_cell_act: null buffer or n <= 0");
  lstm_cell_act_kernel<float><<<(n * 256 + 255) / 256, 256, 0, as_stream(stream)>>>(gates, c_state, h_state, h_out, active, n);
  UNREAL_LAUNCH_CHECK("lstm_cell_act_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_lstm_cell_bwd(const float* gates_act, const float* c_prev, const float* c, const float* dh,
                                    float* dc, void* dgates_bf16, int n, void* stream) {
  UNREAL_REQUIRE(gates_act && c_prev && c && dh && dc && dgates_bf16 && n > 0,
                 "unreal_lstm_cell_bwd: null buffer or n <= 0");
  lstm_cell_bwd_kernel<float><<<(n * 256 + 255) / 256, 256, 0, as_stream(stream)>>>(
      gates_act, c_prev, c, dh, dc, reinterpret_cast<__nv_bfloat16*>(dgates_bf16), n, nullptr);
  UNREAL_LAUNCH_CHECK("lstm_cell_bwd_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_lstm_cell_bwd2(const float* gates_act, const float* c_prev, const float* c, const float* dh,
                                     const float* dh_rec, float* dc, void* dgates_bf16, int n, void* stream) {
  UNREAL_REQUIRE(gates_act && c_prev && c && dh && dc && dgates_bf16 && n > 0,
                 "unreal_lstm_cell_bwd2: null buffer or n <= 0");
  lstm_cell_bwd_kernel<float><<<(n * 256 + 255) / 256, 256, 0, as_stream(stream)>>>(
      gates_act, c_prev, c, dh, dc, reinterpret_cast<__nv_bfloat16*>(dgates_bf16), n, dh_rec);
  UNREAL_LAUNCH_CHECK("lstm_cell_bwd_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_relu_grad(const void* dy, int dy_dtype, const void* y_bf16, void* out_bf16, float* db,
                                int64_t rows, int cols, int out_planes, void* stream) {
  UNREAL_REQUIRE(dy != nullptr && rows > 0 && cols > 0, "unreal_relu_grad: null dy or empty shape");
  UNREAL_REQUIRE(dy_dtype == UNREAL_BF16 || dy_dtype == UNREAL_F32, "unreal_relu_grad: dy must be bf16 or f32");
  UNREAL_REQUIRE((cols & 7) == 0, "unreal_relu_grad: cols must be a multiple of 8");
  UNREAL_REQUIRE(aligned16(dy) && aligned16(y_bf16) && aligned16(out_bf16), "unreal_relu_grad: 16-byte alignment");
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  const int groups = cols / 8;
  UNREAL_REQUIRE(cols <= 8192, "unreal_relu_grad: cols must be <= 8192");
  // grid * 256 must be a multiple of `groups`: grid = k * groups / gcd(groups, 256)
  int g = groups, h = 256;
  while (h) { int t = g % h; g = h; h = t; }
  const int unit = groups / g;
  const int64_t total = rows * groups;
  int64_t want = (total + 255) / 256;
  const int64_t cap = (int64_t)sms * 8;
  if (want > cap) want = cap;
  int64_t gx = (want + unit - 1) / unit * unit;
  if (gx < unit) gx = unit;
  const size_t shm = (size_t)cols * sizeof(float);
  if (dy_dtype == UNREAL_BF16)
    relu_grad_kernel<__nv_bfloat16><<<(unsigned)gx, 256, shm, as_stream(stream)>>>(
        reinterpret_cast<const __nv_bfloat16*>(dy), reinterpret_cast<const __nv_bfloat16*>(y_bf16),
        reinterpret_cast<__nv_bfloat16*>(out_bf16), db, rows, cols, out_planes);
  else
    relu_grad_kernel<float><<<(unsigned)gx, 256, shm, as_stream(stream)>>>(
        reinterpret_cast<const float*>(dy), reinterpret_cast<const __nv_bfloat16*>(y_bf16),
        reinterpret_cast<__nv_bfloat16*>(out_bf16), db, rows, cols, out_planes);
  UNREAL_LAUNCH_CHECK("relu_grad_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_pc_loss(const float* y8, const int32_t* act, const float* target, const float* mask, int a,
                              float lam, int64_t samples, int px_per_sample, double* loss, float* dy8, const float* go,
                              void* stream) {
  UNREAL_REQUIRE(y8 && act && target && mask && samples > 0 && px_per_sample > 0, "unreal_pc_loss: null buffer or empty shape");
  UNREAL_REQUIRE(a >= 1 && a <= 7, "unreal_pc_loss: action count %d not in 1..7 (8-channel padded head)", a);
  UNREAL_REQUIRE(loss != nullptr || dy8 != nullptr, "unreal_pc_loss: nothing to compute");
  UNREAL_REQUIRE(aligned16(y8) && aligned16(dy8), "unreal_pc_loss: 16-byte alignment");
  const int64_t rows = samples * px_per_sample;
  const int grid = grid_for_elems(rows);
  if (grid <= 0) return UNREAL_ECUDA;
  pc_loss_kernel<<<grid, 256, 0, as_stream(stream)>>>(y8, act, target, mask, a, lam, rows, px_per_sample, loss, dy8, go,
                                                      nullptr, nullptr);
  UNREAL_LAUNCH_CHECK("pc_loss_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_pc_loss_grad16(const float* y8, const int32_t* act, const float* target, const float* mask, int a,
                                     float lam, int64_t samples, int px_per_sample, void* dy16_bf16, float* db8,
                                     const float* go, void* stream) {
  UNREAL_REQUIRE(y8 && act && target && mask && dy16_bf16 && samples > 0 && px_per_sample > 0,
                 "unreal_pc_loss_grad16: null buffer or empty shape");
  UNREAL_REQUIRE(a >= 1 && a <= 7, "unreal_pc_loss_grad16: action count %d not in 1..7 (8-channel padded head)", a);
  UNREAL_REQUIRE(aligned16(y8) && aligned16(dy16_bf16), "unreal_pc_loss_grad16: 16-byte alignment");
  const int64_t rows = samples * px_per_sample;
  const int grid = grid_for_elems(rows);
  if (grid <= 0) return UNREAL_ECUDA;
  pc_loss_kernel<<<grid, 256, 0, as_stream(stream)>>>(y8, act, target, mask, a, lam, rows, px_per_sample, nullptr, nullptr, go,
                                                      reinterpret_cast<__nv_bfloat16*>(dy16_bf16), db8);
  UNREAL_LAUNCH_CHECK("pc_loss_kernel(grad16)");
  return UNREAL_OK;
}

extern "C" int unreal_a3c_head_loss(const float* h, const float* wp, const float* bp, const float* wv, const float* bv,
                                    const int32_t* act, const float* adv, const float* r, const float* mask, int64_t m,
                                    int a, float entropy_beta, float value_coef, float* pi_out, float* v_out,
                                    double* sums, float* dz, float* dv, void* stream) {
  UNREAL_REQUIRE(h && m > 0, "unreal_a3c_head_loss: null h or m <= 0");
  UNREAL_REQUIRE(a >= 0 && a <= kHeadMaxAWide, "unreal_a3c_head_loss: action count %d not in 0..15", a);
  UNREAL_REQUIRE(a == 0 || (wp && bp), "unreal_a3c_head_loss: policy weights missing for action count %d", a);
  UNREAL_REQUIRE(act == nullptr || (adv != nullptr && a > 0), "unreal_a3c_head_loss: act needs adv and the policy head");
  UNREAL_REQUIRE(r == nullptr || wv != nullptr, "unreal_a3c_head_loss: returns need the value head");
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  int64_t want = (m + 15) / 16;       // a warp takes two rows per iteration
  const int grid = (int)(want < (int64_t)sms * 4 ? want : (int64_t)sms * 4);
  if (a <= kHeadMaxA)
    a3c_head_loss_kernel<kHeadMaxA><<<grid, 256, 0, as_stream(stream)>>>(h, wp, bp, wv, bv, act, adv, r, mask, m, a, entropy_beta,
                                                                         value_coef, pi_out, v_out, sums, dz, dv);
  else
    a3c_head_loss_kernel<kHeadMaxAWide><<<grid, 256, 0, as_stream(stream)>>>(h, wp, bp, wv, bv, act, adv, r, mask, m, a,
                                                                             entropy_beta, value_coef, pi_out, v_out, sums, dz, dv);
  UNREAL_LAUNCH_CHECK("a3c_head_loss_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_a3c_head_bwd(const float* h, const float* wp, const float* wv, const float* dz, const float* dv,
                                   const float* go2, int64_t m, int a, float* dh, float* dwp, float* dbp, float* dwv,
                                   float* dbv, void* stream) {
  UNREAL_REQUIRE(h && go2 && dh && m > 0, "unreal_a3c_head_bwd: null buffer or m <= 0");
  UNREAL_REQUIRE(a >= 0 && a <= kHeadMaxAWide, "unreal_a3c_head_bwd: action count %d not in 0..15", a);
  UNREAL_REQUIRE(dz == nullptr || (wp && a > 0), "unreal_a3c_head_bwd: dz needs the policy weights");
  UNREAL_REQUIRE(dv == nullptr || wv, "unreal_a3c_head_bwd: dv needs the value weights");
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  int64_t want = (m + kHeadBwdRows - 1) / kHeadBwdRows;
  const int grid = (int)(want < (int64_t)sms * 4 ? want : (int64_t)sms * 4);
  if (a <= kHeadMaxA)
    a3c_head_bwd_kernel<kHeadMaxA><<<grid, 256, 0, as_stream(stream)>>>(h, wp, wv, dz, dv, go2, m, a, dh, dwp, dbp, dwv, dbv);
  else
    a3c_head_bwd_kernel<kHeadMaxAWide><<<grid, 256, 0, as_stream(stream)>>>(h, wp, wv, dz, dv, go2, m, a, dh, dwp, dbp, dwv, dbv);
  UNREAL_LAUNCH_CHECK("a3c_head_bwd_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_rp_loss(const float* logits8, const float* bias, const float* c, int64_t n, float* p_out, double* loss,
                              void* dz16, float* db, const float* go, void* stream) {
  UNREAL_REQUIRE(logits8 && bias && n > 0, "unreal_rp_loss: null buffer or n <= 0");
  UNREAL_REQUIRE(aligned16(logits8) && aligned16(dz16), "unreal_rp_loss: logits8 / dz16 must be 16-byte aligned");
  UNREAL_REQUIRE(c != nullptr || (loss == nullptr && dz16 == nullptr), "unreal_rp_loss: loss / gradient need the targets");
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  int64_t want = (n + 255) / 256;
  const int grid = (int)(want < (int64_t)sms * 4 ? want : (int64_t)sms * 4);
  rp_loss_kernel<<<grid, 256, 0, as_stream(stream)>>>(logits8, bias, c, n, p_out, loss, reinterpret_cast<__nv_bfloat16*>(dz16),
                                                     db, go);
  UNREAL_LAUNCH_CHECK("rp_loss_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_cell_gather(const void* table_bf16, const int32_t* pos, void* out_bf16, int64_t ld_out, int64_t s, int d,
                                  void* stream) {
  UNREAL_REQUIRE(table_bf16 && pos && out_bf16 && s >= 0, "unreal_cell_gather: null buffer or s < 0");
  UNREAL_REQUIRE(d > 0 && d % 8 == 0 && ld_out >= d && ld_out % 8 == 0, "unreal_cell_gather: d and ld_out must be multiples of 8");
  UNREAL_REQUIRE(aligned16(table_bf16) && aligned16(out_bf16), "unreal_cell_gather: buffers must be 16-byte aligned");
  if (s == 0) return UNREAL_OK;
  const int64_t total = s * (d / 8);
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  int64_t want = (total + 255) / 256;
  const int grid = (int)(want < (int64_t)sms * 16 ? want : (int64_t)sms * 16);
  cell_gather_kernel<<<grid, 256, 0, as_stream(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(table_bf16), pos,
                                                         reinterpret_cast<__nv_bfloat16*>(out_bf16), ld_out, s, d / 8);
  UNREAL_LAUNCH_CHECK("cell_gather_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_cell_segment_sum(const void* dy, int dy_dtype, const int32_t* pos, float* out, int64_t s, int d,
                                       void* stream) {
  UNREAL_REQUIRE(dy && pos && out && s >= 0, "unreal_cell_segment_sum: null buffer or s < 0");
  UNREAL_REQUIRE(d == 256, "unreal_cell_segment_sum: rows of 256 columns (fc1's width), got %d", d);
  UNREAL_REQUIRE(dy_dtype == UNREAL_F32 || dy_dtype == UNREAL_BF16, "unreal_cell_segment_sum: dy must be f32 or bf16");
  if (s == 0) return UNREAL_OK;
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  constexpr int kSmem = 49 * 256 * 4;
  int rc = allow_dynamic_smem((const void*)cell_segment_sum_kernel<float>, kSmem);
  if (rc == UNREAL_OK) rc = allow_dynamic_smem((const void*)cell_segment_sum_kernel<__nv_bfloat16>, kSmem);
  if (rc != UNREAL_OK) return rc;
  int64_t ctas = (int64_t)sms * 4;
  if (ctas > (s + 63) / 64) ctas = (s + 63) / 64;
  const int64_t rows_per_cta = (s + ctas - 1) / ctas;
  ctas = (s + rows_per_cta - 1) / rows_per_cta;
  if (dy_dtype == UNREAL_F32)
    cell_segment_sum_kernel<float><<<(unsigned)ctas, 256, kSmem, as_stream(stream)>>>(reinterpret_cast<const float*>(dy), pos, out, s, rows_per_cta);
  else
    cell_segment_sum_kernel<__nv_bfloat16><<<(unsigned)ctas, 256, kSmem, as_stream(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(dy), pos, out, s, rows_per_cta);
  UNREAL_LAUNCH_CHECK("cell_segment_sum_kernel");
  return UNREAL_OK;
}

// ---- the same three cell entry points with bf16 gate storage (gates / gates_act are bf16 [N,1024]) ------------------------
extern "C" int unreal_lstm_cell_fwd_g16(void* gates_bf16, const float* c_prev, float* c_out, float* h_out, void* h16_out,
                                        int h16_ld, int n, void* stream) {
  UNREAL_REQUIRE(gates_bf16 && c_prev && c_out && h_out && h16_out && n > 0, "unreal_lstm_cell_fwd_g16: null buffer or n <= 0");
  UNREAL_REQUIRE(h16_ld >= 256, "unreal_lstm_cell_fwd_g16: h16_ld %d < 256", h16_ld);
  UNREAL_REQUIRE(h16_ld % 8 == 0 && aligned16(gates_bf16) && aligned16(c_prev) && aligned16(c_out) && aligned16(h_out) &&
                     aligned16(h16_out), "unreal_lstm_cell_fwd_g16: buffers must be 16-byte aligned, h16_ld a multiple of 8");
  lstm_cell_fwd8_kernel<<<(n * 32 + 255) / 256, 256, 0, as_stream(stream)>>>(
      reinterpret_cast<__nv_bfloat16*>(gates_bf16), c_prev, c_out, h_out, reinterpret_cast<__nv_bfloat16*>(h16_out), n, h16_ld);
  UNREAL_LAUNCH_CHECK("lstm_cell_fwd_kernel<bf16>");
  return UNREAL_OK;
}

extern "C" int unreal_lstm_cell_act_g16(const void* gates_bf16, float* c_state, float* h_state, float* h_out,
                                        const uint8_t* active, int n, void* stream) {
  UNREAL_REQUIRE(gates_bf16 && c_state && h_state && n > 0, "unreal_lstm_cell_act_g16: null buffer or n <= 0");
  UNREAL_REQUIRE(aligned16(gates_bf16) && aligned16(c_state) && aligned16(h_state) && aligned16(h_out),
                 "unreal_lstm_cell_act_g16: buffers must be 16-byte aligned");
  lstm_cell_act8_kernel<<<(n * 32 + 255) / 256, 256, 0, as_stream(stream)>>>(
      reinterpret_cast<const __nv_bfloat16*>(gates_bf16), c_state, h_state, h_out, active, n);
  UNREAL_LAUNCH_CHECK("lstm_cell_act_kernel<bf16>");
  return UNREAL_OK;
}

extern "C" int unreal_lstm_cell_act_heads(const void* gates_bf16, float* c_state, float* h_state, const uint8_t* active, int n,
                                          const float* wp, const float* bp, const float* wv, const float* bv, int a,
                                          float* pi_out, float* v_out, void* stream) {
  UNREAL_REQUIRE(gates_bf16 && c_state && h_state && wp && bp && wv && pi_out && v_out && n > 0,
                 "unreal_lstm_cell_act_heads: null buffer or n <= 0");
  UNREAL_REQUIRE(a >= 1 && a <= kHeadMaxA, "unreal_lstm_cell_act_heads: action count %d not in 1..7", a);
  UNREAL_REQUIRE(aligned16(gates_bf16) && aligned16(c_state) && aligned16(h_state),
                 "unreal_lstm_cell_act_heads: buffers must be 16-byte aligned");
  const int sms = sm_count();
  if (sms <= 0) return UNREAL_ECUDA;
  const int want = (n + 7) / 8;
  lstm_cell_act_heads8_kernel<<<want < sms * 4 ? want : sms * 4, 256, 0, as_stream(stream)>>>(
      reinterpret_cast<const __nv_bfloat16*>(gates_bf16), c_state, h_state, active, n, wp, bp, wv, bv, a, pi_out, v_out);
  UNREAL_LAUNCH_CHECK("lstm_cell_act_heads8_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_lstm_cell_bwd_g16(const void* gates_act_bf16, const float* c_prev, const float* c, const float* dh,
                                        const float* dh_rec, float* dc, void* dgates_bf16, int n, void* stream) {
  UNREAL_REQUIRE(gates_act_bf16 && c_prev && c && dh && dc && dgates_bf16 && n > 0,
                 "unreal_lstm_cell_bwd_g16: null buffer or n <= 0");
  lstm_cell_bwd_kernel<__nv_bfloat16><<<(n * 256 + 255) / 256, 256, 0, as_stream(stream)>>>(
      reinterpret_cast<const __nv_bfloat16*>(gates_act_bf16), c_prev, c, dh, dc, reinterpret_cast<__nv_bfloat16*>(dgates_bf16), n,
      dh_rec);
  UNREAL_LAUNCH_CHECK("lstm_cell_bwd_kernel<bf16>");
  return UNREAL_OK;
}
