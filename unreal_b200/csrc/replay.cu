// K5: device-resident replay ring with reward-prediction-balanced and sequence sampling.
// Replaces Experience (train/experience.py:48-153) for N envs at once; each env keeps the
// reference's exact index semantics and draws from its own numpy-legacy MT19937 stream, so
// sampled indices are bit-identical to `Experience(H, RandomState(seed_n))` fed the same frames.
//
// HBM layout: rec [N, H] u64 env-major (a sampled sequence is 21 consecutive records = 168
// contiguous bytes; an RP rank-select streams one env's records linearly), top [N] i64,
// count / n_pos / n_neg [N] i32.  8 B per frame: 2000 frames x 8192 envs = 131 MB per GPU,
// where the reference's deque of 84x84x3 float64 frames would be 2.8 TB.
#include <new>

#include "common.cuh"
#include "maze_core.cuh"
#include "mt19937_core.cuh"
#include "ring_core.cuh"

struct unreal_replay {
  int n, h;
  uint64_t* rec;
  int64_t* top;
  int32_t* count;
  int32_t* n_pos;
  int32_t* n_neg;
};

namespace unreal {

__device__ __forceinline__ RingRef ring_of(const unreal_replay& R, int e) {
  return RingRef{R.rec + (size_t)e * R.h, R.h, R.top + e, R.count + e, R.n_pos + e, R.n_neg + e};
}

__global__ void replay_add_kernel(unreal_replay R, const uint64_t* __restrict__ frames) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= R.n) return;
  ring_add(ring_of(R, e), frames[e]);
}

__global__ void replay_state_kernel(unreal_replay R, uint8_t* full, int32_t* count, int64_t* top, int32_t* n_pos,
                                    int32_t* n_neg) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= R.n) return;
  if (full) full[e] = R.count[e] >= R.h;   // is_full :96-97
  if (count) count[e] = R.count[e];
  if (top) top[e] = R.top[e];
  if (n_pos) n_pos[e] = R.n_pos[e];
  if (n_neg) n_neg[e] = R.n_neg[e];
}

// one warp per env; lane 0 owns the RNG stream, lanes gather the records
__global__ void __launch_bounds__(128) replay_sample_sequence_kernel(unreal_replay R, uint32_t* mt, int32_t* mt_pos,
                                                                     int L, int32_t* out_start, int32_t* out_len,
                                                                     uint64_t* out_rec) {
  const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (e >= R.n) return;
  const RingRef r = ring_of(R, e);
  const bool ready = *r.count >= R.h;      // the reference only samples a full buffer (trainer.py:446-448)
  int start = -1;
  if (lane == 0 && ready) {
    MtStream s{mt + e, (int64_t)R.n, mt_pos + e};
    start = (int)mt_randint(s, (uint32_t)(R.h - L - 1));   // randint(0, H - L - 1)  :103
  }
  start = __shfl_sync(0xffffffffu, start, 0);
  if (!ready) {
    if (lane == 0) { out_start[e] = -1; out_len[e] = 0; }
    if (lane < L) out_rec[(size_t)e * L + lane] = 0ull;
    return;
  }
  // lanes 0..L hold raw positions start..start+L; shift by one when the first is terminal (:105-107)
  uint64_t v = (lane <= L) ? ring_at_raw(r, start + lane) : 0ull;
  const int first_term = __shfl_sync(0xffffffffu, frame_terminal(v), 0);
  if (first_term) {
    v = __shfl_down_sync(0xffffffffu, v, 1);
    start += 1;
  }
  const unsigned in_seq = (L >= 32) ? 0xffffffffu : ((1u << L) - 1u);
  const unsigned terms = __ballot_sync(0xffffffffu, frame_terminal(v) != 0) & in_seq;
  const int len = terms ? (__ffs(terms)) : L;            // stop after the first terminal (:111-116)
  if (lane == 0) { out_start[e] = start; out_len[e] = len; }
  if (lane < L) out_rec[(size_t)e * L + lane] = (lane < len) ? v : 0ull;
}

__global__ void __launch_bounds__(128) replay_sample_rp_kernel(unreal_replay R, uint32_t* mt, int32_t* mt_pos,
                                                               int32_t* out_start, uint64_t* out_rec) {
  const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (e >= R.n) return;
  const RingRef r = ring_of(R, e);
  const int n_pos = *r.n_pos, n_neg = *r.n_neg;
  if (n_pos + n_neg <= 0) {                 // fewer than 4 frames: the reference would raise
    if (lane == 0) out_start[e] = -1;
    if (lane < 4) out_rec[(size_t)e * 4 + lane] = 0ull;
    return;
  }
  int from_neg = 0, k = 0;
  if (lane == 0) {
    MtStream s{mt + e, (int64_t)R.n, mt_pos + e};
    from_neg = (mt_randint(s, 2u) == 0u) ? 1 : 0;        // randint(2) == 0  :125-128
    if (n_pos == 0) from_neg = 1;                        // :130-135
    else if (n_neg == 0) from_neg = 0;
    k = (int)mt_randint(s, (uint32_t)(from_neg ? n_neg : n_pos));   // :137-141
  }
  from_neg = __shfl_sync(0xffffffffu, from_neg, 0);
  k = __shfl_sync(0xffffffffu, k, 0);
  // warp rank-select over the eligible absolute range: 32 frames per ballot, the loads of 8 ballots (2 KB of records)
  // issued together -- the scan is a chain of dependent HBM round trips otherwise (55 us at 8192 envs, 0.36 of HBM)
  const int64_t top = *r.top;
  const int64_t lo = top + 3 < 3 ? 3 : top + 3;
  const int64_t hi = top + *r.count - 1;
  int64_t end = -1;
  constexpr int kBatch = 8;
  // slot(abs) = abs % H with ONE 64-bit modulo per env: the eligible range is shorter than H, so a running slot
  // needs a single conditional subtraction (a 64-bit `%` per record was most of this kernel's time)
  const int H = r.H;
  const int slot0 = (int)(lo % H);
  const int span = (int)(hi - lo + 1);                     // <= H - 3
  for (int off0 = 0; off0 < span && end < 0; off0 += 32 * kBatch) {
    uint64_t v[kBatch];
#pragma unroll
    for (int j = 0; j < kBatch; ++j) {
      const int off = off0 + 32 * j + lane;
      int slot = slot0 + off;
      if (slot >= H) slot -= H;
      v[j] = (off < span) ? r.rec[slot] : 0ull;
    }
#pragma unroll
    for (int j = 0; j < kBatch; ++j) {
      const int off = off0 + 32 * j + lane;
      const bool match = (off < span) && (((frame_reward(v[j]) > 0) ? 1 : 0) != from_neg);
      const unsigned b = __ballot_sync(0xffffffffu, match);
      const int c = __popc(b);
      if (end < 0) {
        if (k < c) {
          unsigned bits = b;
          for (int i = 0; i < k; ++i) bits &= bits - 1;     // drop the k lowest set bits
          end = lo + off0 + 32 * j + (__ffs(bits) - 1);
        } else {
          k -= c;
        }
      }
    }
  }
  const int start = (int)(end - 3 - top);                 // raw_start_frame_index :143-144
  if (lane == 0) out_start[e] = start;
  if (lane < 4) out_rec[(size_t)e * 4 + lane] = ring_at_raw(r, start + lane);
}

__global__ void frame_unpack_kernel(const uint64_t* __restrict__ rec, int m, int32_t* pos0, int32_t* pos1,
                                    int32_t* action, float* reward, uint8_t* terminal, int32_t* last_action,
                                    float* last_reward, uint8_t* valid) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const uint64_t r = rec[i];
  if (pos0) { pos0[2 * i] = frame_x0(r); pos0[2 * i + 1] = frame_y0(r); }
  if (pos1) { pos1[2 * i] = frame_x1(r); pos1[2 * i + 1] = frame_y1(r); }
  if (action) action[i] = frame_action(r);
  if (reward) reward[i] = (float)frame_reward(r);
  if (terminal) terminal[i] = (uint8_t)frame_terminal(r);
  if (last_action) last_action[i] = frame_last_action(r);
  if (last_reward) last_reward[i] = (float)frame_last_reward(r);
  if (valid) valid[i] = (uint8_t)frame_valid(r);
}

// ---- framed mode (SURVEY.md 8f-4: lab / gym / indoor / synthetic frames have no closed form) ------------
// The 8-byte record keeps the index logic (action, reward SIGN, terminal, last_action); everything
// the reference's deque holds by reference -- the 84x84x3 frame, the pixel-change map, the float
// reward, the objective vector -- lives in caller-owned payload arrays [N, H, item] addressed by the
// same slot, written by ring_store and read back by replay_gather.

__global__ void replay_add_slots_kernel(unreal_replay R, const uint64_t* __restrict__ frames, int32_t* slot) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= R.n) return;
  const RingRef r = ring_of(R, e);
  const int64_t index = *r.top + *r.count;           // where ring_add writes when it accepts the frame
  slot[e] = ring_add(r, frames[e]) ? (int32_t)(index % R.h) : -1;
}

__global__ void frame_pack_kernel(const int32_t* __restrict__ action, const float* __restrict__ reward,
                                  const uint8_t* __restrict__ terminal, const int32_t* __restrict__ last_action,
                                  const float* __restrict__ last_reward, const uint8_t* __restrict__ active,
                                  uint64_t* __restrict__ rec, int n) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  if (active && !active[e]) { rec[e] = 0ull; return; }
  rec[e] = framed_record(action[e], reward[e], terminal[e], last_action ? last_action[e] : 0,
                         last_reward ? last_reward[e] : 0.f);
}

// payload[e, slot[e], :] <- src[e, :]; one CTA per env walks the item in W-sized words
template <typename W>
__global__ void __launch_bounds__(256) ring_store_kernel(W* __restrict__ payload, const W* __restrict__ src,
                                                         const int32_t* __restrict__ slot, int h, int words) {
  const int e = blockIdx.x;
  const int s = slot[e];
  if (s < 0) return;
  W* dst = payload + ((size_t)e * h + s) * words;
  const W* from = src + (size_t)e * words;
  for (int w = threadIdx.x; w < words; w += blockDim.x) dst[w] = from[w];
}

// out[e, :] <- src[idx ? idx[e] : e, :] for the envs with mask[e] != 0 (mask NULL: all); one CTA per env
template <typename W>
__global__ void __launch_bounds__(256) rows_select_kernel(W* __restrict__ out, const W* __restrict__ src,
                                                          const int64_t* __restrict__ idx, const uint8_t* __restrict__ mask,
                                                          int words) {
  const int e = blockIdx.x;
  if (mask != nullptr && mask[e] == 0) return;
  const W* from = src + (size_t)(idx ? idx[e] : e) * words;
  W* dst = out + (size_t)e * words;
  for (int w = threadIdx.x; w < words; w += blockDim.x) dst[w] = from[w];
}

// small items (a reward, an objective vector): one thread per word
template <typename W>
__global__ void ring_store_flat_kernel(W* __restrict__ payload, const W* __restrict__ src,
                                       const int32_t* __restrict__ slot, int n, int h, int words) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n * words) return;
  const int e = (int)(i / words), w = (int)(i % words);
  const int s = slot[e];
  if (s >= 0) payload[((size_t)e * h + s) * words + w] = src[i];
}

__device__ __forceinline__ long long gather_src_item(const unreal_replay& R, const int32_t* start, const int32_t* len,
                                                     int e, int t) {
  const int st = start[e];
  if (st < 0 || (len && t >= len[e])) return -1;
  return (long long)e * R.h + (R.top[e] + st + t) % R.h;
}

// out item (e, t) <- payload[e, (top + start + t) % H] for t < len[e], zeros beyond; one CTA per item
template <typename W>
__global__ void __launch_bounds__(256) replay_gather_kernel(unreal_replay R, const W* __restrict__ payload,
                                                            const int32_t* __restrict__ start,
                                                            const int32_t* __restrict__ len, int L, int time_major,
                                                            W* __restrict__ out, int words) {
  const int e = blockIdx.x / L, t = blockIdx.x % L;
  const long long src = gather_src_item(R, start, len, e, t);
  W* dst = out + (time_major ? ((size_t)t * R.n + e) : (size_t)blockIdx.x) * words;
  W zero; memset(&zero, 0, sizeof(W));
  if (src < 0) {
    for (int w = threadIdx.x; w < words; w += blockDim.x) dst[w] = zero;
    return;
  }
  const W* from = payload + (size_t)src * words;
  for (int w = threadIdx.x; w < words; w += blockDim.x) dst[w] = from[w];
}

template <typename W>
__global__ void replay_gather_flat_kernel(unreal_replay R, const W* __restrict__ payload,
                                          const int32_t* __restrict__ start, const int32_t* __restrict__ len, int L,
                                          int time_major, W* __restrict__ out, int words) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)R.n * L * words) return;
  const long long item = i / words;
  const int w = (int)(i % words);
  const int e = (int)(item / L), t = (int)(item % L);
  const long long src = gather_src_item(R, start, len, e, t);
  W v; memset(&v, 0, sizeof(W));
  if (src >= 0) v = payload[(size_t)src * words + w];
  out[(time_major ? ((size_t)t * R.n + e) : (size_t)item) * words + w] = v;
}

}  // namespace unreal

using namespace unreal;

extern "C" int unreal_replay_create(unreal_replay_t** out, int n_envs, int history_size) {
  UNREAL_REQUIRE(out != nullptr, "unreal_replay_create: out is null");
  UNREAL_REQUIRE(n_envs >= 1 && history_size >= 4, "unreal_replay_create: need n_envs >= 1 and history_size >= 4");
  unreal_replay* r = new (std::nothrow) unreal_replay();
  if (!r) { set_error("unreal_replay_create: out of host memory"); return UNREAL_ENOMEM; }
  r->n = n_envs; r->h = history_size;
  r->rec = nullptr; r->top = nullptr; r->count = r->n_pos = r->n_neg = nullptr;
  cudaError_t e = cudaMalloc(&r->rec, (size_t)n_envs * history_size * sizeof(uint64_t));
  if (e == cudaSuccess) e = cudaMalloc(&r->top, (size_t)n_envs * sizeof(int64_t));
  if (e == cudaSuccess) e = cudaMalloc(&r->count, (size_t)n_envs * sizeof(int32_t));
  if (e == cudaSuccess) e = cudaMalloc(&r->n_pos, (size_t)n_envs * sizeof(int32_t));
  if (e == cudaSuccess) e = cudaMalloc(&r->n_neg, (size_t)n_envs * sizeof(int32_t));
  if (e != cudaSuccess) {
    unreal_replay_destroy(r);
    cuda_fail(e, "unreal_replay_create: cudaMalloc");
    return e == cudaErrorMemoryAllocation ? UNREAL_ENOMEM : UNREAL_ECUDA;
  }
  *out = r;
  int rc = unreal_replay_reset(r, nullptr);
  if (rc == UNREAL_OK) { cudaError_t s = cudaStreamSynchronize(nullptr); if (s != cudaSuccess) rc = cuda_fail(s, "sync"); }
  return rc;
}

extern "C" int unreal_replay_destroy(unreal_replay_t* r) {
  if (!r) return UNREAL_OK;
  cudaFree(r->rec); cudaFree(r->top); cudaFree(r->count); cudaFree(r->n_pos); cudaFree(r->n_neg);
  delete r;
  return UNREAL_OK;
}

extern "C" int unreal_replay_reset(unreal_replay_t* r, void* stream) {
  UNREAL_REQUIRE(r != nullptr, "unreal_replay_reset: null handle");
  cudaStream_t st = as_stream(stream);
  UNREAL_CUDA(cudaMemsetAsync(r->rec, 0, (size_t)r->n * r->h * sizeof(uint64_t), st));
  UNREAL_CUDA(cudaMemsetAsync(r->top, 0, (size_t)r->n * sizeof(int64_t), st));
  UNREAL_CUDA(cudaMemsetAsync(r->count, 0, (size_t)r->n * sizeof(int32_t), st));
  UNREAL_CUDA(cudaMemsetAsync(r->n_pos, 0, (size_t)r->n * sizeof(int32_t), st));
  UNREAL_CUDA(cudaMemsetAsync(r->n_neg, 0, (size_t)r->n * sizeof(int32_t), st));
  return UNREAL_OK;
}

extern "C" int unreal_replay_add(unreal_replay_t* r, const uint64_t* frame_rec, void* stream) {
  UNREAL_REQUIRE(r && frame_rec, "unreal_replay_add: null argument");
  replay_add_kernel<<<(r->n + 127) / 128, 128, 0, as_stream(stream)>>>(*r, frame_rec);
  UNREAL_LAUNCH_CHECK("replay_add_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_replay_state(unreal_replay_t* r, uint8_t* full, int32_t* count, int64_t* top, int32_t* n_pos,
                                   int32_t* n_neg, void* stream) {
  UNREAL_REQUIRE(r != nullptr, "unreal_replay_state: null handle");
  replay_state_kernel<<<(r->n + 127) / 128, 128, 0, as_stream(stream)>>>(*r, full, count, top, n_pos, n_neg);
  UNREAL_LAUNCH_CHECK("replay_state_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_replay_sample_sequence(unreal_replay_t* r, uint32_t* mt, int32_t* mt_pos, int seq_len,
                                             int32_t* start, int32_t* len, uint64_t* rec, void* stream) {
  UNREAL_REQUIRE(r && mt && mt_pos && start && len && rec, "unreal_replay_sample_sequence: null argument");
  UNREAL_REQUIRE(seq_len >= 1 && seq_len <= 31, "unreal_replay_sample_sequence: seq_len %d not in 1..31", seq_len);
  UNREAL_REQUIRE(r->h - seq_len - 1 >= 1, "unreal_replay_sample_sequence: history %d too small for seq_len %d", r->h, seq_len);
  long long threads = (long long)r->n * 32;
  replay_sample_sequence_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, as_stream(stream)>>>(
      *r, mt, mt_pos, seq_len, start, len, rec);
  UNREAL_LAUNCH_CHECK("replay_sample_sequence_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_replay_sample_rp(unreal_replay_t* r, uint32_t* mt, int32_t* mt_pos, int32_t* start,
                                       uint64_t* rec, void* stream) {
  UNREAL_REQUIRE(r && mt && mt_pos && start && rec, "unreal_replay_sample_rp: null argument");
  long long threads = (long long)r->n * 32;
  replay_sample_rp_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, as_stream(stream)>>>(*r, mt, mt_pos, start, rec);
  UNREAL_LAUNCH_CHECK("replay_sample_rp_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_frame_unpack(const uint64_t* rec, int m, int32_t* pos0, int32_t* pos1, int32_t* action,
                                   float* reward, uint8_t* terminal, int32_t* last_action, float* last_reward,
                                   uint8_t* valid, void* stream) {
  UNREAL_REQUIRE(m >= 0, "unreal_frame_unpack: negative size");
  if (m == 0) return UNREAL_OK;
  UNREAL_REQUIRE(rec != nullptr, "unreal_frame_unpack: rec is null");
  frame_unpack_kernel<<<(m + 255) / 256, 256, 0, as_stream(stream)>>>(rec, m, pos0, pos1, action, reward, terminal,
                                                                     last_action, last_reward, valid);
  UNREAL_LAUNCH_CHECK("frame_unpack_kernel");
  return UNREAL_OK;
}

// Checkpointing (main.py:356,469-519 saves only the network; the replay memory and RNG are lost on
// restart there -- here the ring can be exported / imported verbatim).  direction 0: ring -> caller
// buffers, 1: caller buffers -> ring.  rec [N,H] u64, top [N] i64, count / n_pos / n_neg [N] i32.
extern "C" int unreal_replay_copy(unreal_replay_t* r, int direction, uint64_t* rec, int64_t* top, int32_t* count,
                                  int32_t* n_pos, int32_t* n_neg, void* stream) {
  UNREAL_REQUIRE(r && rec && top && count && n_pos && n_neg, "unreal_replay_copy: null argument");
  UNREAL_REQUIRE(direction == 0 || direction == 1, "unreal_replay_copy: direction must be 0 (export) or 1 (import)");
  cudaStream_t st = as_stream(stream);
  const size_t n = (size_t)r->n;
  struct { void* ring; void* user; size_t bytes; } parts[5] = {
      {r->rec, rec, n * r->h * sizeof(uint64_t)}, {r->top, top, n * sizeof(int64_t)},
      {r->count, count, n * sizeof(int32_t)}, {r->n_pos, n_pos, n * sizeof(int32_t)}, {r->n_neg, n_neg, n * sizeof(int32_t)}};
  for (auto& p : parts) {
    if (direction == 0) UNREAL_CUDA(cudaMemcpyAsync(p.user, p.ring, p.bytes, cudaMemcpyDeviceToDevice, st));
    else UNREAL_CUDA(cudaMemcpyAsync(p.ring, p.user, p.bytes, cudaMemcpyDeviceToDevice, st));
  }
  return UNREAL_OK;
}

// ---- framed mode ---------------------------------------------------------------------------------------
extern "C" int unreal_frame_pack(const int32_t* action, const float* reward, const uint8_t* terminal,
                                 const int32_t* last_action, const float* last_reward, const uint8_t* active,
                                 uint64_t* rec, int n, void* stream) {
  UNREAL_REQUIRE(n >= 0, "unreal_frame_pack: negative size");
  if (n == 0) return UNREAL_OK;
  UNREAL_REQUIRE(action && reward && terminal && rec, "unreal_frame_pack: null argument");
  frame_pack_kernel<<<(n + 255) / 256, 256, 0, as_stream(stream)>>>(action, reward, terminal, last_action, last_reward,
                                                                   active, rec, n);
  UNREAL_LAUNCH_CHECK("frame_pack_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_replay_add_slots(unreal_replay_t* r, const uint64_t* frame_rec, int32_t* slot, void* stream) {
  UNREAL_REQUIRE(r && frame_rec && slot, "unreal_replay_add_slots: null argument");
  replay_add_slots_kernel<<<(r->n + 127) / 128, 128, 0, as_stream(stream)>>>(*r, frame_rec, slot);
  UNREAL_LAUNCH_CHECK("replay_add_slots_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_ring_store(void* payload, const void* src, const int32_t* slot, int n_envs, int history_size,
                                 long long item_bytes, void* stream) {
  UNREAL_REQUIRE(payload && src && slot, "unreal_ring_store: null argument");
  UNREAL_REQUIRE(n_envs >= 1 && history_size >= 1, "unreal_ring_store: bad ring shape %d x %d", n_envs, history_size);
  UNREAL_REQUIRE(item_bytes >= 4 && item_bytes % 4 == 0 && item_bytes < (1ll << 31),
                 "unreal_ring_store: item_bytes %lld must be a positive multiple of 4", item_bytes);
  cudaStream_t st = as_stream(stream);
  const bool v16 = item_bytes % 16 == 0 && aligned16(payload) && aligned16(src);
  const int words = (int)(item_bytes / (v16 ? 16 : 4));
  if (words >= 128) {
    if (v16) ring_store_kernel<uint4><<<n_envs, 256, 0, st>>>((uint4*)payload, (const uint4*)src, slot, history_size, words);
    else ring_store_kernel<uint32_t><<<n_envs, 256, 0, st>>>((uint32_t*)payload, (const uint32_t*)src, slot, history_size, words);
  } else {
    const long long total = (long long)n_envs * words;
    const unsigned grid = (unsigned)((total + 255) / 256);
    if (v16) ring_store_flat_kernel<uint4><<<grid, 256, 0, st>>>((uint4*)payload, (const uint4*)src, slot, n_envs, history_size, words);
    else ring_store_flat_kernel<uint32_t><<<grid, 256, 0, st>>>((uint32_t*)payload, (const uint32_t*)src, slot, n_envs, history_size, words);
  }
  UNREAL_LAUNCH_CHECK("ring_store_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_rows_select(void* out, const void* src, const int64_t* idx, const uint8_t* mask, int n,
                                  long long item_bytes, void* stream) {
  UNREAL_REQUIRE(out && src && n >= 0, "unreal_rows_select: null argument or n < 0");
  UNREAL_REQUIRE(item_bytes >= 4 && item_bytes % 4 == 0 && item_bytes < (1ll << 31),
                 "unreal_rows_select: item_bytes %lld must be a positive multiple of 4", item_bytes);
  if (n == 0) return UNREAL_OK;
  const bool v16 = item_bytes % 16 == 0 && aligned16(out) && aligned16(src);
  const int words = (int)(item_bytes / (v16 ? 16 : 4));
  if (v16) rows_select_kernel<uint4><<<n, 256, 0, as_stream(stream)>>>((uint4*)out, (const uint4*)src, idx, mask, words);
  else rows_select_kernel<uint32_t><<<n, 256, 0, as_stream(stream)>>>((uint32_t*)out, (const uint32_t*)src, idx, mask, words);
  UNREAL_LAUNCH_CHECK("rows_select_kernel");
  return UNREAL_OK;
}

extern "C" int unreal_replay_gather(unreal_replay_t* r, const void* payload, long long item_bytes, const int32_t* start,
                                    const int32_t* len, int seq_len, int time_major, void* out, void* stream) {
  UNREAL_REQUIRE(r && payload && start && out, "unreal_replay_gather: null argument");
  UNREAL_REQUIRE(seq_len >= 1 && seq_len <= r->h, "unreal_replay_gather: seq_len %d not in 1..%d", seq_len, r->h);
  UNREAL_REQUIRE(item_bytes >= 4 && item_bytes % 4 == 0 && item_bytes < (1ll << 31),
                 "unreal_replay_gather: item_bytes %lld must be a positive multiple of 4", item_bytes);
  cudaStream_t st = as_stream(stream);
  const bool v16 = item_bytes % 16 == 0 && aligned16(payload) && aligned16(out);
  const int words = (int)(item_bytes / (v16 ? 16 : 4));
  const long long items = (long long)r->n * seq_len;
  UNREAL_REQUIRE(items < (1ll << 31), "unreal_replay_gather: %lld items exceed the grid", items);
  if (words >= 128) {
    if (v16) replay_gather_kernel<uint4><<<(unsigned)items, 256, 0, st>>>(*r, (const uint4*)payload, start, len, seq_len, time_major, (uint4*)out, words);
    else replay_gather_kernel<uint32_t><<<(unsigned)items, 256, 0, st>>>(*r, (const uint32_t*)payload, start, len, seq_len, time_major, (uint32_t*)out, words);
  } else {
    const long long total = items * words;
    const unsigned grid = (unsigned)((total + 255) / 256);
    if (v16) replay_gather_flat_kernel<uint4><<<grid, 256, 0, st>>>(*r, (const uint4*)payload, start, len, seq_len, time_major, (uint4*)out, words);
    else replay_gather_flat_kernel<uint32_t><<<grid, 256, 0, st>>>(*r, (const uint32_t*)payload, start, len, seq_len, time_major, (uint32_t*)out, words);
  }
  UNREAL_LAUNCH_CHECK("replay_gather_kernel");
  return UNREAL_OK;
}
