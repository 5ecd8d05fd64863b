// Evaluation of a frozen policy on the maze (Evaluator, unreal_b200/train/evaluator.py): everything of one step after
// the policy, for all envs in one launch.
//
// Per step the evaluator runs the acting GEMM on its own bf16 [x, h] operand, the model's cell + heads kernel(s), and
// this kernel, which for each active env picks the action, steps the maze, keeps the episode accounting (eval_core.cuh)
// and then writes the env's row of the NEXT step's GEMM operand itself: fc1 of the new cell from the 49-row acting
// table, one-hot(last action) ++ [last reward], zero padding, and h rounded to bf16 (round-to-nearest-even, what
// `xh[:, kx:].copy_(h)` does) -- or zeros for h and the LSTM state rows when the episode ended.  That replaces the cell
// gather, the lar build, the casts and copies and the accounting ops of the generic loop.
//
// Block of 32 envs: phase 1, one thread per env (warp 0), runs the scalar logic (the MT19937 words of adjacent envs are
// adjacent, as in choose_action_kernel); phase 2, 8 warps with 4 envs each, writes the 1 KB operand rows with 16-byte
// stores (all loads of a warp issued before its stores) and zeroes the state rows of the envs that were reset.
#include <cuda_bf16.h>

#include "common.cuh"
#include "eval_core.cuh"

namespace unreal {

namespace {

constexpr int kEvalEnvs = 32;                          // envs per block: phase 1 is one warp
constexpr int kEvalThreads = 256;                      // phase 2: 8 warps
constexpr int kEnvsPerWarp = kEvalEnvs / (kEvalThreads / 32);

struct EvalRows {
  float* lstm_c;                 // [M,256]
  float* lstm_h;                 // [M,256]
  const __nv_bfloat16* fc_tab;   // [49,256]
  __nv_bfloat16* xh;             // [M, ld_xh]: columns [0,256) fc1, [256,kx) lar + padding, [kx,kx+256) h
  int64_t ld_xh;
  int kx;
};

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  const __nv_bfloat16 l = __float2bfloat16_rn(lo), h = __float2bfloat16_rn(hi);
  return (uint32_t)__bfloat16_as_ushort(l) | ((uint32_t)__bfloat16_as_ushort(h) << 16);
}

template <int kA>
__global__ void __launch_bounds__(kEvalThreads) maze_eval_act_kernel(EvalState S, MazeLayout L, EvalRows R,
                                                                     const float* __restrict__ pi, int a, int greedy,
                                                                     uint32_t* mt, int32_t* mt_pos) {
  // phase 1 (warp 0): bit 0 stepped, bit 1 done, bits 2..7 cell, bits 8..15 last action, bits 16..17 last reward + 1
  __shared__ int s_info[kEvalEnvs];
  const int aa = kA > 0 ? kA : a;
  if (threadIdx.x < kEvalEnvs) {
    const int e = blockIdx.x * kEvalEnvs + threadIdx.x;
    int info = 0;
    if (e < S.m) {
      MtStream s{mt + e, (int64_t)S.m, mt_pos + e};
      const EvalOut o = eval_env_step(S, L, e, pi + (int64_t)e * aa, aa, greedy, s);
      if (o.stepped)
        info = 1 | (o.done << 1) | (eval_cell_index(o.x, o.y) << 2) | (o.last_action << 8) | ((o.last_reward + 1) << 16);
    }
    s_info[threadIdx.x] = info;
  }
  __syncthreads();

  // phase 2: the operand rows (and the state rows of reset envs); each warp owns kEnvsPerWarp envs and issues all their
  // loads before any store, so the round trips overlap
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int inf[kEnvsPerWarp];
  uint4 fc[kEnvsPerWarp], hv[kEnvsPerWarp];
#pragma unroll
  for (int j = 0; j < kEnvsPerWarp; ++j) {
    const int t = warp * kEnvsPerWarp + j;
    inf[j] = s_info[t];
    fc[j] = make_uint4(0u, 0u, 0u, 0u);
    hv[j] = make_uint4(0u, 0u, 0u, 0u);
    if ((inf[j] & 1) == 0) continue;
    const int64_t ee = (int64_t)blockIdx.x * kEvalEnvs + t;
    fc[j] = reinterpret_cast<const uint4*>(R.fc_tab + ((inf[j] >> 2) & 63) * 256)[lane];
    if ((inf[j] & 2) == 0) {     // h of the step just taken, rounded to bf16 (a reset env gets zeros)
      const float4* h4 = reinterpret_cast<const float4*>(R.lstm_h + ee * 256);
      const float4 v0 = h4[2 * lane], v1 = h4[2 * lane + 1];
      hv[j] = make_uint4(pack_bf16x2(v0.x, v0.y), pack_bf16x2(v0.z, v0.w), pack_bf16x2(v1.x, v1.y), pack_bf16x2(v1.z, v1.w));
    }
  }
  const int chunks_lar = (R.kx - 256) >> 3;
#pragma unroll
  for (int j = 0; j < kEnvsPerWarp; ++j) {
    if ((inf[j] & 1) == 0) continue;
    const int64_t ee = (int64_t)blockIdx.x * kEvalEnvs + warp * kEnvsPerWarp + j;
    __nv_bfloat16* row = R.xh + ee * R.ld_xh;
    reinterpret_cast<uint4*>(row)[lane] = fc[j];
    reinterpret_cast<uint4*>(row + R.kx)[lane] = hv[j];
    if (inf[j] & 2) {
      float4* c4 = reinterpret_cast<float4*>(R.lstm_c + ee * 256);
      float4* h4 = reinterpret_cast<float4*>(R.lstm_h + ee * 256);
      const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      c4[2 * lane] = z; c4[2 * lane + 1] = z; h4[2 * lane] = z; h4[2 * lane + 1] = z;
    }
    const int la = (inf[j] >> 8) & 255, lr = ((inf[j] >> 16) & 3) - 1;
    for (int q = lane; q < chunks_lar; q += 32) {
      uint32_t w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
        w[i] = pack_bf16x2(eval_lar_col(q * 8 + 2 * i, aa, la, lr), eval_lar_col(q * 8 + 2 * i + 1, aa, la, lr));
      reinterpret_cast<uint4*>(row + 256)[q] = make_uint4(w[0], w[1], w[2], w[3]);
    }
  }
}

}  // namespace
}  // namespace unreal

using namespace unreal;

extern "C" int unreal_maze_eval_act(const float* pi, int a, int greedy, uint32_t* mt, int32_t* mt_pos, int32_t* pos,
                                    int32_t* last_action, float* last_reward, float* ep_score, int32_t* ep_length,
                                    int32_t* ep_index, uint8_t* active, float* res_score, int32_t* res_length,
                                    uint8_t* res_finished, int episodes, int max_steps, float* lstm_c, float* lstm_h,
                                    const void* fc_tab_bf16, void* xh_bf16, int64_t ld_xh, int kx, int n, void* stream) {
  UNREAL_REQUIRE(n >= 0, "unreal_maze_eval_act: n < 0");
  UNREAL_REQUIRE(pi && pos && last_action && last_reward && ep_score && ep_length && ep_index && active && res_score &&
                 res_length && res_finished && lstm_c && lstm_h && fc_tab_bf16 && xh_bf16,
                 "unreal_maze_eval_act: null buffer");
  UNREAL_REQUIRE(greedy || (mt && mt_pos), "unreal_maze_eval_act: sampling needs the MT19937 streams");
  UNREAL_REQUIRE(a >= 1 && a <= 32, "unreal_maze_eval_act: action size %d not in 1..32", a);
  UNREAL_REQUIRE(episodes >= 1 && max_steps >= 1, "unreal_maze_eval_act: episodes and max_steps must be >= 1");
  UNREAL_REQUIRE(kx >= 256 + a + 1 && kx % 8 == 0 && ld_xh >= kx + 256 && ld_xh % 8 == 0,
                 "unreal_maze_eval_act: kx (%d) must be a multiple of 8 holding 256 + a + 1 columns, ld_xh (%lld) >= kx + 256",
                 kx, (long long)ld_xh);
  UNREAL_REQUIRE(aligned16(lstm_c) && aligned16(lstm_h) && aligned16(fc_tab_bf16) && aligned16(xh_bf16),
                 "unreal_maze_eval_act: LSTM state, table and operand must be 16-byte aligned");
  if (n == 0) return UNREAL_OK;
  const MazeLayout L = maze_layout_host();
  EvalState S{pos, last_action, last_reward, ep_score, ep_length, ep_index, active, res_score, res_length, res_finished,
              n, episodes, max_steps};
  EvalRows R{lstm_c, lstm_h, reinterpret_cast<const __nv_bfloat16*>(fc_tab_bf16), reinterpret_cast<__nv_bfloat16*>(xh_bf16),
             ld_xh, kx};
  const unsigned grid = (unsigned)((n + kEvalEnvs - 1) / kEvalEnvs);
  cudaStream_t st = as_stream(stream);
  switch (a) {   // the common action counts with the choice loops unrolled (the cdf stays in registers)
    case 3: maze_eval_act_kernel<3><<<grid, kEvalThreads, 0, st>>>(S, L, R, pi, a, greedy, mt, mt_pos); break;
    case 4: maze_eval_act_kernel<4><<<grid, kEvalThreads, 0, st>>>(S, L, R, pi, a, greedy, mt, mt_pos); break;
    default: maze_eval_act_kernel<0><<<grid, kEvalThreads, 0, st>>>(S, L, R, pi, a, greedy, mt, mt_pos); break;
  }
  UNREAL_LAUNCH_CHECK("maze_eval_act_kernel");
  return UNREAL_OK;
}
