// TEST INFRASTRUCTURE, not a product path: compiles unreal_b200/csrc/eval_core.cuh (the per-env logic of the evaluator's
// fused maze step, unreal_maze_eval_act) with plain g++ and drives it with caller-supplied pi rows, so the step can be
// checked against a numpy restatement on a machine without a GPU.  Nothing in the package loads this library.
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../../unreal_b200/csrc/eval_core.cuh"

using namespace unreal;

static MazeLayout parse_layout(const char* m) {
  MazeLayout L;
  memset(&L, 0, sizeof(L));
  for (int i = 0; i < 49; ++i) {
    int x = i % 7, y = i / 7;
    if (m[i] == '+') L.wall_rows[y] |= 1u << x;
    if (m[i] == 'S') { L.start_x = x; L.start_y = y; }
    if (m[i] == 'G') { L.goal_x = x; L.goal_y = y; }
  }
  return L;
}

extern "C" {

// `steps` evaluation steps of m envs on the 49-character map `map49`, every env starting a fresh episode.
//   pi [steps, m, a] f32: the policy rows fed at each step (independent of the state)
//   log [steps, m, 8] i32: stepped, action, reward, terminal, x, y, done, episode index after the step
//   lar [steps, m, kl] f32: the last-action / reward columns written for the next step (stepped envs only, else 0)
//   res_* [m, episodes]; mt_out [624, m] u32 and mt_pos_out [m]: the streams after the run
void h_eval_run(const char* map49, int m, int a, int episodes, int cap, int greedy, const uint32_t* seeds,
                const float* pi, int steps, int32_t* log, float* lar, int kl, float* res_score, int32_t* res_length,
                uint8_t* res_finished, uint32_t* mt_out, int32_t* mt_pos_out) {
  const MazeLayout L = parse_layout(map49);
  std::vector<int32_t> pos(2 * m), la(m, 0), len(m, 0), ep(m, 0);
  std::vector<float> lr(m, 0.f), score(m, 0.f);
  std::vector<uint8_t> active(m, 1);
  for (int e = 0; e < m; ++e) { pos[2 * e] = L.start_x; pos[2 * e + 1] = L.start_y; }
  for (int e = 0; e < m; ++e) {
    MtStream s{mt_out + e, (int64_t)m, mt_pos_out + e};
    mt_seed_core(s, seeds[e]);
  }
  EvalState S{pos.data(), la.data(), lr.data(), score.data(), len.data(), ep.data(), active.data(), res_score, res_length,
              res_finished, m, episodes, cap};
  for (int t = 0; t < steps; ++t) {
    for (int e = 0; e < m; ++e) {
      MtStream s{mt_out + e, (int64_t)m, mt_pos_out + e};
      const EvalOut o = eval_env_step(S, L, e, pi + ((int64_t)t * m + e) * a, a, greedy, s);
      int32_t* q = log + ((int64_t)t * m + e) * 8;
      q[0] = o.stepped; q[1] = o.action; q[2] = o.reward; q[3] = o.terminal; q[4] = o.x; q[5] = o.y; q[6] = o.done;
      q[7] = ep[e];
      float* l = lar + ((int64_t)t * m + e) * kl;
      for (int j = 0; j < kl; ++j) l[j] = o.stepped ? eval_lar_col(j, a, o.last_action, o.last_reward) : 0.f;
      if (o.stepped && eval_cell_index(o.x, o.y) != o.y * 7 + o.x) q[0] = -1;   // a cell off the grid: flagged
    }
  }
}

}  // extern "C"
