// Per-env logic of the evaluator's fused maze step (unreal_maze_eval_act), host+device so the CPU test harness can
// drive it.  For one active env and one step of Evaluator.run (unreal_b200/train/evaluator.py):
//   action   RandomState.choice(A, p=pi) on the env's own stream (trainer.py:147-148) or argmax(pi), lowest index on ties
//   step     the maze transition of maze_environment.py:98-128 (maze_step_core)
//   episode  score += reward, length += 1; the episode ends at a terminal or at `cap` steps: its [env, episode] result
//            row is written and the env is reset as after a terminal (trainer.py:201-202, :279-296; reset() :50-55),
//            last action / reward 0; after its last episode the env becomes inactive (no step, no draw from then on).
#pragma once
#include "common.cuh"
#include "maze_core.cuh"
#include "mt19937_core.cuh"

namespace unreal {

// Per-env evaluation state, SoA over M envs; results [M, episodes] row-major.
struct EvalState {
  int32_t* pos;          // [M,2] cell x, y
  int32_t* last_action;  // [M]
  float* last_reward;    // [M]
  float* score;          // [M] score of the running episode
  int32_t* length;       // [M] steps of the running episode
  int32_t* episode;      // [M] index of the running episode
  uint8_t* active;       // [M] 0 once the env has played all its episodes
  float* res_score;      // [M, episodes]
  int32_t* res_length;   // [M, episodes]
  uint8_t* res_finished; // [M, episodes] 1: the episode ended at a terminal (the goal), 0: at the step cap
  int m, episodes, cap;
};

struct EvalOut {
  int stepped;      // 0: the env was inactive, nothing was read, drawn or written
  int done;         // the episode ended in this step (the env was reset; its LSTM state must be zeroed)
  int action;
  int reward;       // of the transition (+1 goal, -1 hit, 0)
  int terminal;
  int x, y;         // the env's cell after the step (the start cell after a reset)
  int last_action;  // the next step's one-hot(last action) ++ [last reward]
  int last_reward;
};

// argmax(pi) with the lowest index on ties (numpy / torch argmax) or RandomState.choice(A, p=pi) (two words).
UNREAL_HD int eval_pick(const float* pi, int a, int greedy, MtStream s) {
  if (greedy) {
    int k = 0;
    float best = pi[0];
    for (int i = 1; i < a; ++i)
      if (pi[i] > best) { best = pi[i]; k = i; }
    return k;
  }
  return mt_choice(s, pi, a);
}

UNREAL_HD EvalOut eval_env_step(const EvalState& S, const MazeLayout& L, int e, const float* pi, int a, int greedy,
                                MtStream s) {
  EvalOut o;
  o.stepped = 0; o.done = 0; o.action = 0; o.reward = 0; o.terminal = 0; o.x = 0; o.y = 0; o.last_action = 0; o.last_reward = 0;
  if (S.active[e] == 0) return o;
  o.stepped = 1;
  const int act = eval_pick(pi, a, greedy, s);
  const MazeStep st = maze_step_core(L, S.pos[2 * e], S.pos[2 * e + 1], act);
  float sc = S.score[e] + (float)st.reward;
  int len = S.length[e] + 1;
  o.action = act; o.reward = st.reward; o.terminal = st.terminal;
  if (st.terminal || len >= S.cap) {
    const int k = S.episode[e];
    const int64_t r = (int64_t)e * S.episodes + k;
    S.res_score[r] = sc;
    S.res_length[r] = len;
    S.res_finished[r] = (uint8_t)(st.terminal ? 1 : 0);
    S.episode[e] = k + 1;
    if (k + 1 >= S.episodes) S.active[e] = 0;
    o.done = 1;
    o.x = L.start_x; o.y = L.start_y;
    sc = 0.f; len = 0;
  } else {
    o.x = st.x1; o.y = st.y1;
    o.last_action = act; o.last_reward = st.reward;
  }
  S.pos[2 * e] = o.x; S.pos[2 * e + 1] = o.y;
  S.last_action[e] = o.last_action;
  S.last_reward[e] = (float)o.last_reward;
  S.score[e] = sc;
  S.length[e] = len;
  return o;
}

// Column j of the last-action / reward block of the LSTM input (ExperienceFrame.concat_action_and_reward,
// experience.py:34-46, objective size 0), j in [0, kx - 256): one-hot(last_action, a) ++ [last_reward], zero padding.
UNREAL_HD float eval_lar_col(int j, int a, int last_action, int last_reward) {
  if (j < a) return j == last_action ? 1.f : 0.f;
  return j == a ? (float)last_reward : 0.f;
}

// Row of the 49-entry cell table for a cell (as unreal_cell_gather: clamped to the grid).
UNREAL_HD int eval_cell_index(int x, int y) {
  x = x < 0 ? 0 : (x > UNREAL_MAZE_GRID - 1 ? UNREAL_MAZE_GRID - 1 : x);
  y = y < 0 ? 0 : (y > UNREAL_MAZE_GRID - 1 ? UNREAL_MAZE_GRID - 1 : y);
  return y * UNREAL_MAZE_GRID + x;
}

}  // namespace unreal
