"""numpy restatement of the evaluator's per-env rules (unreal_b200/train/evaluator.py, csrc/eval_core.cuh) on the oracle
maze, for the CPU harness test and the GPU kernel test: state-independent pi rows in, every step's action / transition /
episode accounting out."""
import numpy as np

from oracle import unreal_oracle as O


def optimal_path(map49=O.MAZE_MAP):
  """Shortest action sequence from S to G (breadth-first search over the oracle's maze_step)."""
  walls, start, goal = O.maze_layout(map49)
  prev = {start: None}
  queue = [start]
  while queue:
    cur = queue.pop(0)
    if cur == goal:
      break
    for act in range(4):
      nx, ny, _, _ = O.maze_step(cur[0], cur[1], act, walls, goal)
      if (nx, ny) not in prev:
        prev[(nx, ny)] = (cur, act)
        queue.append((nx, ny))
  path, cur = [], goal
  while prev[cur] is not None:
    cur, act = prev[cur]
    path.append(act)
  return path[::-1]


def restate(map49, seeds, pi, episodes, cap, greedy, kl=None):
  """pi [steps, m, a] -> dict(log [steps,m,8] i32 (stepped, action, reward, terminal, x, y, done, episode index after
  the step), lar [steps,m,kl] f32 (the next step's one-hot(last action) ++ [last reward], zero padded; zero for envs
  that did not step), score / length / finished [m, episodes], streams (the RandomState objects after the run))."""
  walls, start, goal = O.maze_layout(map49)
  steps, m, a = pi.shape
  kl = a + 1 if kl is None else kl
  rs = [np.random.RandomState(int(s)) for s in seeds]
  x = [start[0]] * m; y = [start[1]] * m
  score = [np.float32(0.0)] * m; length = [0] * m; ep = [0] * m; active = [True] * m
  la = [0] * m; lr = [0] * m
  log = np.zeros((steps, m, 8), np.int32)
  lar = np.zeros((steps, m, kl), np.float32)
  res_s = np.zeros((m, episodes), np.float32); res_l = np.zeros((m, episodes), np.int32)
  res_f = np.zeros((m, episodes), np.uint8)
  for t in range(steps):
    for e in range(m):
      if not active[e]:
        log[t, e, 7] = ep[e]
        continue
      act = int(np.argmax(pi[t, e])) if greedy else int(rs[e].choice(a, p=pi[t, e]))
      nx, ny, r, term = O.maze_step(x[e], y[e], act, walls, goal)
      score[e] = np.float32(score[e] + np.float32(r))
      length[e] += 1
      done = bool(term) or length[e] >= cap
      if done:
        k = ep[e]
        res_s[e, k] = score[e]; res_l[e, k] = length[e]; res_f[e, k] = 1 if term else 0
        ep[e] = k + 1
        active[e] = ep[e] < episodes
        x[e], y[e] = start
        la[e], lr[e] = 0, 0
        score[e] = np.float32(0.0); length[e] = 0
      else:
        x[e], y[e] = nx, ny
        la[e], lr[e] = act, r
      log[t, e] = (1, act, r, 1 if term else 0, x[e], y[e], 1 if done else 0, ep[e])
      lar[t, e, :a + 1] = O.concat_action_and_reward(la[e], a, lr[e])
  return dict(log=log, lar=lar, score=res_s, length=res_l, finished=res_f, streams=rs)


def random_pi(rs, steps, m, a, ties=False):
  """Random policy rows (f32, rows sum to 1); `ties`: values from a few levels so that rows often have equal maxima."""
  p = rs.randint(0, 3, size=(steps, m, a)).astype(np.float32) + 1 if ties else rs.rand(steps, m, a).astype(np.float32) + 0.05
  return (p / p.sum(-1, keepdims=True)).astype(np.float32)


def one_hot_pi(actions, m, a):
  """pi rows one-hot on actions[t] for every env: [len(actions), m, a]."""
  p = np.zeros((len(actions), m, a), np.float32)
  p[np.arange(len(actions)), :, np.asarray(actions)] = 1.0
  return p
