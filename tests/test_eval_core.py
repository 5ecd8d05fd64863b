"""CPU checks of csrc/eval_core.cuh, the per-env logic of the evaluator's fused maze step (unreal_maze_eval_act),
compiled with g++ (tests/cpu_harness/eval_harness.cpp) and driven with state-independent pi rows against the numpy
restatement on the oracle maze (tests/eval_restatement.py): actions, cells, rewards, result rows, the written
last-action / reward columns and the MT19937 stream positions must be bit-equal."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import unreal_oracle as O
import eval_restatement as R

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "cpu_harness", "eval_harness.cpp")
CUDA_INC = "/usr/local/cuda/include"
OPEN_MAP = "S-----+" "-+-+---" "---G-+-" "-+-----" "----+--" "--+----" "-------"   # many short paths to the goal
KL = 8            # last-action / reward columns of a 4-action model: kx - 256 = 264 - 256


@pytest.fixture(scope="module")
def H(tmp_path_factory):
  if shutil.which("g++") is None or not os.path.exists(os.path.join(CUDA_INC, "cuda_runtime.h")):
    pytest.skip("g++ or CUDA headers not available")
  out = str(tmp_path_factory.mktemp("eval_harness") / "libeval_harness.so")
  subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", CUDA_INC, SRC, "-o", out])
  return ctypes.CDLL(out)


def _p(a):
  return a.ctypes.data_as(ctypes.c_void_p)


def run_harness(H, map49, seeds, pi, episodes, cap, greedy):
  steps, m, a = pi.shape
  pi = np.ascontiguousarray(pi, np.float32)
  seeds = np.asarray(seeds, np.uint32)
  log = np.zeros((steps, m, 8), np.int32)
  lar = np.zeros((steps, m, KL), np.float32)
  rs_ = np.zeros((m, episodes), np.float32); rl = np.zeros((m, episodes), np.int32); rf = np.zeros((m, episodes), np.uint8)
  mt = np.zeros((624, m), np.uint32); pos = np.zeros(m, np.int32)
  H.h_eval_run(map49.encode(), m, a, episodes, cap, 1 if greedy else 0, _p(seeds), _p(pi), steps, _p(log), _p(lar), KL,
               _p(rs_), _p(rl), _p(rf), _p(mt), _p(pos))
  return dict(log=log, lar=lar, score=rs_, length=rl, finished=rf, mt=mt, pos=pos)


def check_equal(got, want, greedy):
  assert np.array_equal(got["log"], want["log"])
  assert np.array_equal(got["lar"], want["lar"])
  for k in ("score", "length", "finished"):
    assert np.array_equal(got[k], want[k]), k
  for e, rs in enumerate(want["streams"]):
    _, key, pos, _, _ = rs.get_state()
    assert int(got["pos"][e]) == int(pos)
    if greedy:
      assert int(pos) == 624           # seeded, never drawn from
    assert np.array_equal(got["mt"][:, e], key)


@pytest.mark.parametrize("map49", [O.MAZE_MAP, OPEN_MAP], ids=["reference_map", "open_map"])
@pytest.mark.parametrize("greedy", [False, True], ids=["sample", "greedy"])
@pytest.mark.parametrize("cap", [7, 60, 900])
def test_eval_core_matches_restatement(H, map49, greedy, cap):
  m, a, episodes = 5, 4, 3
  steps = min(3 * cap + 40, 3000)
  gen = np.random.RandomState(cap + 7 * greedy)
  pi = R.random_pi(gen, steps, m, a, ties=greedy)
  seeds = [11, 0, 2 ** 32 - 1, 5, 1234567]
  got = run_harness(H, map49, seeds, pi, episodes, cap, greedy)
  want = R.restate(map49, seeds, pi, episodes, cap, greedy, kl=KL)
  check_equal(got, want, greedy)
  stepped = got["log"][..., 0]
  assert stepped.min() >= 0                       # every written cell is on the grid
  if steps > 3 * cap:                             # every env played its episodes, then went quiet: no step, no draw
    assert stepped[-1].sum() == 0 and (got["log"][-1, :, 7] == episodes).all()
  if map49 == OPEN_MAP and cap >= 60:
    assert got["finished"].sum() > 0                # goals reached: the terminal branch is covered too


def test_greedy_ties_take_the_lowest_index(H):
  m, a = 3, 4
  pi = np.full((6, m, a), 0.25, np.float32)      # all four tied: UP every step
  pi[:, 1] = [0.1, 0.4, 0.1, 0.4]                # DOWN and RIGHT tied: DOWN
  pi[:, 2] = [0.2, 0.2, 0.3, 0.3]                # LEFT and RIGHT tied: LEFT
  got = run_harness(H, O.MAZE_MAP, [1, 2, 3], pi, 1, 100, True)
  assert (got["log"][:, 0, 1] == 0).all() and (got["log"][:, 1, 1] == 1).all() and (got["log"][:, 2, 1] == 2).all()
  check_equal(got, R.restate(O.MAZE_MAP, [1, 2, 3], pi, 1, 100, True, kl=KL), True)


@pytest.mark.parametrize("greedy", [False, True], ids=["sample", "greedy"])
def test_cap_at_the_terminal_step(H, greedy):
  """The optimal path reaches the goal on its last move: with the cap equal to its length the episode is finished
  (a terminal wins over the cap); one step shorter, it is capped at score 0 and not finished."""
  path = R.optimal_path()
  assert len(path) == 20
  m, a = 2, 4
  pi = R.one_hot_pi(path * 2 + path[:5], m, a)
  for cap, fin in ((len(path), 1), (len(path) - 1, 0)):
    got = run_harness(H, O.MAZE_MAP, [3, 4], pi, 2, cap, greedy)
    want = R.restate(O.MAZE_MAP, [3, 4], pi, 2, cap, greedy, kl=KL)
    check_equal(got, want, greedy)
    assert (got["finished"] == fin).all() and (got["length"] == cap).all()
    if fin:
      assert (got["score"] == 1.0).all()


def test_inactive_envs_draw_nothing(H):
  """An env that has played its episodes takes no step and no draw: its stream stays where its last episode left it."""
  m, a, cap = 4, 4, 5
  pi = R.random_pi(np.random.RandomState(3), 200, m, a)
  got = run_harness(H, O.MAZE_MAP, [9, 8, 7, 6], pi, 2, cap, False)
  assert got["log"][2 * cap:, :, 0].sum() == 0
  for e in range(m):
    rs = np.random.RandomState([9, 8, 7, 6][e])
    for t in range(2 * cap):
      rs.choice(a, p=pi[t, e])
    assert int(got["pos"][e]) == rs.get_state()[2] and np.array_equal(got["mt"][:, e], rs.get_state()[1])
