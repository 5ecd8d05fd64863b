"""unreal_maze_rollout_targets (R, advantages and PC targets of a maze pass from its frame records) against the two
kernels it stands in for, unreal_nstep_returns on the pass's rewards / terminals and unreal_pc_targets on its
pixel-change maps: bit for bit, on K1's own outputs at the benchmark's size, on scripted episodes whose terminals fall
at the first and the last step, on invalid records, and with sentinel bands around every output."""
from collections import deque

import numpy as np
import pytest
import torch

from oracle import unreal_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GAMMA, GAMMA_PC = 0.99, 0.9


@pytest.fixture(scope="module")
def K():
  from unreal_b200 import kernels, _lib
  _lib.require_device()
  return kernels


def _two_kernels(K, reward, terminal, pc, values, boot, boot_q):
  R, adv = K.nstep_returns(reward, values, terminal, boot, GAMMA)
  return R, adv, K.pc_targets(pc, terminal, None, boot_q, GAMMA_PC)


def _assert_equal(got, want):
  for name, g, w in zip(("R", "adv", "pc_tgt"), got, want):
    assert torch.equal(g, w), "%s differs" % name


@pytest.mark.parametrize("window", [False, True], ids=["k1-per-step", "k1-window"])
def test_equals_returns_and_pc_targets_on_the_benched_pass(K, window):
  """RolloutTargets at 4096 x 20 with f32 frames: its targets launch against the two kernels on the same K1 outputs."""
  from unreal_b200.train.rollout import RolloutTargets
  n, t = 4096, 20
  eng = RolloutTargets(n, t, GAMMA, GAMMA_PC, torch.float32, torch.device(DEV), auto_reset=True, use_graphs=True,
                       window_kernel=window)
  g = torch.Generator(device=DEV).manual_seed(7)
  for _ in range(2):
    eng.actions.copy_(torch.randint(0, 4, (t, n), device=DEV, dtype=torch.int32, generator=g))
    eng.values.copy_(torch.randn(t, n, device=DEV, generator=g))
    eng.boot_value.copy_(torch.randn(n, device=DEV, generator=g))
    eng.boot_q.copy_(torch.rand(n, 20, 20, device=DEV, generator=g))
    eng.run_device()
    want = _two_kernels(K, eng.reward, eng.terminal, eng.pc, eng.values, eng.boot_value, eng.boot_q)
    _assert_equal((eng.R, eng.adv, eng.pc_tgt), want)


def _distances_to_goal():
  """BFS distance of every reachable cell to the goal, and the first action of a shortest path from it."""
  dist, step = {O.GOAL: 0}, {}
  dq = deque([O.GOAL])
  while dq:
    c = dq.popleft()
    for y in range(7):
      for x in range(7):
        if (x, y) in dist or O.WALLS[y, x]:
          continue
        for a in range(4):
          nx, ny, hit = O.maze_move(x, y, a)
          if not hit and (nx, ny) == c:
            dist[(x, y)] = dist[c] + 1
            step[(x, y)] = a
            dq.append((x, y))
            break
  return dist, step


def _scripted(T, N, rs):
  """Start cells and [T,N] actions: a third of the envs reach the goal at step 0, a third at step T-1 (walking a
  shortest path, through an auto-reset when T exceeds the start cell's 20 moves), the rest move at random."""
  dist, step = _distances_to_goal()
  by_dist = {}
  for c, d in dist.items():
    by_dist.setdefault(d, []).append(c)
  d_last = T if T in by_dist else T - dist[O.START]
  assert d_last in by_dist, T
  starts = np.zeros((N, 2), np.int32)
  actions = rs.randint(0, 4, size=(T, N)).astype(np.int32)
  for e in range(N):
    kind = e % 3
    cells = by_dist[1] if kind == 0 else (by_dist[d_last] if kind == 1 else [O.START])
    c = cells[rs.randint(len(cells))]
    starts[e] = c
    for s in range(T):
      if kind == 1 or (kind == 0 and s == 0):
        actions[s, e] = step[c]
      nx, ny, _, term = O.maze_step(c[0], c[1], int(actions[s, e]))
      c = O.START if term else (nx, ny)
  return starts, actions


@pytest.mark.parametrize("T", [1, 7, 32])
@pytest.mark.parametrize("N", [1, 67, 1000])
def test_equals_returns_and_pc_targets_on_scripted_episodes(K, T, N):
  rs = np.random.RandomState(T * 1000 + N)
  starts, actions = _scripted(T, N, rs)
  st = K.MazeState(N, DEV)
  st.pos.copy_(torch.from_numpy(starts))
  pc = torch.empty(T, N, 20, 20, device=DEV)
  rec = torch.empty(T, N, dtype=torch.int64, device=DEV)
  reward, terminal = K.maze_window(st, torch.from_numpy(actions).to(DEV), pc=pc, frame_rec=rec, auto_reset=True)
  term = terminal.cpu().numpy()
  assert term[0, ::3].all() and term[T - 1, 1::3].all()
  values = torch.from_numpy(rs.randn(T, N).astype(np.float32)).to(DEV)
  boot = torch.from_numpy(rs.randn(N).astype(np.float32)).to(DEV)
  boot_q = torch.from_numpy(rs.rand(N, 20, 20).astype(np.float32)).to(DEV)
  got = K.maze_rollout_targets(rec, values, boot, boot_q, GAMMA, GAMMA_PC)
  _assert_equal(got, _two_kernels(K, reward, terminal, pc, values, boot, boot_q))


@pytest.mark.parametrize("T,N", [(1, 1), (7, 67), (32, 1000)])
def test_invalid_records_are_reward_0_not_terminal_map_0(K, T, N):
  rs = np.random.RandomState(N)
  values = torch.from_numpy(rs.randn(T, N).astype(np.float32)).to(DEV)
  boot = torch.from_numpy(rs.randn(N).astype(np.float32)).to(DEV)
  boot_q = torch.from_numpy(rs.rand(N, 20, 20).astype(np.float32)).to(DEV)
  want = _two_kernels(K, torch.zeros(T, N, device=DEV), torch.zeros(T, N, dtype=torch.uint8, device=DEV),
                      torch.zeros(T, N, 20, 20, device=DEV), values, boot, boot_q)
  zeros = torch.zeros(T, N, dtype=torch.int64, device=DEV)
  junk = rs.randint(0, 2 ** 62, size=(T, N), dtype=np.int64) & ~np.int64(1 << 39)   # every field set, valid bit 0
  for rec in (zeros, torch.from_numpy(junk).to(DEV)):
    _assert_equal(K.maze_rollout_targets(rec, values, boot, boot_q, GAMMA, GAMMA_PC), want)


PAD = 4096      # bytes of sentinel on each side (a multiple of 16: the views stay 16-byte aligned)


class Guarded(object):
  def __init__(self, shape, dtype):
    self.n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
    body = (self.n + 15) // 16 * 16
    self.raw = torch.full((PAD + body + PAD,), 0xA5, dtype=torch.uint8, device=DEV)
    self.t = self.raw[PAD:PAD + self.n].view(dtype).view(*shape)

  def ok(self):
    return bool((self.raw[:PAD] == 0xA5).all()) and bool((self.raw[PAD + self.n:] == 0xA5).all())


@pytest.mark.parametrize("T,N", [(1, 1), (7, 67), (13, 129), (32, 1000)])
def test_rollout_targets_write_stay_inside(K, T, N):
  rs = np.random.RandomState(3)
  st = K.MazeState(N, DEV)
  rec = torch.empty(T, N, dtype=torch.int64, device=DEV)
  K.maze_window(st, torch.from_numpy(rs.randint(0, 4, size=(T, N)).astype(np.int32)).to(DEV), frame_rec=rec,
                auto_reset=True)
  values = torch.randn(T, N, device=DEV)
  R, adv, tgt = Guarded((T, N), torch.float32), Guarded((T, N), torch.float32), Guarded((T, N, 20, 20), torch.float32)
  K.maze_rollout_targets(rec, values, torch.randn(N, device=DEV), torch.rand(N, 20, 20, device=DEV), GAMMA, GAMMA_PC,
                         R=R.t, adv=adv.t, pc_tgt=tgt.t)
  torch.cuda.synchronize()
  for name, g in (("R", R), ("adv", adv), ("pc_tgt", tgt)):
    assert g.ok(), "%s was written outside its bounds" % name
