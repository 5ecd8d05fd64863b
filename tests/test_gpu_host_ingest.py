"""Host simulators on worker threads + unreal_host_frames_ingest (one launch per env step, frames read from pinned
staging) against the composition it replaces: rows_select of HostEnvProducer._u8-converted frames, K2, frame_pack and
the adapter's torch.where updates -- bit-equal on every output row."""
import threading

import numpy as np
import pytest
import torch

from oracle import unreal_oracle as O
from fake_net import FakeNet
from test_gpu_frames import _EndAwareNet, _close, _u8

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _pinned(a):
  return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()


def _guarded(shape, dtype, pad=64):
  """A device buffer inside NaN (floats) / 0xAB (integers) guard bands: (view, whole buffer, pristine copy)."""
  n = int(np.prod(shape))
  whole = torch.empty(n + 2 * pad, dtype=dtype, device=DEV)
  if dtype.is_floating_point:
    whole.fill_(float("nan"))
  else:
    whole.view(torch.uint8).fill_(0xAB)
  return whole[pad:pad + n].view(*shape), whole, pad


def _bands_intact(whole, pad):
  w = whole.view(torch.uint8) if not whole.dtype.is_floating_point else whole
  k = pad * (1 if whole.dtype.is_floating_point else whole.element_size())
  for band in (w[:k], w[-k:]):
    if whole.dtype.is_floating_point:
      assert torch.isnan(band).all()
    else:
      assert (band == 0xAB).all()


def _frames(rs, n, shape, f32):
  u = rs.randint(0, 256, size=(n,) + shape).astype(np.uint8)
  if not f32:
    return u
  f = u.astype(np.float32) / np.float32(255.0)
  odd = rs.rand(n, *shape).astype(np.float32)            # values between the k/255 grid points as well
  pick = rs.rand(n, *shape) < 0.3
  return np.where(pick, odd, f).astype(np.float32)


def _old_composition(st, action, active, prev, out, own, last_action, last_reward, objective):
  """BatchedFrameEnvironment.process over the per-step HostEnvProducer it replaces (rows_select of the _u8-converted
  staging, K2, frame_pack, reset of the terminal envs, torch.where updates)."""
  from unreal_b200 import kernels as K
  from unreal_b200.environment.frame_environment import HostEnvProducer as HP
  n = out.shape[0]
  m = torch.ones(n, dtype=torch.uint8, device=DEV) if active is None else active
  mh = m.cpu().numpy().astype(bool)
  if own:
    out.copy_(prev)
  stage = np.zeros(out.shape, np.uint8)
  for e in np.flatnonzero(mh):
    stage[e] = HP._u8(st["step_frames"][e])
  K.rows_select(out, torch.from_numpy(stage).to(DEV), None, m)
  reward = torch.from_numpy(np.where(mh, st["reward"], 0).astype(np.float32)).to(DEV)
  terminal = torch.from_numpy(np.where(mh, st["terminal"], 0).astype(np.uint8)).to(DEV)
  g = 0 if objective is None else objective.shape[1]
  if g:
    objective.copy_(torch.where(m.bool()[:, None], torch.from_numpy(st["step_obj"]).to(DEV), objective))
  pc = K.pixel_change(out, prev)
  rec = K.frame_pack(action, reward, terminal, last_action, last_reward, active)
  term = terminal & m
  th = term.cpu().numpy().astype(bool)
  stage2 = np.zeros(out.shape, np.uint8)
  for e in np.flatnonzero(th):
    stage2[e] = HP._u8(st["reset_frames"][e])
  K.rows_select(out, torch.from_numpy(stage2).to(DEV), None, term)
  if g:
    objective.copy_(torch.where(term.bool()[:, None], torch.from_numpy(st["reset_obj"]).to(DEV), objective))
  act_m, ended = m.bool(), term.bool()
  last_action.copy_(torch.where(act_m, torch.where(ended, torch.zeros_like(last_action), action), last_action))
  last_reward.copy_(torch.where(act_m, torch.where(ended, torch.zeros_like(last_reward), reward), last_reward))
  return pc, rec, reward, terminal


@pytest.mark.parametrize("f32", [False, True])
@pytest.mark.parametrize("n", [1, 3, 257, 1024])
@pytest.mark.parametrize("hw", [(84, 84), (40, 40)])
@pytest.mark.parametrize("g", [0, 2])
@pytest.mark.parametrize("own", [True, False])
def test_ingest_step_equals_the_old_composition(f32, n, hw, g, own):
  from unreal_b200 import kernels as K
  rs = np.random.RandomState(n * 7 + hw[0] + g + 2 * own + f32)
  shape = hw + (3,)
  ph, pw = (hw[0] - 4) // 4, (hw[1] - 4) // 4
  for case in ("random", "inactive", "all_terminal", "none"):
    st = dict(step_frames=_frames(rs, n, shape, f32), reset_frames=_frames(rs, n, shape, f32),
              reward=(rs.randint(-2, 3, size=n) * 0.5).astype(np.float32),
              terminal=(rs.rand(n) < 0.3).astype(np.uint8),
              step_obj=rs.randn(n, max(1, g)).astype(np.float32), reset_obj=rs.randn(n, max(1, g)).astype(np.float32))
    if case == "all_terminal":
      st["terminal"][:] = 1
    active = {"random": (rs.rand(n) < 0.7), "inactive": np.zeros(n, bool), "all_terminal": np.ones(n, bool),
              "none": None}[case]
    active = None if active is None else torch.from_numpy(active.astype(np.uint8)).to(DEV)
    action = torch.from_numpy(rs.randint(0, 3, size=n).astype(np.int32)).to(DEV)
    prev = torch.from_numpy(rs.randint(0, 256, size=(n,) + shape).astype(np.uint8)).to(DEV)
    out0 = torch.from_numpy(rs.randint(0, 256, size=(n,) + shape).astype(np.uint8)).to(DEV)
    la0 = torch.from_numpy(rs.randint(0, 3, size=n).astype(np.int32)).to(DEV)
    lr0 = torch.from_numpy((rs.randint(-2, 3, size=n) * 0.5).astype(np.float32)).to(DEV)
    obj0 = torch.from_numpy(rs.randn(n, g).astype(np.float32)).to(DEV) if g else None

    want_out, want_la, want_lr = out0.clone(), la0.clone(), lr0.clone()
    want_obj = obj0.clone() if g else None
    w_pc, w_rec, w_rew, w_term = _old_composition(st, action, active, prev, want_out, own, want_la, want_lr, want_obj)

    out, out_w, out_p = _guarded((n,) + shape, torch.uint8)
    out.copy_(out0)
    pc, pc_w, pc_p = _guarded((n, ph, pw), torch.float32)
    rec, rec_w, rec_p = _guarded((n,), torch.int64)
    rew, rew_w, rew_p = _guarded((n,), torch.float32)
    term, term_w, term_p = _guarded((n,), torch.uint8)
    la, la_w, la_p = _guarded((n,), torch.int32)
    la.copy_(la0)
    lr, lr_w, lr_p = _guarded((n,), torch.float32)
    lr.copy_(lr0)
    obj = obj_w = None
    if g:
      obj, obj_w, obj_p = _guarded((n, g), torch.float32)
      obj.copy_(obj0)
    K.host_frames_ingest(_pinned(st["reset_frames"]), out, step_frames=_pinned(st["step_frames"]),
                         step_reward=_pinned(st["reward"]), step_terminal=_pinned(st["terminal"]),
                         step_objective=_pinned(st["step_obj"]), reset_objective=_pinned(st["reset_obj"]),
                         action=action, active=active, prev=prev, copy_inactive=own, pc=pc, rec=rec, reward=rew,
                         terminal=term, last_action=la, last_reward=lr, objective=obj)
    torch.cuda.synchronize()
    assert torch.equal(out, want_out), case
    assert torch.equal(pc.view(torch.int32), w_pc.view(torch.int32)), case     # every row, bit for bit
    assert torch.equal(rec, w_rec) and torch.equal(rew, w_rew) and torch.equal(term, w_term), case
    assert torch.equal(la, want_la) and torch.equal(lr.view(torch.int32), want_lr.view(torch.int32)), case
    if g:
      assert torch.equal(obj, want_obj), case
    for whole, pad in ((out_w, out_p), (pc_w, pc_p), (rec_w, rec_p), (rew_w, rew_p), (term_w, term_p), (la_w, la_p),
                       (lr_w, lr_p)) + (((obj_w, obj_p),) if g else ()):
      _bands_intact(whole, pad)


@pytest.mark.parametrize("f32", [False, True])
@pytest.mark.parametrize("g", [0, 2])
def test_ingest_reset_mode(f32, g):
  from unreal_b200 import kernels as K
  from unreal_b200.environment.frame_environment import HostEnvProducer as HP
  n, shape = 257, (40, 40, 3)
  rs = np.random.RandomState(3 + g + f32)
  frames = _frames(rs, n, shape, f32)
  robj = rs.randn(n, max(1, g)).astype(np.float32)
  for mask in (torch.from_numpy((rs.rand(n) < 0.5).astype(np.uint8)).to(DEV), None):
    out0 = torch.from_numpy(rs.randint(0, 256, size=(n,) + shape).astype(np.uint8)).to(DEV)
    out, out_w, out_p = _guarded((n,) + shape, torch.uint8)
    out.copy_(out0)
    la, la_w, la_p = _guarded((n,), torch.int32)
    la.fill_(2)
    lr, lr_w, lr_p = _guarded((n,), torch.float32)
    lr.fill_(0.5)
    obj = None
    if g:
      obj, obj_w, obj_p = _guarded((n, g), torch.float32)
      obj.fill_(7.0)
    K.host_frames_ingest(_pinned(frames), out, reset_objective=_pinned(robj), active=mask, last_action=la,
                         last_reward=lr, objective=obj)
    torch.cuda.synchronize()
    m = np.ones(n, bool) if mask is None else mask.cpu().numpy().astype(bool)
    want = out0.cpu().numpy()
    for e in np.flatnonzero(m):
      want[e] = HP._u8(frames[e])
    assert np.array_equal(out.cpu().numpy(), want)
    assert np.array_equal(la.cpu().numpy(), np.where(m, 0, 2)) and np.array_equal(lr.cpu().numpy(), np.where(m, 0, 0.5))
    if g:
      assert np.array_equal(obj.cpu().numpy(), np.where(m[:, None], robj, 7.0).astype(np.float32))
      _bands_intact(obj_w, obj_p)
    for whole, pad in ((out_w, out_p), (la_w, la_p), (lr_w, lr_p)):
      _bands_intact(whole, pad)


def test_float_conversion_is_bit_equal_to_the_host_twin():
  """every k/255, the float32 neighbours (+-4 ulps) of every rounding midpoint (k+0.5)/255, 10^6 uniform draws."""
  from unreal_b200 import kernels as K
  from unreal_b200.environment.frame_environment import HostEnvProducer as HP
  k = np.arange(256, dtype=np.float32)
  grid = k / np.float32(255.0)
  mid = ((np.arange(256, dtype=np.float64) + 0.5) / 255.0).astype(np.float32)
  near = [mid]
  for d in range(1, 5):
    up, dn = mid.copy(), mid.copy()
    for _ in range(d):
      up = np.nextafter(up, np.float32(np.inf)); dn = np.nextafter(dn, np.float32(-np.inf))
    near += [up, dn]
  draws = np.random.RandomState(0).rand(10 ** 6).astype(np.float32)
  vals = np.concatenate([grid, np.concatenate(near), draws, np.float32([0.0, 1.0, -0.0])])
  shape = (84, 84, 3)
  per = int(np.prod(shape))
  n = -(-vals.size // per)
  flat = np.zeros(n * per, np.float32)
  flat[:vals.size] = vals
  frames = flat.reshape((n,) + shape)
  out = torch.zeros((n,) + shape, dtype=torch.uint8, device=DEV)
  K.host_frames_ingest(_pinned(frames), out)
  want = HP._u8(frames)
  assert np.array_equal(out.cpu().numpy(), want)


class _ThreadRecorder(object):
  """A TableFrameEnvOracle that records the thread of every call."""

  def __init__(self, env):
    self.env, self.threads = env, set()

  @property
  def last_state(self):
    return self.env.last_state

  def reset(self):
    self.threads.add(threading.get_ident())
    self.env.reset()

  def process(self, action, flag=1):
    self.threads.add(threading.get_ident())
    return self.env.process(action, flag)


@pytest.mark.parametrize("workers", [1, 2, 7])
def test_workers_give_the_device_producer_stream(workers):
  from unreal_b200.environment import frame_environment as FE
  N = 9
  table = FE.TableFrameProducer.make_table(9)
  host_envs = [_ThreadRecorder(O.TableFrameEnvOracle(e, table)) for e in range(N)]
  dev_env = FE.BatchedFrameEnvironment(FE.TableFrameProducer(N, DEV, 3, seed=9), DEV)
  for o in host_envs:
    o.env.counter = 0
  prod = FE.HostEnvProducer(host_envs, DEV, 3, workers=workers)
  assert prod.stage_dtype == torch.float32
  host_env = FE.BatchedFrameEnvironment(prod, DEV)
  rs = np.random.RandomState(1)
  assert torch.equal(dev_env.last_state['image'], host_env.last_state['image'])
  for step in range(60):
    act = torch.from_numpy(rs.randint(0, 3, size=N).astype(np.int32)).to(DEV)
    active = torch.from_numpy((rs.rand(N) < 0.8).astype(np.uint8)).to(DEV)
    a = dev_env.process(act, active=active)
    b = host_env.process(act, active=active)
    m = active.bool()
    assert torch.equal(a[0]['image'], b[0]['image'])
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]) and torch.equal(a[3][m], b[3][m])
    assert torch.equal(dev_env.frame_rec, host_env.frame_rec)
    assert torch.equal(dev_env.last_action, host_env.last_action) and torch.equal(dev_env.last_reward, host_env.last_reward)
  owner = [o.threads for o in host_envs]
  assert all(len(t) == 1 for t in owner), "every env is called from exactly one thread"
  if workers == 1:
    assert owner[0] == {threading.get_ident()}
  else:
    assert len(set.union(*owner)) == workers and threading.get_ident() not in set.union(*owner)
  host_env.stop()


def test_worker_threads_drive_the_trainer():
  """A registered host env type with workers=4: the framed trainer's feeds equal one oracle worker per env."""
  from unreal_b200.environment import frame_environment as FE
  from unreal_b200.environment.environment import Environment
  from unreal_b200.train.trainer import Trainer
  N, H, T = 5, 40, 20
  table = O.make_frame_table(12)
  sims = [O.TableFrameEnvOracle(e, table) for e in range(N)]
  for sim in sims:
    sim.counter = 0
  made = []
  Environment.register('hostsim_mt', lambda name, args, tt, ti: made.append(FE.BatchedFrameEnvironment(
      FE.HostEnvProducer(sims, args['device'], 3, workers=4), args['device'])) or made[-1], action_size=3)
  try:
    Environment.action_size = -1
    seeds = [7 + e for e in range(N)]
    net_seeds = [90 + e for e in range(N)]
    net = _EndAwareNet(net_seeds, DEV, action_size=3)
    tr = Trainer(1, net, 7e-4, None, None, 'hostsim_mt', '', True, True, True, True, 0.05, 1e-3, 20, T, 0.99, 0.9, H,
                 10 ** 7, DEV, {'segnet_mode': 0}, (84, 84), True, 0, np.random.RandomState(0), 50.0, 0.0, 0.0,
                 num_envs=N, seeds=seeds)
    net.attach(tr)
    tr.prepare()
    workers = [O.RolloutOracle(H, np.random.RandomState(s), FakeNet(ns, 3), n_step_TD=T, action_size=3,
                               env=O.TableFrameEnvOracle(e, table)) for e, (s, ns) in enumerate(zip(seeds, net_seeds))]
    while not tr.experience.is_full():
      tr.process(None, 0)
      for w in workers:
        w.fill_step()
    for it in range(4):
      tr.process(None, 0)
      f = tr.last_feed
      for e, w in enumerate(workers):
        b = w.process_base(); p = w.process_pc(); w.process_vr(); r = w.process_rp()
        L = len(b['states'])
        assert int(f['base']['length'][e]) == L
        assert np.array_equal(f['base']['si'][:L, e].cpu().numpy(), np.stack([_u8(s['image']) for s in b['states']]))
        _close(f['base']['R'][:L, e].cpu().numpy(), np.array(b['R'], np.float64))
        Lp = len(p['states'])
        assert int(f['pc']['length'][e]) == Lp
        _close(f['pc']['R'][e, :Lp].cpu().numpy(), np.stack(p['R']).astype(np.float64))
        assert list(f['rp']['c'][e].cpu().numpy()) == r['c']
  finally:
    Environment._registry.pop('hostsim_mt', None)
    Environment.action_size = -1
    for env in made:
      env.stop()


class _FailsAt(object):
  def __init__(self, env, at):
    self.env, self.at, self.calls = env, at, 0

  @property
  def last_state(self):
    return self.env.last_state

  def reset(self):
    self.env.reset()

  def process(self, action, flag=1):
    self.calls += 1
    if self.calls == self.at:
      raise ValueError("simulator died")
    return self.env.process(action, flag)


class _U8Later(_FailsAt):
  def process(self, action, flag=1):
    s, r, t, pc = self.env.process(action, flag)
    return {'image': _u8(s['image'])}, r, t, pc


@pytest.mark.parametrize("workers", [1, 3])
def test_env_errors_name_the_env_and_stop_the_producer(workers):
  from unreal_b200 import _lib
  from unreal_b200.environment import frame_environment as FE
  table = FE.TableFrameProducer.make_table(2)
  envs = [O.TableFrameEnvOracle(e, table) for e in range(6)]
  envs[4] = _FailsAt(envs[4], 5)
  env = FE.BatchedFrameEnvironment(FE.HostEnvProducer(envs, DEV, 3, workers=workers), DEV)
  act = torch.zeros(6, dtype=torch.int32, device=DEV)
  for _ in range(4):
    env.process(act)
  with pytest.raises(_lib.UnrealError, match="env 4") as info:
    env.process(act)
  assert isinstance(info.value.__cause__, ValueError)
  with pytest.raises(_lib.UnrealError):
    env.process(act)
  env.stop()

  envs = [O.TableFrameEnvOracle(e, table) for e in range(3)]
  envs[1] = _U8Later(envs[1], 0)
  env = FE.BatchedFrameEnvironment(FE.HostEnvProducer(envs, DEV, 3, workers=workers), DEV)
  with pytest.raises(_lib.UnrealError, match="env 1") as info:
    env.process(torch.zeros(3, dtype=torch.int32, device=DEV))
  assert "uint8" in str(info.value)
  env.stop()


def test_close_ends_the_threads():
  from unreal_b200.environment import frame_environment as FE
  before = threading.active_count()
  table = FE.TableFrameProducer.make_table(2)
  env = FE.BatchedFrameEnvironment(FE.HostEnvProducer([O.TableFrameEnvOracle(e, table) for e in range(8)], DEV, 3,
                                                      workers=4), DEV)
  assert threading.active_count() == before + 4
  env.process(torch.ones(8, dtype=torch.int32, device=DEV))
  env.stop()
  assert threading.active_count() == before


def test_one_ingest_launch_and_no_upload_per_step():
  from torch.autograd import DeviceType
  from unreal_b200.environment import frame_environment as FE
  N, steps = 16, 20
  table = FE.TableFrameProducer.make_table(4)
  env = FE.BatchedFrameEnvironment(FE.HostEnvProducer([O.TableFrameEnvOracle(e, table) for e in range(N)], DEV, 3,
                                                      workers=4), DEV)
  rs = np.random.RandomState(0)
  acts = torch.from_numpy(rs.randint(0, 3, size=(steps, N)).astype(np.int32)).to(DEV)
  active = torch.from_numpy((rs.rand(steps, N) < 0.8).astype(np.uint8)).to(DEV)
  env.process(acts[0], active=active[0])
  torch.cuda.synchronize()
  # the activity trace can miss records at its very start when a profiler ran earlier in the process: trace two
  # warm-up steps and discard them, then keep exactly the `steps` steps of the active window
  warm = 2
  kept = []
  sched = torch.profiler.schedule(wait=0, warmup=warm, active=steps, repeat=1)
  with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA],
                              schedule=sched, on_trace_ready=kept.append) as prof:
    for i in range(warm + steps):
      env.process(acts[i % steps], active=active[i % steps])
      if i == warm + steps - 1:
        torch.cuda.synchronize()
      prof.step()
  env.stop()
  assert len(kept) == 1
  gpu = [e.name for e in kept[0].events() if e.device_type == DeviceType.CUDA]
  dtoh = sum("DtoH" in n for n in gpu)
  assert sum("host_frames_ingest" in n for n in gpu) == steps, (dtoh, gpu)
  assert not [n for n in gpu if "HtoD" in n], gpu
