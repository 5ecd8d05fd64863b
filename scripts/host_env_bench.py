"""Host simulators behind BatchedFrameEnvironment (INTEGRATION.md B2): env-steps/s of the adapter's process() and of a
FrameTrainer update loop with a real UnrealModel (A = 3), for the HostEnvProducer of this tree (worker threads, one
ingest launch per step reading pinned staging) against the per-step producer it replaced (serial env calls, host u8
conversion, staging upload, rows_select, stream synchronize, a dozen small launches), run alternately in one process.

The simulator has the reference's instance contract and returns TableFrameEnvOracle frames (float32 `uint8 / 255`, or
uint8 with --u8); each process() spends --sim-us in time.sleep, which releases the GIL like the Pipe round trip of the
reference's lab / gym env classes.  It starts no processes.

  python scripts/host_env_bench.py [--part process|trainer|all] [--n 64,256,1024] [--sim-us 0,500,2000]
                                   [--workers 1,8,32] [--u8] [--out-dir DIR]

Writes DIR/r6_host_env_<part>_<frames>.jsonl (one line per measurement, the first with the card, its power limit and
SM clock) and, for the process() part, DIR/r6_host_env_profile_<frames>.json (launches, copies and host
synchronisations per process() call, torch.profiler, in a run of its own after the timed ones).
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from oracle import unreal_oracle as O


class SleepySim(object):
  """A host env with the reference's instance contract (environment.py:76-86): TableFrameEnvOracle's frame stream,
  rewards and terminals, `sim_us` of simulated simulator time per process() (a shared, settable value)."""

  def __init__(self, env_id, table, clock, u8=False):
    self.oracle = O.TableFrameEnvOracle.__new__(O.TableFrameEnvOracle)
    self.oracle.env_id, self.oracle.table, self.oracle.counter = int(env_id), table, 0
    self.frames = table if u8 else table.astype(np.float32) / np.float32(255.0)
    self.clock = clock
    self.reset()

  def reset(self):
    o = self.oracle
    o.counter += 1
    self.last_state = {'image': self.frames[o._hash(0) % o.K_FRAMES]}

  def process(self, action, flag=1):
    if self.clock[0]:
      time.sleep(self.clock[0] * 1e-6)
    o = self.oracle
    o.counter += 1
    h = o._hash(int(action) + 1)
    reward = float(((h // o.K_FRAMES) % 5) - 2) * 0.5 if h % 3 == 0 else 0.0
    state = {'image': self.frames[h % o.K_FRAMES]}
    self.last_state = state
    return state, reward, h % 29 == 0, None


def baseline_producer_class():
  """HostEnvProducer as it was before the worker threads and the ingest kernel (kept here as the baseline)."""
  from unreal_b200 import kernels as K
  from unreal_b200.environment.frame_environment import FrameProducer

  def _rows(mask, like):
    return mask.to(torch.bool).view(-1, *([1] * (like.dim() - 1)))

  class BaselineHostEnvProducer(FrameProducer):
    def __init__(self, envs, device, action_size, objective_size=0, frame_shape=(84, 84, 3)):
      self.envs = list(envs)
      self.num_envs = len(self.envs)
      self.device = torch.device(device)
      self.action_size = int(action_size)
      self.objective_size = int(objective_size)
      self.frame_shape = tuple(frame_shape)
      n = self.num_envs
      self._stage = torch.empty(n, *self.frame_shape, dtype=torch.uint8).pin_memory()
      self._rt = torch.zeros(n, 2, dtype=torch.float32).pin_memory()
      self._obj = torch.zeros(n, max(1, self.objective_size), dtype=torch.float32).pin_memory()

    @staticmethod
    def _u8(image):
      a = np.asarray(image)
      if a.dtype == np.uint8:
        return a
      return np.rint(a.astype(np.float64) * 255.0).clip(0, 255).astype(np.uint8)

    def _put(self, e, state):
      self._stage[e].copy_(torch.from_numpy(np.ascontiguousarray(self._u8(state['image']))))
      if self.objective_size:
        self._obj[e, :self.objective_size] = torch.as_tensor(np.asarray(state['objective'], dtype=np.float32))

    def _upload(self, mask_host, out, objective):
      m = torch.from_numpy(mask_host).to(self.device)
      K.rows_select(out, self._stage.to(self.device, non_blocking=True), None, m)
      if objective is not None and self.objective_size:
        fresh = self._obj[:, :self.objective_size].to(self.device, non_blocking=True)
        objective.copy_(torch.where(_rows(m, objective), fresh, objective))
      torch.cuda.current_stream().synchronize()

    def reset(self, mask, out, objective=None):
      mask_host = np.ones(self.num_envs, bool) if mask is None else mask.to(torch.bool).cpu().numpy()
      for e in np.flatnonzero(mask_host):
        self.envs[e].reset()
        self._put(e, self.envs[e].last_state)
      if mask_host.any():
        self._upload(mask_host, out, objective)

    def step(self, action, active, out, reward, terminal, objective=None):
      act = action.cpu().numpy()
      mask_host = np.ones(self.num_envs, bool) if active is None else active.to(torch.bool).cpu().numpy()
      self._rt.zero_()
      for e in np.flatnonzero(mask_host):
        state, r, t, _ = self.envs[e].process(int(act[e]))
        self._put(e, state if isinstance(state, dict) else {'image': state})
        self._rt[e, 0] = float(r)
        self._rt[e, 1] = 1.0 if t else 0.0
      rt = self._rt.to(self.device, non_blocking=True)
      reward.copy_(rt[:, 0])
      terminal.copy_(rt[:, 1].to(torch.uint8))
      self._upload(mask_host, out, objective)

  return BaselineHostEnvProducer


def make_env(kind, n, clock, u8, dev, workers=1, table=None):
  from unreal_b200.environment import frame_environment as FE
  table = O.make_frame_table(3) if table is None else table
  sims = [SleepySim(e, table, clock, u8) for e in range(n)]
  if kind == "old":
    prod = baseline_producer_class()(sims, dev, 3)
  else:
    prod = FE.HostEnvProducer(sims, dev, 3, workers=workers)
  return FE.BatchedFrameEnvironment(prod, dev)


def check_equal(dev, u8, n=64, steps=30):
  """old and new producers give bit-identical frames, records, pixel change and scalars on the same stream."""
  clock = [0]
  old, new = make_env("old", n, clock, u8, dev), make_env("new", n, clock, u8, dev, workers=8)
  rs = np.random.RandomState(0)
  ok = torch.equal(old.last_state['image'], new.last_state['image'])
  for _ in range(steps):
    act = torch.from_numpy(rs.randint(0, 3, size=n).astype(np.int32)).to(dev)
    active = torch.from_numpy((rs.rand(n) < 0.8).astype(np.uint8)).to(dev)
    a = old.process(act, active=active)
    b = new.process(act, active=active)
    ok &= all(torch.equal(x, y) for x, y in ((a[0]['image'], b[0]['image']), (a[1], b[1]), (a[2], b[2]), (a[3], b[3]),
                                            (old.frame_rec, new.frame_rec), (old.last_action, new.last_action),
                                            (old.last_reward, new.last_reward)))
  new.stop()
  return bool(ok)


def process_rate(env, n, steps, dev, rs):
  acts = torch.from_numpy(rs.randint(0, 3, size=(steps + 2, n)).astype(np.int32)).to(dev)
  for i in range(2):
    env.process(acts[i])
  torch.cuda.synchronize()
  t0 = time.perf_counter()
  for i in range(steps):
    env.process(acts[2 + i])
  torch.cuda.synchronize()
  return n * steps / (time.perf_counter() - t0)


def make_trainer(env, n, dev, hist):
  from unreal_b200.environment.environment import Environment
  from unreal_b200.model.model import UnrealModel
  from unreal_b200.train.rmsprop_applier import RMSPropApplier
  from unreal_b200.train.trainer import Trainer
  Environment.register('hostbench', lambda name, args, tt, ti: env, action_size=3)
  Environment.action_size = -1
  net = UnrealModel(3, 0, -1, True, True, True, True, 0.05, 0.001, dev, {'segnet_mode': 0}, (84, 84), True, 0, 0.0,
                    0.0, num_envs=n, seed=0)
  applier = RMSPropApplier(7e-4, decay=0.99, momentum=0.0, epsilon=0.1, clip_norm=40.0)
  tr = Trainer(0, net, 7e-4, None, applier, 'hostbench', '', True, True, True, True, 0.05, 0.001, 20, 20, 0.99, 0.9,
               hist, 10 ** 8, str(dev), {'segnet_mode': 0}, (84, 84), True, 0, np.random.RandomState(1), 50.0, 0.0, 0.0,
               num_envs=n, seeds=np.arange(n) + 11, use_graphs=False)
  tr.prepare()
  Environment._registry.pop('hostbench', None)
  ex = tr.experience
  act = torch.zeros(n, dtype=torch.int32, device=dev)
  while not ex.is_full():
    prev = env.last_state['image']
    lr = env.last_reward.clone()
    act.random_(0, 3)
    _, r, _, pc = env.process(act)
    ex.add_frames(env.frame_rec, frame=prev, pixel_change=pc, reward=r, last_reward=lr)
  tr._ring_full = True
  tr.process(None, 0)
  torch.cuda.synchronize()
  return tr


def trainer_rate(tr, n, iters):
  torch.cuda.synchronize()
  t0 = time.perf_counter()
  for _ in range(iters):
    tr.process(None, 0)
  torch.cuda.synchronize()
  return n * 20 * iters / (time.perf_counter() - t0)


def profile_counts(env, n, dev, steps=20):
  from torch.autograd import DeviceType
  rs = np.random.RandomState(2)
  acts = torch.from_numpy(rs.randint(0, 3, size=(steps + 1, n)).astype(np.int32)).to(dev)
  active = torch.from_numpy((rs.rand(steps + 1, n) < 0.9).astype(np.uint8)).to(dev)
  env.process(acts[0], active=active[0])
  torch.cuda.synchronize()
  acts_ = [torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]
  with torch.profiler.profile(activities=acts_) as prof:
    for i in range(steps):
      env.process(acts[1 + i], active=active[1 + i])
    torch.cuda.synchronize()
  ev = prof.events()
  gpu = [e.name for e in ev if e.device_type == DeviceType.CUDA]
  cpu = [e.name for e in ev if e.device_type == DeviceType.CPU]
  copies = [g for g in gpu if g.startswith("Memcpy") or g.startswith("Memset")]
  kernels = [g for g in gpu if g not in copies]
  syncs = [c for c in cpu if c.startswith("cuda") and "Synchronize" in c]
  syncs_in_loop = len(syncs) - 1                       # the profile window's closing torch.cuda.synchronize()
  return dict(steps=steps, kernels_per_step=len(kernels) / steps,
              htod_per_step=sum("HtoD" in g for g in copies) / steps,
              dtoh_per_step=sum("DtoH" in g for g in copies) / steps,
              host_syncs_per_step=syncs_in_loop / steps,
              kernel_names=sorted(set(k.split("(")[0][:90] for k in kernels)), sync_calls=sorted(set(syncs)))


def card():
  q = "name,power.limit,clocks.sm,clocks.max.sm"
  try:
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True,
                         text=True, timeout=30).stdout.strip()
  except Exception as ex:   # noqa: BLE001
    out = "nvidia-smi failed: %s" % ex
  return dict(zip(q.split(","), [s.strip() for s in out.split(",")])) if "," in out else {"nvidia_smi": out}


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--n", default="64,256,1024")
  ap.add_argument("--sim-us", default="0,500,2000")
  ap.add_argument("--workers", default="1,8,32")
  ap.add_argument("--steps", type=int, default=5, help="timed process() calls per measurement")
  ap.add_argument("--iters", type=int, default=1, help="timed trainer updates (20 env steps each) per measurement")
  ap.add_argument("--reps", type=int, default=2, help="alternating old / new rounds of the process() rates")
  ap.add_argument("--hist", type=int, default=40)
  ap.add_argument("--u8", action="store_true", help="simulators return uint8 frames instead of float32")
  ap.add_argument("--part", choices=("process", "trainer", "all"), default="all",
                  help="process(): rates, equality check and the profile; trainer: update-loop rates")
  ap.add_argument("--out-dir", default="profiles")
  a = ap.parse_args()
  from unreal_b200 import _lib
  _lib.require_device()
  dev = torch.device("cuda", 0)
  ns = [int(x) for x in a.n.split(",")]
  sims = [int(x) for x in a.sim_us.split(",")]
  wks = [int(x) for x in a.workers.split(",")]
  os.makedirs(a.out_dir, exist_ok=True)
  frames = "uint8" if a.u8 else "float32"
  path = os.path.join(a.out_dir, "r6_host_env_%s_%s.jsonl" % (a.part, frames))
  out = open(path, "w")

  def emit(d):
    out.write(json.dumps(d) + "\n")
    out.flush()
    print(json.dumps(d), flush=True)

  head = dict(kind="card", **card(), torch=torch.__version__, frames=frames)
  if a.part != "trainer":
    head["equal_old_new"] = check_equal(dev, a.u8)
  emit(head)

  rs = np.random.RandomState(5)
  for n in ns if a.part != "trainer" else ():
    clock = [0]
    envs = {"old": make_env("old", n, clock, a.u8, dev)}
    for w in wks:
      envs["new_w%d" % w] = make_env("new", n, clock, a.u8, dev, workers=w)
    for sim in sims:
      clock[0] = sim
      rates = {k: [] for k in envs}
      for _ in range(a.reps):
        for k, env in envs.items():
          rates[k].append(process_rate(env, n, a.steps, dev, rs))
      for k, r in rates.items():
        emit(dict(kind="process", n=n, sim_us=sim, producer=k, env_steps_per_s=max(r), all=r, frames=frames))
    for k, env in envs.items():
      if k != "old":
        env.stop()

  if a.part != "process":
    for n in ns:
      clock = [0]
      trainers = {"old": make_trainer(make_env("old", n, clock, a.u8, dev), n, dev, a.hist)}
      for w in wks:
        trainers["new_w%d" % w] = make_trainer(make_env("new", n, clock, a.u8, dev, workers=w), n, dev, a.hist)
      for sim in sims:
        for k, tr in trainers.items():
          clock[0] = sim
          r = trainer_rate(tr, n, a.iters)
          clock[0] = 0
          emit(dict(kind="trainer", n=n, sim_us=sim, producer=k, env_steps_per_s=r, iters=a.iters, frames=frames,
                    finite=bool(torch.isfinite(tr.last_losses["total"]))))
      for k, tr in trainers.items():
        tr.environment.stop()
      del trainers
      torch.cuda.empty_cache()

  out.close()
  if a.part == "trainer":
    return
  prof = dict(card=head, n=256, sim_us=0, frames=frames)
  for k, env in (("old", make_env("old", 256, [0], a.u8, dev)), ("new_w8", make_env("new", 256, [0], a.u8, dev, 8))):
    prof[k] = profile_counts(env, 256, dev)
    env.stop()
  with open(os.path.join(a.out_dir, "r6_host_env_profile_%s.json" % frames), "w") as f:
    json.dump(prof, f, indent=1)
  print(json.dumps(prof))


if __name__ == "__main__":
  main()
