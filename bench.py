#!/usr/bin/env python
"""Headline benchmark: maze env-steps/s including pixel-change + returns (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--obs-dtype f32|u8] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1], per GPU): 4096 batched maze envs; one *step* = one pass of
the hot path over that batch = 20 rollout steps of K1 (fused maze step + 84x84x3 render +
20x20 pixel-change) + K3 (20-step n-step returns and advantages) + K4 (pixel-control Q
targets) = 81 920 env-steps.  Envs shard across GPUs with no data-path collective (weak
scaling).  Prints ONE JSON line (rank 0).

`value`     device-resident throughput (inputs already in HBM), CUDA events, max over ranks.
`e2e`       the same pass through the host-buffer entry point RolloutTargets.run_host():
            pinned host inputs copied H2D and rewards/terminals/returns/advantages copied
            D2H inside the timed region every step.
`roofline`  K1 (the dominant kernel): algorithmic bytes per launch / its average launch
            duration, measured with CUDA events inside the timed region.
`cpu_baseline` the numpy oracle port of the reference path on this box's host cores.

--impl reference  times the reference's CPU implementation of the path (the oracle port: the
reference is Python and is not part of this repository) on all host cores.

--dump-outputs DIR  after the timed steps, writes what the last timed pass of rank 0 computed as
DIR/<name>.npy (float32 / float64, fixed samples of the larger buffers, at most about 41 MB), so
that two builds can be compared output for output: the inputs are seeded, identical for identical
arguments.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "maze env-steps/s incl. pixel-change+returns"
UNIT = "env-steps/s"
ENVS_PER_GPU = 4096
ROLLOUT = 20
# SURVEY.md 8(d) / DESIGN.md: algorithmic bytes per env-step of K1
K1_BYTES = {"f32": 86313, "u8": 22809}
K3_BYTES_PER_ENV_STEP = 17.2
K4_BYTES_PER_ENV_STEP = 3280


def parse():
  p = argparse.ArgumentParser()
  p.add_argument("--gpus", type=int, default=1)
  p.add_argument("--steps", type=int, default=300)
  p.add_argument("--warmup", type=int, default=10)
  p.add_argument("--impl", default="b200", choices=["b200", "reference"])
  p.add_argument("--obs-dtype", default="f32", choices=["f32", "u8"])
  p.add_argument("--envs-per-gpu", type=int, default=ENVS_PER_GPU)
  p.add_argument("--window-kernel", default="auto", choices=["auto", "on", "off"],
                 help="K1 as ONE launch over the T steps of a pass (the T actions are inputs) instead of T launches; "
                      "auto = on")
  p.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
  p.add_argument("--no-cpu-baseline", action="store_true")
  p.add_argument("--no-agent", action="store_true", help="skip the full-agent (configs[2]) side measurement")
  p.add_argument("--agent-envs", type=int, default=8192, help="envs per GPU of the full-agent side measurement")
  p.add_argument("--agent-updates", type=int, default=6)
  p.add_argument("--agent-obs", default="cells", choices=["cells", "s2d", "f32"],
                 help="full-agent observations: agent cells (conv1 renders its tiles in shared memory, no frame in HBM), "
                      "K1-rendered x'' planes, or f32 frames")
  p.add_argument("--dump-outputs", metavar="DIR", default=None,
                 help="write the outputs of the last timed pass as DIR/<name>.npy (see dump_outputs)")
  args = p.parse_args()
  if args.steps < 1:
    p.error("--steps must be at least 1")
  return args


def workload_config(args):
  return {
      "workload": "configs[1]: %d batched maze envs per GPU, fused step/render/pixel-change (K1) x %d + "
                  "20-step n-step returns/advantages (K3) + PC Q-targets (K4)" % (args.envs_per_gpu, ROLLOUT),
      "envs_per_gpu": args.envs_per_gpu, "rollout_len": ROLLOUT, "obs_dtype": args.obs_dtype,
      "k1_launches_per_pass": "1 (window kernel)" if args.window_kernel != "off" else str(ROLLOUT),
      "gamma": 0.99, "gamma_pc": 0.9,
      "l2": "every pass writes a %.1f GB rollout buffer (obs+pc+targets), far larger than the 126 MB L2" % (
          args.envs_per_gpu * ROLLOUT * (K1_BYTES[args.obs_dtype] + 1600) / 1e9),
  }


# --------------------------------------------------------------------------- clocks
class ClockSampler(object):
  """Samples SM clock and throttle reasons through NVML while the timed region runs."""

  def __init__(self, index):
    self.samples = []
    self.reasons = set()
    self.max_mhz = None
    self._stop = threading.Event()
    self._thr = None
    try:
      import pynvml
      pynvml.nvmlInit()
      self.nv = pynvml
      self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
      self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
    except Exception as e:  # NVML missing: report that, do not fail the run
      self.nv = None
      self.err = repr(e)

  def _loop(self):
    nv = self.nv
    names = {}
    for k in dir(nv):
      if k.startswith("nvmlClocksThrottleReason") or k.startswith("nvmlClocksEventReason"):
        v = getattr(nv, k)
        if isinstance(v, int) and v:
          names[v] = k.replace("nvmlClocksThrottleReason", "").replace("nvmlClocksEventReason", "")
    while not self._stop.is_set():
      try:
        self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        try:
          mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
          mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for bit, name in names.items():
          if mask & bit and bit & (bit - 1) == 0:
            self.reasons.add(name)
      except Exception:
        pass
      time.sleep(0.02)

  def start(self):
    if self.nv is not None:
      self._thr = threading.Thread(target=self._loop, daemon=True)
      self._thr.start()

  def stop(self):
    self._stop.set()
    if self._thr is not None:
      self._thr.join()
    s = sorted(self.samples)
    reasons = sorted(r for r in self.reasons if r not in ("None", "GpuIdle", "ApplicationsClocksSetting"))
    return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
            "samples": len(s)} if self.nv is not None else {"sm_mhz": None, "sm_max_mhz": None, "reasons": [],
                                                            "error": self.err}


# --------------------------------------------------------------------------- CPU arm
def cpu_throughput(seconds, procs):
  """Bounded sample of the same workload on host cores -> (env-steps/s, env-steps, description)."""
  from oracle import cpu_path
  steps0, wall0 = cpu_path.run_parallel(1, 1, ROLLOUT, 10)          # calibrate one core
  rate = steps0 / wall0
  passes = max(1, int(seconds * rate / (2 * ROLLOUT)))               # 2 envs per process
  steps, wall = cpu_path.run_parallel(procs, 2, ROLLOUT, passes)
  return steps / wall, steps, "%d processes x 2 envs x %d passes x %d steps = %d env-steps in %.1f s" % (
      procs, passes, ROLLOUT, steps, wall)


def run_reference(args):
  """The reference's CPU implementation of the path (oracle port), all host cores."""
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return 0
  from oracle import cpu_path
  import multiprocessing as mp
  procs = cpu_path.host_cores()
  steps0, wall0 = cpu_path.run_parallel(1, 1, ROLLOUT, 10)
  rate = steps0 / wall0
  # size each step so that warmup + steps finish in about two minutes
  budget = 120.0
  envs = max(1, min(64, int(budget * rate / (ROLLOUT * (args.steps + args.warmup)))))
  pool = mp.get_context("fork").Pool(procs) if procs > 1 else None
  for _ in range(args.warmup):
    cpu_path.run_parallel(procs, envs, ROLLOUT, 1, pool)
  t0 = time.perf_counter()
  total = 0
  for _ in range(args.steps):
    s, _w = cpu_path.run_parallel(procs, envs, ROLLOUT, 1, pool)
    total += s
  wall = time.perf_counter() - t0
  if pool is not None:
    pool.close(); pool.join()
  value = total / wall
  sample = "each step = %d processes x %d envs x %d rollout steps of the numpy oracle port (bounded sample)" % (
      procs, envs, ROLLOUT)
  line = {
      "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
      "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
      "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(args),
      "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": "port", "sample": sample},
      "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
      "gpu_launches": 0,
  }
  print(json.dumps(line), flush=True)
  return 0



# --------------------------------------------------------------------------- full agent (side measurement)
def measure_agent(torch, dist, dev, rank, world, envs, updates, history=2000, obs='cells'):
  """BASELINE configs[2] slice per GPU: `envs` mazes, per-env `history`-frame replay ring, RP/VR/PC
  sampling, UnrealModel forward/backward on tcgen05 (K7), NCCL gradient exchange + fused RMSProp
  (K6).  One update = 20 env-steps per env.  Reported beside the headline, never instead of it."""
  import numpy as np
  from unreal_b200.environment.environment import Environment
  from unreal_b200.model.model import UnrealModel
  from unreal_b200.train.rmsprop_applier import RMSPropApplier
  from unreal_b200.train.sharding import env_seeds, env_shard
  from unreal_b200.train.trainer import Trainer
  Environment.action_size = -1
  lo, hi = env_shard(envs * world, world, rank)
  net = UnrealModel(4, 0, -1, True, True, True, True, 0.05, 0.001, dev, {'segnet_mode': 0}, (84, 84), True, 0, 0.0,
                    0.0, num_envs=envs, seed=0)
  applier = RMSPropApplier(7e-4, decay=0.99, momentum=0.0, epsilon=0.1, clip_norm=40.0)
  tr = Trainer(rank, net, 7e-4, None, applier, 'maze', '', True, True, True, True, 0.05, 0.001, 20, 20, 0.99, 0.9,
               history, 10 ** 9, str(dev), {'segnet_mode': 0}, (84, 84), True, 0, np.random.RandomState(1), 50.0, 0.0,
               0.0, num_envs=envs, seeds=env_seeds(0xA3C, lo, hi), use_graphs=True, obs_s2d=(obs == 's2d'), obs_cells=(obs == 'cells'))
  tr.prepare()
  t0 = time.perf_counter()
  while not tr.experience.is_full():
    tr.process(None, 0)
  torch.cuda.synchronize(dev)
  fill_s = time.perf_counter() - t0
  for _ in range(2):
    tr.process(None, 0)
  upd = []
  orig = tr._update          # the learner step: eager net.update() or the replay of its CUDA graph

  def timed(feed, lr):
    a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
    a.record(); out = orig(feed, lr); b.record(); upd.append((a, b))
    return out

  tr._update = timed
  e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
  if world > 1:
    dist.barrier()
  torch.cuda.synchronize(dev)
  e0.record()
  steps = 0
  for _ in range(updates):
    d, _ = tr.process(None, 0)
    steps += d
  e1.record()
  if world > 1:
    dist.barrier()
  torch.cuda.synchronize(dev)
  ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
  if world > 1:
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
  ms = float(ms)
  steps_t = torch.tensor([float(steps)], device=dev, dtype=torch.float64)
  if world > 1:
    dist.all_reduce(steps_t, op=dist.ReduceOp.SUM)
  steps_all = int(steps_t.item())
  upd_ms = sum(a.elapsed_time(b) for a, b in upd) / len(upd)
  nccl_parity = check_nccl_parity(torch, dist, dev, rank, world, net, applier) if world > 1 else None
  losses = {k: float(v) for k, v in tr.last_losses.items()}
  mem = torch.cuda.max_memory_allocated(dev) / 1e9
  tr.stop()
  return {"workload": "configs[2] slice: %d maze envs per GPU, %d-frame replay ring per env, PC/VR/RP sampling, "
                      "UnrealModel fwd/bwd (bf16 tcgen05 GEMMs, fp32 accumulate), %s fused clip+RMSProp"
                      % (envs, history, "NCCL gradient exchange +" if world > 1 else "single-GPU"),
          "envs_per_gpu": envs, "history": history, "updates": updates,
          "observations": {"cells": "agent cells int32 [N,2]; conv1 fwd / wgrad synthesise their x'' tiles in shared memory "
                                    "(render fused into the consumer: no frame is written to or read from HBM)",
                           "s2d": "x'' bf16 planes rendered by K1 (42 KB per frame)",
                           "f32": "f32 frames rendered by K1 (85 KB per frame) + space-to-depth pass"}[obs],
          # env steps actually taken: the sum over envs of the rollout lengths Trainer.process() returns (an env whose
          # episode ends mid-window idles for the rest of it, trainer.py:279-296), summed over ranks
          "value": steps_all / (ms * 1e-3), "env_steps": steps_all, "slot_steps": world * envs * 20 * updates,
          "unit": "env-steps/s", "ms_per_update": ms / updates, "model_update_ms": upd_ms,
          "updates_per_s": updates / (ms * 1e-3), "ring_fill_s": fill_s, "params": net.num_parameters,
          "finite": bool(all(np.isfinite(v) for v in losses.values())), "grad_norm": losses.get("grad_norm"),
          "peak_mem_gb": mem, "update_cuda_graph": tr._ugraph is not None,
          "update_graph_mode": ("none (eager)" if tr._ugraph is None else
                                "one graph incl. the NCCL exchange" if (world > 1 and tr.nccl_in_graph) else
                                "graph A (fwd+bwd) + eager NCCL exchange around K6 (5 launches) + graph B (shadow refresh)"
                                if world > 1 else "one graph"),
          "timing": "CUDA events around %d Trainer.process() calls, max over ranks" % updates,
          "nccl_parity": nccl_parity}


def check_nccl_parity(torch, dist, dev, rank, world, net, applier):
  """The assertions of tests/test_gpu_multi.py on the live learner group, outside every timed region (SURVEY 8e):
  (1) the NCCL-sharded clip + RMSProp (reduce-scatter -> shard update -> all-gather) equals the single-GPU K6 kernels
  applied to the mean gradient; (2) the learners' parameters are bit-identical on all ranks."""
  from unreal_b200 import kernels as K
  from unreal_b200.train.rmsprop_applier import RMSPropApplier
  out = {}
  try:
    p = net.flat.numel()
    gen = torch.Generator(device=dev).manual_seed(77)                    # same `var` on every rank
    var0 = torch.randn(p, device=dev, generator=gen)
    grad = torch.randn(p, device=dev, generator=torch.Generator(device=dev).manual_seed(1000 + rank)) * 0.05
    ap = RMSPropApplier(7e-4, decay=0.99, momentum=0.0, epsilon=0.1, clip_norm=40.0)
    flat = var0.clone()
    norm = ap.apply_flat_to(flat, grad.clone(), 7e-4)
    gsum = grad.clone()
    dist.all_reduce(gsum, op=dist.ReduceOp.SUM)
    gmean = gsum / world
    ref = var0.clone(); rms = torch.ones(p, device=dev)
    ref_norm = torch.zeros(1, device=dev)
    K.rmsprop_update(ref, rms, None, gmean, K.grad_sumsq(gmean), 7e-4, 0.99, 0.0, 0.1, 40.0, grad_norm=ref_norm)
    err = float(((flat - ref).abs() / ref.abs().clamp_min(1.0)).max())
    out["sharded_vs_single_gpu_max_rel_err"] = err
    out["grad_norm_rel_err"] = abs(float(norm) - float(ref_norm)) / max(float(ref_norm), 1e-12)
    # (2) the agent's own parameters after its updates: compare every rank's buffer with rank 0's, bit for bit
    mine = net.flat.detach().clone()
    zero = mine.clone()
    dist.broadcast(zero, src=0)
    same = torch.tensor([1.0 if torch.equal(mine, zero) else 0.0], device=dev)
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    sh = flat.clone()
    dist.broadcast(sh, src=0)
    same2 = torch.tensor([1.0 if torch.equal(sh, flat) else 0.0], device=dev)
    dist.all_reduce(same2, op=dist.ReduceOp.MIN)
    out["params_bit_identical_across_ranks"] = bool(same.item() == 1.0 and same2.item() == 1.0)
    out["tolerance"] = 1e-5
    out["status"] = "ok" if (err <= 1e-5 and out["grad_norm_rel_err"] <= 1e-5 and
                             out["params_bit_identical_across_ranks"]) else "FAILED"
  except Exception as e:
    out = {"status": "error", "error": repr(e)[:300]}
  return out


def parity_check(torch, eng, envs=64):
  """After the timed loops: ONE more pass of the benched engine (4096 envs, CUDA graphs, the state the timed passes left
  behind), checked against the oracle on a slice of `envs` environments -- transitions, pixel change, last frames,
  n-step returns, PC targets, all bit for bit (the oracle only checks; nothing it computes is timed or shipped)."""
  import numpy as np
  from oracle import unreal_oracle as O
  t = eng.t
  try:
    torch.cuda.synchronize(eng.device)
    pos0 = eng.state.pos[:envs].cpu().numpy().copy()
    eng.run_device()
    torch.cuda.synchronize(eng.device)
    acts = eng.actions[:, :envs].cpu().numpy(); vals = eng.values[:, :envs].cpu().numpy()
    boot = eng.boot_value[:envs].cpu().numpy(); bq = eng.boot_q[:envs].cpu().numpy()
    rew = np.zeros((t, envs), np.float32); term = np.zeros((t, envs), np.uint8)
    pcs = np.zeros((t, envs, 20, 20), np.float32)
    last = [None] * envs
    for e in range(envs):
      env = O.MazeOracle()
      env.x, env.y = int(pos0[e, 0]), int(pos0[e, 1])
      env.last_state = {'image': O.maze_render(env.x, env.y)}
      for i in range(t):
        img, r, tm, pc = env.process(int(acts[i, e]))
        rew[i, e] = r; term[i, e] = tm; pcs[i, e] = pc
        if tm:
          env.reset()
      last[e] = env.last_state['image']
    scale = 255.0 if eng.obs.dtype == torch.uint8 else 1.0
    ok = np.array_equal(eng.reward[:, :envs].cpu().numpy(), rew) and np.array_equal(eng.terminal[:, :envs].cpu().numpy(), term)
    ok = ok and np.array_equal(eng.pc[:, :envs].cpu().numpy(), pcs)
    got_obs = eng.obs[t - 1, :envs].cpu().numpy()
    ok = ok and all(np.array_equal(got_obs[e], (last[e] * scale).astype(got_obs.dtype)) for e in range(envs))
    R, adv = O.nstep_returns_segmented(rew, vals, term, boot, eng.gamma, np.float32)
    ok = ok and np.array_equal(eng.R[:, :envs].cpu().numpy(), R) and np.array_equal(eng.adv[:, :envs].cpu().numpy(), adv)
    want = np.zeros_like(pcs)
    acc = bq.astype(np.float32).copy()
    for i in range(t - 1, -1, -1):
      acc = np.where(term[i][:, None, None] != 0, np.float32(0), acc)
      acc = pcs[i] + np.float32(eng.gamma_pc) * acc
      want[i] = acc
    ok = ok and np.array_equal(eng.pc_tgt[:, :envs].cpu().numpy(), want)
    return "ok" if ok else "FAILED", "%d envs x %d steps of the benched engine vs the oracle, bit-exact" % (envs, t)
  except Exception as e:
    return "error: " + repr(e)[:200], ""


def dump_outputs(torch, eng, out_dir, max_envs=4096, map_envs=256, frames=256):
  """Writes the buffers the last pass of `eng` left for its caller as out_dir/<name>.npy, about 41 MB at most.
  reward, terminal, R, adv and frame_rec ([T, S, 2]: its low and high 32 bits, as float64 holds 53) for a sample of
  `max_envs` envs (all of them up to that many); pc and pc_tgt for a sample of `map_envs` envs ([T, S, 20, 20]); obs
  for a sample of `frames` (step, env) pairs in ascending order of step * N + env.  The samples are sorted and drawn
  from RandomState(0), so they depend on N and T only."""
  import numpy as np
  t, n = eng.t, eng.n
  rs = np.random.RandomState(0)

  def pick(m, k):
    return torch.from_numpy(np.sort(rs.choice(m, min(m, k), replace=False))).to(eng.device)

  envs, map_sel, rows = pick(n, max_envs), pick(n, map_envs), pick(t * n, frames)
  torch.cuda.synchronize(eng.device)
  rec = eng.frame_rec.index_select(1, envs).cpu().numpy().view(np.uint64)
  outs = {
      "reward": eng.reward.index_select(1, envs), "terminal": eng.terminal.index_select(1, envs),
      "R": eng.R.index_select(1, envs), "adv": eng.adv.index_select(1, envs),
      "pc": eng.pc.index_select(1, map_sel), "pc_tgt": eng.pc_tgt.index_select(1, map_sel),
      "obs": eng.obs.view(t * n, 84, 84, 3).index_select(0, rows),
  }
  os.makedirs(out_dir, exist_ok=True)
  for name, v in outs.items():
    np.save(os.path.join(out_dir, name + ".npy"), v.float().cpu().numpy())
  np.save(os.path.join(out_dir, "frame_rec.npy"),
          np.stack([rec & np.uint64(0xFFFFFFFF), rec >> np.uint64(32)], -1).astype(np.float64))


def measure_pc_stress(torch, dev, peak, seq=50000, dtype_name="u8"):
  """BASELINE configs[3]: pixel-control target stress -- synthetic 84x84x3 frame stream (u8, scaled by /255 on load like
  lab / indoor / gym frames), 20x20 cells, n = 20, gamma_pc = 0.9, 1 M frames per batch: K2 (stream pixel change, every
  frame read from HBM once) + K4 (PC Q-target scan).  Frames/s and the fraction of measured HBM on SURVEY 8(d)'s bytes."""
  from unreal_b200 import kernels as K
  L = 20
  dtype = torch.uint8 if dtype_name == "u8" else torch.float32
  g = torch.Generator(device=dev).manual_seed(0)
  frames = torch.empty(seq, L + 1, 84, 84, 3, dtype=dtype, device=dev)
  for i in range(0, seq, 2500):
    chunk = frames[i:i + 2500]
    chunk.copy_(torch.randint(0, 256, chunk.shape, dtype=torch.uint8, device=dev, generator=g) if dtype == torch.uint8
                else torch.rand(chunk.shape, device=dev, generator=g))
  boot = torch.rand(seq, 20, 20, device=dev, generator=g)
  pc = torch.empty(seq, L, 20, 20, device=dev)
  pc_t = torch.empty(L, seq, 20, 20, device=dev)
  tgt = torch.empty(L, seq, 20, 20, device=dev)

  def timed(fn, iters=5):
    for _ in range(3):
      fn()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
      fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / iters * 1e-3

  n_frames = seq * L
  t2 = timed(lambda: K.pixel_change_stream(frames, pc))
  b2 = seq * (L + 1) * 21168 * frames.element_size() + n_frames * 1600
  pc_t.copy_(pc.transpose(0, 1))
  t4 = timed(lambda: K.pc_targets(pc_t, None, None, boot, 0.9, tgt))
  b4 = n_frames * 3200 + seq * 1600
  checksum = float(tgt[:, :64].double().sum())
  del frames, pc, pc_t, tgt
  torch.cuda.empty_cache()
  return {"workload": "configs[3]: %d sequences x (20+1) %s frames 84x84x3 = %d frames per batch (%.1f GB resident, >> L2), "
                      "K2 stream pixel change + K4 PC Q-targets, gamma_pc 0.9" % (seq, dtype_name, n_frames, b2 / 1e9),
          "frames": n_frames, "value": n_frames / (t2 + t4), "unit": "frames/s", "ms_per_batch": (t2 + t4) * 1e3,
          "k2": {"ms": t2 * 1e3, "frames_per_s": n_frames / t2, "gbs": b2 / t2 / 1e9, "frac": b2 / t2 / 1e9 / peak,
                 "algorithmic_bytes_per_frame": b2 / n_frames},
          "k4": {"ms": t4 * 1e3, "gbs": b4 / t4 / 1e9, "frac": b4 / t4 / 1e9 / peak},
          "pass_gbs": (b2 + b4) / (t2 + t4) / 1e9, "pass_frac": (b2 + b4) / (t2 + t4) / 1e9 / peak,
          "target": "SURVEY 8(d): >= 0.6 of measured HBM (>= 150 M u8 frames/s)", "checksum_tgt": checksum}


def measure_a3c(torch, dist, dev, rank, world, envs=1024, iters=10):
  """BASELINE configs[4] per GPU: MINOS-shaped synthetic observations (u8 84x84 RGB; the reference model consumes no depth
  channel, SURVEY 8a-a24), 3 pointgoal actions, goal vector G = 2, A3C-LSTM forward/backward + shared RMSProp on
  `envs` envs x T = 20 per GPU (batch 8192 x T over 8 GPUs).  The update replays CUDA graphs; under NCCL the gradient
  exchange sits between graph A (fwd+bwd) and graph B (shadow refresh)."""
  from unreal_b200 import _lib
  from unreal_b200.model.model import UnrealModel
  from unreal_b200.train.rmsprop_applier import RMSPropApplier
  N, T, A, G = envs, 20, 3, 2
  m = UnrealModel(A, G, -1, True, False, False, False, 0.05, 0.001, dev, {'segnet_mode': 0}, (84, 84), True, 0, 0.0, 0.0,
                  num_envs=N, seed=0)
  ap = RMSPropApplier(7e-4, decay=0.99, momentum=0.0, epsilon=0.1, clip_norm=40.0)
  g = torch.Generator(device=dev).manual_seed(rank)
  img = torch.randint(0, 256, (T, N, 84, 84, 3), dtype=torch.uint8, device=dev, generator=g)
  lar = torch.zeros(T, N, A + 1 + G, device=dev)
  lar.scatter_(2, torch.randint(0, A, (T, N, 1), device=dev, generator=g), 1.0)
  lar[..., A + 1:] = torch.rand(T, N, G, device=dev, generator=g)
  a = torch.zeros(T, N, A, device=dev).scatter_(2, torch.randint(0, A, (T, N, 1), device=dev, generator=g), 1.0)
  feed = {"base": dict(images=img, lar=lar, a=a, adv=torch.randn(T, N, device=dev, generator=g),
                       R=torch.randn(T, N, device=dev, generator=g), mask=torch.ones(T, N, device=dev),
                       c0=torch.zeros(N, 256, device=dev), h0=torch.zeros(N, 256, device=dev))}
  lr = torch.full((1,), 7e-4, device=dev)
  for _ in range(3):
    out = m.update(feed, lr, ap)
  torch.cuda.synchronize(dev)
  ga = torch.cuda.CUDAGraph()
  if world == 1:
    with _lib.graph_capture(ga):
      out = m.update(feed, lr, ap)
    step = ga.replay
    mode = "one graph"
  else:
    with _lib.graph_capture(ga):
      total, parts, grad = m.update_gradient(feed)
    gb = torch.cuda.CUDAGraph()
    with _lib.graph_capture(gb):
      m.refresh_shadow()
    out = {"total": total}

    def step():
      ga.replay(); ap.apply_flat_to(m.flat, grad, lr); gb.replay()
    mode = "graph A (fwd+bwd) + eager NCCL exchange around K6 + graph B (shadow refresh)"
  for _ in range(2):
    step()
  if world > 1:
    dist.barrier()
  torch.cuda.synchronize(dev)
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(iters):
    step()
  e1.record()
  if world > 1:
    dist.barrier()
  torch.cuda.synchronize(dev)
  t_ms = torch.tensor([e0.elapsed_time(e1) / iters], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
  ms = float(t_ms)
  samples = N * T * world
  return {"workload": "configs[4]: %d envs x T=20 per GPU (batch %d x 20 over %d GPU%s), u8 84x84x3 synthetic indoor-shaped frames, "
                      "A=3, goal vector G=2, A3C-LSTM fwd/bwd + %sfused clip+RMSProp" % (
                          N, N * world, world, "s" if world > 1 else "", "NCCL-sharded " if world > 1 else ""),
          "value": samples / (ms * 1e-3), "unit": "samples/s", "ms_per_update": ms, "update_graph_mode": mode,
          "model_tflops": samples * 18.5e6 / (ms * 1e-3) / 1e12,
          "frac_of_sustained_bf16_peak_per_gpu": samples * 18.5e6 / (ms * 1e-3) / 1e12 / 1393.1 / world,
          "finite": bool(torch.isfinite(out["total"])), "params": m.num_parameters}


def agent_cpu_baseline(envs=4, seconds=10.0):
  """SURVEY 8(d)(ii): the reference algorithm with a PyTorch-CPU learner (TensorFlow cannot run here):
  the oracle's env + replay + target path feeding oracle/model_oracle.py's forward/backward and the
  numpy RMSProp, all host cores through torch's intra-op threads.  Bounded sample."""
  import numpy as np
  import torch
  from oracle import model_oracle as MO, unreal_oracle as O, cpu_path
  cores = cpu_path.host_cores()
  torch.set_num_threads(cores)
  A, T = 4, 20
  params = MO.init_params(A, seed=0)
  oracle = MO.ModelOracle(params, A, 0, 0.05, 0.001)
  rs = np.random.RandomState(0)
  mazes = [O.MazeOracle() for _ in range(envs)]

  def frames_for(L):
    out = np.zeros((L, envs, 84, 84, 3), np.float32)
    for t in range(L):
      for e, m in enumerate(mazes):
        img, r, term, pc = m.process(int(rs.randint(4)))
        if term:
          m.reset()
        out[t, e] = m.last_state['image']
    return torch.from_numpy(out)

  def lar(L):
    x = torch.zeros(L, envs, A + 1); x[..., 0] = 1.0
    return x

  def one_update():
    a = torch.zeros(T, envs, A); a[..., 1] = 1.0
    feed = {"base": dict(images=frames_for(T), lar=lar(T), a=a, adv=torch.randn(T, envs), R=torch.randn(T, envs),
                         mask=torch.ones(T, envs), c0=torch.zeros(envs, 256), h0=torch.zeros(envs, 256)),
            "pc": dict(images=frames_for(T), lar=lar(T), a=a, R=torch.rand(T, envs, 20, 20), mask=torch.ones(T, envs)),
            "vr": dict(images=frames_for(T), lar=lar(T), R=torch.randn(T, envs), mask=torch.ones(T, envs)),
            "rp": dict(images=frames_for(3).permute(1, 0, 2, 3, 4).contiguous(), c=torch.eye(3)[torch.zeros(envs, dtype=torch.long)])}
    total, parts, grads = oracle.loss_and_grads(feed)
    for k, g in grads.items():      # shared RMSProp, rmsprop_applier.py:83-93 (no slots kept: timing only)
      params[k] -= 7e-4 * g / torch.sqrt(g * g * 0.01 + 1.0 * 0.99 + 0.1)
  one_update()
  t0 = time.perf_counter(); n = 0
  while time.perf_counter() - t0 < seconds:
    one_update(); n += 1
  wall = time.perf_counter() - t0
  return {"value": n * envs * T / wall, "unit": UNIT, "cores": cores, "kind": "port",
          "sample": "%d updates of %d envs x %d steps: numpy maze + PyTorch-CPU fp32 model fwd/bwd (oracle/model_oracle.py, "
                    "%d torch threads) + RMSProp in %.1f s -- the stand-in for the reference's TensorFlow CPU trainer"
                    % (n, envs, T, cores, wall)}

# --------------------------------------------------------------------------- B200 arm
def run_b200(args):
  import torch
  import torch.distributed as dist
  rank = int(os.environ.get("RANK", "0"))
  world = int(os.environ.get("WORLD_SIZE", "1"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  if world != args.gpus and world > 1:
    raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
  if not torch.cuda.is_available():
    raise SystemExit("bench.py needs a CUDA device (B200); there is no CPU fallback. "
                     "Use --impl reference for the CPU arm.")
  torch.cuda.set_device(local)
  dev = torch.device("cuda", local)
  if world > 1:
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
      os.environ["NCCL_DEBUG"] = "WARN"      # keep stdout to the one JSON line (no version banner)
    dist.init_process_group("nccl", device_id=dev)

  from unreal_b200 import _lib
  from unreal_b200.train.rollout import RolloutTargets
  _lib.require_device()
  n, t = args.envs_per_gpu, ROLLOUT
  obs_dtype = torch.float32 if args.obs_dtype == "f32" else torch.uint8
  eng = RolloutTargets(n, t, 0.99, 0.9, obs_dtype, dev, auto_reset=True, use_graphs=True,
                       window_kernel={"auto": None, "on": True, "off": False}[args.window_kernel])
  window = eng.window_kernel
  g = torch.Generator(device=dev).manual_seed(1234 + rank)
  eng.actions.copy_(torch.randint(0, 4, (t, n), device=dev, dtype=torch.int32, generator=g))
  eng.values.copy_(torch.randn(t, n, device=dev, generator=torch.Generator(device=dev).manual_seed(rank)))
  eng.boot_value.copy_(torch.randn(n, device=dev, generator=g))
  eng.boot_q.copy_(torch.rand(n, 20, 20, device=dev, generator=g))

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize(dev)

  # ---- device-resident arm ----
  for _ in range(max(args.warmup, 3)):
    eng.run_device()
  K = args.steps
  evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(K)]
  sampler = ClockSampler(local)
  barrier()
  sampler.start()
  for k in range(K):
    eng.run_device(evs[k])
  barrier()
  clocks = sampler.stop()
  total_ms = evs[0][0].elapsed_time(evs[-1][3])
  k1_ms = sum(e[0].elapsed_time(e[1]) for e in evs) / (K * (1 if window else t))    # per K1 launch
  k3_ms = sum(e[1].elapsed_time(e[2]) for e in evs) / K
  k4_ms = sum(e[2].elapsed_time(e[3]) for e in evs) / K
  if args.dump_outputs and rank == 0:
    dump_outputs(torch, eng, args.dump_outputs)

  # ---- host-buffer (e2e) arm: same pass through run_host() ----
  # the caller's host buffers are the engine's pinned staging arrays (filled in place once)
  hbuf = eng.host_inputs()
  hbuf["actions"][...] = eng.actions.cpu().numpy(); hbuf["values"][...] = eng.values.cpu().numpy()
  hbuf["boot_value"][...] = eng.boot_value.cpu().numpy(); hbuf["boot_q"][...] = eng.boot_q.cpu().numpy()
  h_act, h_val, h_bv, h_bq = hbuf["actions"], hbuf["values"], hbuf["boot_value"], hbuf["boot_q"]
  for _ in range(3):
    out = eng.run_host(h_act, h_val, h_bv, h_bq)
  ke = K
  e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
  barrier()
  e0.record()
  for _ in range(ke):
    out = eng.run_host(h_act, h_val, h_bv, h_bq)
  e1.record()
  barrier()
  e2e_ms = e0.elapsed_time(e1)
  checksum = float(out["R"].sum())
  parity, parity_what = parity_check(torch, eng) if rank == 0 else ("", "")
  # context for a K1 fraction above 1.0: K1 only WRITES, the roofline denominator (MEASURED_PEAKS.json) is a COPY.  A plain
  # device fill of the same buffer, timed here the same way, is the write-only bandwidth of this GPU.
  fill_gbs = None
  if rank == 0:
    try:
      buf = eng.obs.view(-1)
      if buf.dtype == torch.uint8 and buf.numel() % 4 == 0:
        buf = buf.view(torch.float32)          # torch's byte fill is not a bandwidth test; same bytes as 4-byte words
      for _ in range(2):
        buf.zero_()
      f0 = torch.cuda.Event(enable_timing=True); f1 = torch.cuda.Event(enable_timing=True)
      torch.cuda.synchronize(dev)
      f0.record()
      for _ in range(3):
        buf.zero_()
      f1.record()
      torch.cuda.synchronize(dev)
      fill_gbs = 3 * buf.numel() * buf.element_size() / (f0.elapsed_time(f1) * 1e-3) / 1e9
    except Exception:
      fill_gbs = None

  h2d_bytes, d2h_bytes, launches_per_pass = eng.h2d_bytes_per_pass, eng.d2h_bytes_per_pass, eng.launches_per_pass
  agent = None
  if not args.no_agent:
    try:
      del eng, out, hbuf, h_act, h_val, h_bv, h_bq
      torch.cuda.empty_cache()
      agent = measure_agent(torch, dist, dev, rank, world, args.agent_envs, args.agent_updates, obs=args.agent_obs)
    except Exception as e:  # the side measurement must never cost the headline line
      agent = {"error": repr(e)[:300]}

  side = {}
  if not args.no_agent:
    peak_gbs = 6535.7
    try:
      with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
        peak_gbs = float(json.load(f).get("hbm_gbs", peak_gbs))
    except Exception:
      pass
    try:
      torch.cuda.empty_cache()
      side["a3c"] = measure_a3c(torch, dist, dev, rank, world)
    except Exception as e:
      side["a3c"] = {"error": repr(e)[:300]}
    if world == 1:
      try:
        torch.cuda.empty_cache()
        side["pc_stress"] = measure_pc_stress(torch, dev, peak_gbs)
      except Exception as e:
        side["pc_stress"] = {"error": repr(e)[:300]}

  times = torch.tensor([total_ms, e2e_ms], device=dev, dtype=torch.float64)
  if world > 1:
    dist.all_reduce(times, op=dist.ReduceOp.MAX)
  total_ms, e2e_ms = times.tolist()

  if rank == 0:
    steps_per_pass = n * t
    value = world * steps_per_pass * K / (total_ms * 1e-3)
    e2e = world * steps_per_pass * ke / (e2e_ms * 1e-3)
    peaks = {}
    try:
      with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
        peaks = json.load(f)
    except Exception:
      pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    k1_bytes = n * K1_BYTES[args.obs_dtype] * (t if window else 1)
    achieved = k1_bytes / (k1_ms * 1e-3) / 1e9
    path_bytes = steps_per_pass * (K1_BYTES[args.obs_dtype] + K3_BYTES_PER_ENV_STEP + K4_BYTES_PER_ENV_STEP)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": max(args.warmup, 3),
        "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": args.obs_dtype, "data": "synthetic", "config": workload_config(args), "clocks": clocks,
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
                "d2h_bytes_per_step": d2h_bytes, "steps": ke, "ms_per_step": e2e_ms / ke,
                "api": "unreal_b200.train.rollout.RolloutTargets.run_host (pinned host in/out, copies "
                       "pipelined around the phases on a second stream; frames, pixel-change maps and PC "
                       "targets stay in HBM for the learner)", "checksum_R": checksum},
        "gpu_launches": K * launches_per_pass, "parity_check": parity, "parity_check_what": parity_what,
        "roofline": {"bound": "hbm", "kernel": ("maze_window_%s_kernel (K1, all %d steps of a pass in one launch + the state kernel)" % (
                         "cta" if args.obs_dtype == "f32" else "warp", t)) if window else (
                         "maze_cta_kernel (K1)" if args.obs_dtype == "f32" else "maze_warp_kernel (K1)"),
                     "achieved": achieved, "peak": peak,
                     "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650",
                     "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                     "algorithmic_bytes_per_launch": k1_bytes, "us_per_launch": k1_ms * 1e3,
                     "whole_pass_gbs": path_bytes / (total_ms / K * 1e-3) / 1e9,
                     "whole_pass_frac": path_bytes / (total_ms / K * 1e-3) / 1e9 / peak,
                     "k3_us": k3_ms * 1e3, "k4_us": k4_ms * 1e3,
                     "k4_gbs": n * 65600 / (k4_ms * 1e-3) / 1e9,
                     "write_only_fill_gbs": fill_gbs,
                     "note": "K1 is a pure writer; `peak` is the measured COPY bandwidth (read + write), which a write-only "
                             "stream can exceed: `write_only_fill_gbs` is torch's zero_() over the same obs buffer, timed in "
                             "this run"},
    }
    traffic_file = os.path.join(ROOT, "profiles", "k1_traffic.json")
    if os.path.exists(traffic_file):
      try:
        with open(traffic_file) as f:
          line["roofline"]["traffic"] = json.load(f).get(args.obs_dtype if window else args.obs_dtype + "_per_step")
      except Exception:
        pass
    if agent is not None:
      if not args.no_cpu_baseline and world == 1 and "error" not in agent:
        try:
          agent["cpu_baseline"] = agent_cpu_baseline()
        except Exception as e:
          agent["cpu_baseline"] = {"error": repr(e)[:200]}
      line["agent"] = agent
    line.update(side)
    if not args.no_cpu_baseline and world == 1:
      from oracle import cpu_path
      procs = cpu_path.host_cores()
      v, steps, sample = cpu_throughput(args.cpu_seconds, procs)
      line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": procs, "kind": "port", "sample": sample}
    print(json.dumps(line), flush=True)
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()
  return 0


def main():
  args = parse()
  if args.impl == "reference":
    return run_reference(args)
  return run_b200(args)


if __name__ == "__main__":
  sys.exit(main())
