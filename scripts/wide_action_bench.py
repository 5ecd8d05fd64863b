"""Cost of 8..15 actions (the 16-channel pixel-control head and the 15-wide policy / value head kernels) against the
narrow builds, one JSON document on stdout (or --out):

  * the pixel-control tower, forward + backward (PcTowerFusedFn: pc_fc1 GEMM, deconv + loss, the two backward
    convolutions, pc_fc1's gradients) at S samples: A = 4 (8-channel head, plane-major gradient) against A = 12
    (16-channel head, conv2-geometry gradient);
  * the A3C head loss forward + backward (A3CHeadLossFn) at S rows: A = 7 against A = 15, and at A = 15 the torch ops the
    model ran before the 15-wide kernels existed;
  * a FrameTrainer update (table producer, uint8 frames, CUDA graphs) at --envs envs: A = 3 against A = 12.

Device time from CUDA events after warm-up, median over alternating windows (--rounds).  The GPU's name and power limit
are read in the same run and recorded with the numbers.

    python scripts/wide_action_bench.py [--samples 20480] [--envs 1024] [--out profiles/r4_wide_actions.json]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

DEV = torch.device("cuda", 0)


def _gpu():
  info = {"name": torch.cuda.get_device_name(0)}
  try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30).stdout.strip().splitlines()
    info["power_limit, max_sm_clock"] = q[0] if q else None
  except (OSError, subprocess.SubprocessError):
    info["power_limit, max_sm_clock"] = None
  return info


def _time_us(fn, reps):
  fn()
  torch.cuda.synchronize()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(reps):
    fn()
  e1.record()
  torch.cuda.synchronize()
  return e0.elapsed_time(e1) / reps * 1e3


def _alternate(fns, reps, rounds):
  times = {k: [] for k in fns}
  for _ in range(rounds):
    for k, fn in fns.items():
      times[k].append(_time_us(fn, reps))
  return {k: round(float(np.median(v)), 2) for k, v in times.items()}


def _model(a, n=4):
  from unreal_b200.environment.environment import Environment
  from unreal_b200.model.model import UnrealModel
  Environment.action_size = -1
  return UnrealModel(a, 0, -1, True, True, True, True, 0.05, 0.001, DEV, {'segnet_mode': 0}, (84, 84), True, 0, 0.0, 0.0,
                     num_envs=n, seed=0)


def pc_tower(a, s):
  from unreal_b200.model.layers import PcTowerFusedFn
  m = _model(a)
  g = torch.Generator(device=DEV).manual_seed(a)
  p = {k: v.detach().clone().requires_grad_(True) for k, v in m.named_vars().items()}
  h = torch.randn(s, 256, device=DEV, generator=g).requires_grad_(True)
  act = torch.randint(0, a, (s,), device=DEV, dtype=torch.int32, generator=g)
  tgt = torch.rand(s, 400, device=DEV, generator=g)
  msk = torch.ones(s, device=DEV)
  taps, b, lin = (m.pc_taps16, m.pc_b16, m.pc_lin_taps) if a > 7 else (m.pc_taps, m.pc_b8, m.pc_w_planes)
  leaves = [h] + [p[k] for k in ("W_pc_fc1", "b_pc_fc1", "W_pc_deconv_v", "b_pc_deconv_v", "W_pc_deconv_a", "b_pc_deconv_a")]

  def step():
    loss = PcTowerFusedFn.apply(h, m.v16["W_pc_fc1"], p["W_pc_fc1"], p["b_pc_fc1"], taps, b, lin, p["W_pc_deconv_v"],
                                p["b_pc_deconv_v"], p["W_pc_deconv_a"], p["b_pc_deconv_a"], act, tgt, msk, a, 0.05)
    torch.autograd.grad(loss, leaves)
  return step


def heads(a, m, torch_ops=False):
  from unreal_b200.model.layers import A3CHeadLossFn
  g = torch.Generator(device=DEV).manual_seed(a)
  h = torch.randn(m, 256, device=DEV, generator=g).requires_grad_(True)
  wp = (torch.randn(256, a, device=DEV, generator=g) * 0.1).requires_grad_(True)
  bp = torch.zeros(a, device=DEV, requires_grad=True)
  wv = (torch.randn(256, 1, device=DEV, generator=g) * 0.1).requires_grad_(True)
  bv = torch.zeros(1, device=DEV, requires_grad=True)
  act = torch.randint(0, a, (m,), device=DEV, dtype=torch.int32, generator=g)
  onehot = torch.nn.functional.one_hot(act.long(), a).float()
  adv, ret, mask = torch.randn(m, device=DEV, generator=g), torch.randn(m, device=DEV, generator=g), torch.ones(m, device=DEV)
  leaves = [h, wp, bp, wv, bv]

  def kernel_step():
    pol, val, _ = A3CHeadLossFn.apply(h, wp, bp, wv, bv, act, adv, ret, mask, 0.001, 0.25)
    torch.autograd.grad(pol + val, leaves)

  def torch_step():        # UnrealModel.loss's base-loss branch without the fused heads
    pi = torch.softmax(h @ wp + bp, -1); v = (h @ wv + bv).squeeze(-1)
    lp = torch.log(pi.clamp(1e-20, 1.0)); ent = -(pi * lp).sum(-1)
    pol = -((((lp * onehot).sum(-1)) * adv + ent * 0.001) * mask).sum()
    val = 0.25 * (((ret - v) ** 2) * mask).sum()
    torch.autograd.grad(pol + val, leaves)
  return torch_step if torch_ops else kernel_step


def _register_wide(a):
  from unreal_b200.environment import frame_environment as FE
  from unreal_b200.environment.environment import Environment
  Environment.register('table%d' % a, lambda name, args, tt, ti: FE.BatchedFrameEnvironment(
      FE.TableFrameProducer(args['num_envs'], args['device'], a, seed=ti), args['device']), action_size=a)


def _trainer(a, n, history):
  from unreal_b200.train.rmsprop_applier import RMSPropApplier
  from unreal_b200.train.trainer import Trainer
  net = _model(a, n)
  ap = RMSPropApplier(7e-4, decay=0.99, momentum=0.0, epsilon=0.1, clip_norm=40.0)
  if a == 3:
    env, kw = 'synthetic', dict(env_args={'producer': 'table', 'seed': 0})
  else:
    _register_wide(a)
    env, kw = 'table%d' % a, {}
  tr = Trainer(0, net, 7e-4, None, ap, env, '', True, True, True, True, 0.05, 0.001, 20, 20, 0.99, 0.9, history, 10 ** 8,
               "cuda:0", {'segnet_mode': 0}, (84, 84), True, 0, np.random.RandomState(1), 50.0, 0.0, 0.0, num_envs=n,
               seeds=np.arange(n) + 11, use_graphs=True, **kw)
  tr.prepare()
  while not tr.experience.is_full():
    tr.process(None, 0)
  for _ in range(3):                 # capture the graphs, then replay
    tr.process(None, 0)
  torch.cuda.synchronize()
  return tr


def updates(n, history, iters, rounds):
  from unreal_b200.environment.environment import Environment
  out = {}
  for a in (3, 12):
    Environment.action_size = -1
    tr = _trainer(a, n, history)
    out["A%d" % a] = tr
  res = _alternate({k: (lambda tr=tr: tr.process(None, 0)) for k, tr in out.items()}, iters, rounds)
  for tr in out.values():
    tr.stop()
  return {"envs": n, "history": history, "ms_per_update": {k: round(v / 1e3, 3) for k, v in res.items()},
          "ratio_A12_over_A3": round(res["A12"] / res["A3"], 4)}


def main():
  p = argparse.ArgumentParser()
  p.add_argument("--samples", type=int, default=20480)
  p.add_argument("--reps", type=int, default=20)
  p.add_argument("--envs", type=int, default=1024)
  p.add_argument("--history", type=int, default=100, help="replay ring per env (the update's cost does not depend on it)")
  p.add_argument("--iters", type=int, default=10, help="updates per timing window")
  p.add_argument("--rounds", type=int, default=5, help="alternating timing windows per case")
  p.add_argument("--out", default="-")
  args = p.parse_args()
  import __graft_entry__ as ge
  ge.build()
  s = args.samples
  tower = _alternate({"A4_planes_8ch_us": pc_tower(4, s), "A12_c16_16ch_us": pc_tower(12, s)}, args.reps, args.rounds)
  head = _alternate({"A7_kernels_us": heads(7, s), "A15_kernels_us": heads(15, s), "A15_torch_ops_us": heads(15, s, True)},
                    args.reps, args.rounds)
  res = {"gpu": _gpu(), "unit": "device time from CUDA events after warm-up, median over alternating windows",
         "pc_tower_fwd_bwd_at_samples": s, "pc_tower_fwd_bwd": tower,
         "a3c_head_loss_fwd_bwd_at_rows": s, "a3c_head_loss_fwd_bwd": head,
         "frame_trainer_update_table_producer": updates(args.envs, args.history, args.iters, args.rounds)}
  text = json.dumps(res, indent=1)
  if args.out != "-":
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
      f.write(text + "\n")
  print(text)


if __name__ == "__main__":
  main()
