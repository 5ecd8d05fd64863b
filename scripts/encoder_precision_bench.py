"""Cost of UnrealModel(encoder_precision='bf16x3') against the default 'bf16', one JSON document on stdout (or --out):

  * the encoder's forward kernels alone at S frames (default 20 480 = 20 steps x 1024 envs): s2d, conv1 over x'' planes,
    render-fused maze conv1, conv2 -- each in its bf16 and its split form, CUDA events over --reps launches;
  * a maze agent update (Trainer.process with CUDA graphs: 20-step rollout + update, --maze-envs cell observations);
  * a config-5 update (the synthetic framed env, --frame-envs envs, uint8 frames, CUDA graphs).

The two modes run in one process and are timed in alternating windows (--rounds of them); the report gives the median
per mode.  The GPU's name and power limit are recorded with the numbers.

    python scripts/encoder_precision_bench.py [--frames 20480] [--maze-envs 8192] [--frame-envs 1024] [--out f.json]
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


def kernels(s, reps, rounds):
  from unreal_b200 import kernels as K
  g = torch.Generator(device=DEV).manual_seed(0)
  frames = torch.randint(0, 256, (s, 84, 84, 3), device=DEV, dtype=torch.uint8, generator=g)
  pos = torch.randint(0, 7, (s, 2), device=DEV, dtype=torch.int32, generator=g)
  w1 = (torch.rand(8, 8, 3, 16, device=DEV, generator=g) - 0.5) * 0.3
  w2 = (torch.rand(4, 4, 16, 32, device=DEV, generator=g) - 0.5) * 0.3
  b1, b2 = torch.zeros(16, device=DEV), torch.zeros(32, device=DEV)
  w1h, w1l = K.split_bf16(w1)
  w2h, w2l = K.split_bf16(w2)
  t1h, t1l, t2h, t2l = K.conv1_w_planes(w1h), K.conv1_w_planes(w1l), K.conv_taps(w2h, 2), K.conv_taps(w2l, 2)
  xh, xl = K.s2d_frames_split(frames)
  h1h, h1l = K.conv1_fwd_split(xh, xl, t1h, t1l, b1)
  pos49 = torch.tensor([[x, y] for y in range(7) for x in range(7)], dtype=torch.int32, device=DEV)
  cases = {
      "s2d_u8": (lambda: K.s2d_frames(frames), lambda: K.s2d_frames_split(frames)),
      "conv1_planes": (lambda: K.conv_fwd(xh, 1, t1h, b1), lambda: K.conv1_fwd_split(xh, xl, t1h, t1l, b1)),
      "conv1_planes_exact_input": (lambda: K.conv_fwd(xh, 1, t1h, b1), lambda: K.conv1_fwd_split(xh, None, t1h, t1l, b1)),
      "conv1_maze": (lambda: K.conv1_fwd_maze(pos, t1h, b1), lambda: K.conv1_fwd_maze_split(pos, t1h, t1l, b1)),
      "conv1_maze_49_cells": (lambda: K.conv1_fwd_maze(pos49, t1h, b1), lambda: K.conv1_fwd_maze_split(pos49, t1h, t1l, b1)),
      "conv2": (lambda: K.conv_fwd(h1h, 2, t2h, b2), lambda: K.conv2_fwd_split(h1h, h1l, t2h, t2l, b2)),
  }
  out = {}
  for name, (fb, fs) in cases.items():
    tb, ts = [], []
    for _ in range(rounds):
      tb.append(_time_us(fb, reps)); ts.append(_time_us(fs, reps))
    b, sp = float(np.median(tb)), float(np.median(ts))
    out[name] = {"bf16_us": round(b, 2), "bf16x3_us": round(sp, 2), "ratio": round(sp / b, 3)}
  return out


def _trainer(env, n, precision, history):
  from unreal_b200.environment.environment import Environment
  from unreal_b200.model.model import UnrealModel
  from unreal_b200.train.rmsprop_applier import RMSPropApplier
  from unreal_b200.train.trainer import Trainer
  Environment.action_size = -1
  a = 4 if env == 'maze' else 3
  net = UnrealModel(a, 0, -1, True, True, True, True, 0.05, 0.001, DEV, {'segnet_mode': 0}, (84, 84), True, 0, 0.0, 0.0,
                    num_envs=n, seed=0, encoder_precision=precision)
  ap = RMSPropApplier(7e-4, decay=0.99, momentum=0.0, epsilon=0.1, clip_norm=40.0)
  kw = dict(obs_cells=True) if env == 'maze' else dict(env_args={'producer': 'table', 'seed': 0})
  tr = Trainer(0, net, 7e-4, None, ap, env, '', True, True, True, True, 0.05, 0.001, 20, 20, 0.99, 0.9, history, 10 ** 8,
               "cuda:0", {'segnet_mode': 0}, (84, 84), True, 0, np.random.RandomState(1), 50.0, 0.0, 0.0, num_envs=n,
               seeds=np.arange(n) + 11, use_graphs=True, **kw)
  tr.prepare()
  while not tr.experience.is_full():
    tr.process(None, 0)
  for _ in range(3):                 # capture both graphs, then replay
    tr.process(None, 0)
  torch.cuda.synchronize()
  return tr


def updates(env, n, history, iters, rounds):
  trs = {p: _trainer(env, n, p, history) for p in ("bf16", "bf16x3")}
  times = {p: [] for p in trs}
  for _ in range(rounds):
    for p, tr in trs.items():
      times[p].append(_time_us(lambda: tr.process(None, 0), iters) / 1e3)
  for tr in trs.values():
    tr.stop()
  b, s = float(np.median(times["bf16"])), float(np.median(times["bf16x3"]))
  return {"envs": n, "history": history, "bf16_ms_per_update": round(b, 3), "bf16x3_ms_per_update": round(s, 3),
          "ratio": round(s / b, 4), "windows_bf16_ms": [round(t, 3) for t in times["bf16"]],
          "windows_bf16x3_ms": [round(t, 3) for t in times["bf16x3"]]}


def main():
  p = argparse.ArgumentParser()
  p.add_argument("--frames", type=int, default=20480)
  p.add_argument("--reps", type=int, default=50)
  p.add_argument("--maze-envs", type=int, default=8192)
  p.add_argument("--frame-envs", type=int, default=1024)
  p.add_argument("--history", type=int, default=100, help="replay ring per env (the update's cost does not depend on it)")
  p.add_argument("--iters", type=int, default=10, help="updates per timing window")
  p.add_argument("--rounds", type=int, default=5, help="alternating timing windows per mode")
  p.add_argument("--out", default="-")
  args = p.parse_args()
  import __graft_entry__ as ge
  ge.build()
  res = {"gpu": _gpu(), "unit": "device time from CUDA events, median over alternating windows",
         "kernels_at_frames": args.frames, "kernels": kernels(args.frames, args.reps, args.rounds),
         "maze_agent_update_cells": updates('maze', args.maze_envs, args.history, args.iters, args.rounds),
         "config5_update_frames": updates('synthetic', args.frame_envs, args.history, args.iters, args.rounds)}
  text = json.dumps(res, indent=1)
  if args.out == "-":
    print(text)
  else:
    with open(args.out, "w") as f:
      f.write(text + "\n")
    print(text)


if __name__ == "__main__":
  main()
