"""Evaluation step: the fused maze path (acting GEMM + cell / heads + unreal_maze_eval_act) against the generic loop (the
public acting step, choose_action, K1, torch accounting) on the same untrained model and maze, cell observations, both
captured into CUDA graphs.  An untrained policy runs every episode to the step cap, so every step is a full step.

    python scripts/eval_bench.py [--envs 1024,8192] [--cap 512] [--repeats 5] [--out profiles/eval_bench.json]

Per env count: both evaluators are built, warmed up (one run each: the eager first chunk + the capture), then timed
alternately `--repeats` times; a run of one episode per env is cap / 32 graph replays.  Reported per path: median wall time
per step (host clock around the run, which ends in a device synchronise), env-steps/s, and the device-side launches per
step (torch.profiler over one eager chunk).  The card name and power limit are read in the same process.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from unreal_b200 import _lib
from unreal_b200.model.model import UnrealModel
from unreal_b200.train.evaluator import Evaluator


def card():
  info = {"name": torch.cuda.get_device_name(0)}
  try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30).stdout.strip().splitlines()
    info["power_limit_and_max_sm_clock"] = q[0] if q else None
  except (OSError, subprocess.SubprocessError):
    info["power_limit_and_max_sm_clock"] = None
  return info


def launches_per_step(ev):
  """CUDA kernels / memsets / copies of one eager chunk, per step (torch.profiler, a run of its own)."""
  from torch.profiler import ProfilerActivity, profile
  ev._start(1)
  torch.cuda.synchronize()
  with torch.no_grad(), profile(activities=[ProfilerActivity.CUDA]) as prof:
    ev._chunk()
    torch.cuda.synchronize()
  n = sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)
  return (n - 1) / ev.CHUNK          # minus the chunk's running-env count


def main():
  p = argparse.ArgumentParser()
  p.add_argument("--envs", default="1024,8192")
  p.add_argument("--cap", type=int, default=512)
  p.add_argument("--repeats", type=int, default=5)
  p.add_argument("--out", default=None)
  args = p.parse_args()
  _lib.require_device()
  dev = torch.device("cuda", 0)
  rows = []
  for m in [int(x) for x in args.envs.split(",")]:
    net = UnrealModel(4, 0, -1, True, True, True, True, 0.05, 0.001, dev, {'segnet_mode': 0}, (84, 84), False, 0, 0.0, 0.0,
                      num_envs=1, seed=0)
    evs = {path: Evaluator(net, 'maze', '', num_envs=m, mode='sample', max_episode_steps=args.cap, device=dev,
                           fused=(path == 'fused')) for path in ('fused', 'generic')}
    res = {path: ev.run(1) for path, ev in evs.items()}             # warm-up: eager chunk + capture + replays
    same = all(torch.equal(res['fused'][k], res['generic'][k]) for k in ("score", "length", "finished"))
    times = {path: [] for path in evs}
    summ = {}
    for _ in range(args.repeats):
      for path, ev in evs.items():                                   # alternating
        s = ev.run(1)["summary"]
        times[path].append(s["wall_s"] / ev.steps)
        summ[path] = s
    row = {"envs": m, "cap": args.cap, "results_identical": bool(same)}
    for path, ev in evs.items():
      t = float(np.median(times[path]))
      row[path] = {"us_per_step_median": t * 1e6, "us_per_step_all": [x * 1e6 for x in times[path]],
                   "env_steps_per_s": summ[path]["env_steps"] / (t * evs[path].steps),
                   "finished_episodes": int(round(summ[path]["success_rate"] * summ[path]["episodes"])),
                   "launches_per_step": launches_per_step(ev)}
    row["speedup_fused_over_generic"] = row["generic"]["us_per_step_median"] / row["fused"]["us_per_step_median"]
    rows.append(row)
    print(json.dumps(row), flush=True)
    del evs, res, net
    torch.cuda.empty_cache()
  out = {"bench": "eval_bench", "card": card(), "torch": torch.__version__, "timing": "host clock around Evaluator.run "
         "(ends in a device synchronise), divided by the steps replayed; median of the repeats", "rows": rows}
  line = json.dumps(out)
  print(line)
  if args.out:
    with open(args.out, "w") as f:
      f.write(line + "\n")


if __name__ == "__main__":
  main()
