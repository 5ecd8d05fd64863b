"""Write ceiling of the f32 window render: how fast can anything fill the [T, N, 84, 84, 3] f32 rollout frame buffer
(T = 20, N = 4096: 6.94 GB) on this GPU?

    python scripts/k1_store_ceiling.py [--envs 4096] [--steps 20] [--reps 20] [--out FILE]

Times, with CUDA events over --reps back-to-back launches each, after a warm-up:
  cta_per_item   constant 16-byte words in maze_window_cta_kernel's address order, one 256-thread CTA per item
  persistent     the same stores from a persistent grid (8 CTAs per SM) walking the time-major items in order
  torch_zero     torch's zero_() over the same buffer
  render         unreal_maze_window itself on the same buffer (the render + its state kernel)
and prints one JSON line with the card's name, power limit and clocks.  scripts/k1_store_ceiling.cu is compiled
into a temporary directory.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _compile(tmp):
  nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
  so = os.path.join(tmp, "k1_store_ceiling.so")
  subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-shared", "-Xcompiler", "-fPIC",
                         os.path.join(ROOT, "scripts", "k1_store_ceiling.cu"), "-o", so])
  lib = ctypes.CDLL(so)
  lib.k1_ceiling_cta_per_item.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p]
  lib.k1_ceiling_persistent.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_void_p]
  return lib


def _card():
  try:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                          "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    name, power, sm, sm_max = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power, "sm_clock": sm, "sm_clock_max": sm_max}
  except Exception as e:  # the numbers still stand; say why the card is missing
    return {"error": repr(e)[:200]}


def main():
  p = argparse.ArgumentParser()
  p.add_argument("--envs", type=int, default=4096)
  p.add_argument("--steps", type=int, default=20)
  p.add_argument("--reps", type=int, default=20)
  p.add_argument("--out", default=None)
  args = p.parse_args()
  import torch
  from unreal_b200 import _lib, kernels as K
  _lib.require_device()
  dev = torch.device("cuda", 0)
  n, t, reps = args.envs, args.steps, args.reps
  items = n * t
  buf = torch.empty(t, n, 84, 84, 3, dtype=torch.float32, device=dev)
  nbytes = buf.numel() * 4
  sms = torch.cuda.get_device_properties(dev).multi_processor_count
  state = K.MazeState(n, dev)
  actions = torch.randint(0, 4, (t, n), dtype=torch.int32, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
  pc = torch.empty(t, n, 20, 20, dtype=torch.float32, device=dev)
  rec = torch.empty(t, n, dtype=torch.int64, device=dev)

  with tempfile.TemporaryDirectory() as tmp:
    lib = _compile(tmp)

    def stream():
      return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    shapes = {
        "cta_per_item": lambda: lib.k1_ceiling_cta_per_item(buf.data_ptr(), items, stream()),
        "persistent": lambda: lib.k1_ceiling_persistent(buf.data_ptr(), items, 8 * sms, stream()),
        "torch_zero": lambda: buf.zero_(),
        "render": lambda: K.maze_window(state, actions, obs=buf, pc=pc, frame_rec=rec, auto_reset=True),
    }
    res = {}
    for name, fn in shapes.items():
      for _ in range(3):
        fn()
      torch.cuda.synchronize(dev)
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      for _ in range(reps):
        fn()
      e1.record()
      torch.cuda.synchronize(dev)
      us = e0.elapsed_time(e1) * 1e3 / reps
      res[name] = {"us": us, "frame_gbs": nbytes / (us * 1e-6) / 1e9}
    # the render writes the 20x20 maps and the records as well (1.9 % more bytes than the frames)
    res["render"]["all_bytes_gbs"] = (nbytes + pc.numel() * 4 + rec.numel() * 8) / (res["render"]["us"] * 1e-6) / 1e9
  best = min(v["us"] for k, v in res.items() if k != "render")
  line = {"what": "f32 window render write ceiling", "envs": n, "steps": t, "frame_bytes": nbytes, "reps": reps,
          "timing": "CUDA events over %d back-to-back launches per shape, after 3 warm-up launches" % reps,
          "card": _card(), "device": torch.cuda.get_device_name(dev), "shapes": res,
          "render_over_best_ceiling": res["render"]["us"] / best}
  print(json.dumps(line), flush=True)
  if args.out:
    with open(args.out, "a") as f:
      f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
  main()
