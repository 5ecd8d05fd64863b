"""Builds libunreal_b200.so in-tree with nvcc for sm_100a (no JIT cache, no torch extension).

    python -m unreal_b200.build [--force] [--verbose]

The shared library lands next to this file so that it travels with the repo snapshot to the
GPU box.  Cross-compiles without a GPU.
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libunreal_b200.so")

SOURCES = ["api.cu", "maze.cu", "returns.cu", "rng.cu", "pixel_change.cu", "pixel_change84.cu", "replay.cu", "rmsprop.cu", "gemm_tcgen05.cu", "model_ops.cu", "conv_tcgen05.cu", "lstm_tcgen05.cu", "rollout_ops.cu", "evaluate.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-Wall,-Wno-unused-function", "--expt-relaxed-constexpr",
]


def _nvcc():
  for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
    if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
      return c
  raise RuntimeError("nvcc not found")


def _digest(paths):
  h = hashlib.sha256()
  h.update(" ".join(NVCC_FLAGS).encode())
  for p in sorted(paths):
    with open(p, "rb") as f:
      h.update(p.encode() + b"\0" + f.read())
  return h.hexdigest()


def build(force=False, verbose=False):
  os.makedirs(OBJ, exist_ok=True)
  headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
  headers.append(os.path.join(HERE, "..", "include", "unreal_b200.h"))
  srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
  stamp = os.path.join(OBJ, "stamp")
  digest = _digest(headers + srcs)
  if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == digest:
    return LIB
  nvcc = _nvcc()
  objs = []
  procs = []
  for s in srcs:
    o = os.path.join(OBJ, os.path.basename(s)[:-3] + ".o")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
    procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs.append(o)
  for s, p in procs:
    out, _ = p.communicate()
    if verbose or p.returncode != 0:
      sys.stderr.write(out)
    if p.returncode != 0:
      raise RuntimeError("nvcc failed on %s" % s)
  cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
  subprocess.check_call(cmd)
  with open(stamp, "w") as f:
    f.write(digest)
  return LIB


if __name__ == "__main__":
  print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
