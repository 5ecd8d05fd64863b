"""Evaluate a trained maze agent: whole episodes of the frozen policy in M envs (unreal_b200.train.evaluator.Evaluator), one
JSON summary line on stdout.

    python scripts/evaluate.py --checkpoint agent.pt [--envs 256] [--episodes 4] [--mode sample|greedy] [--max-steps 2000]
                               [--seed 0] [--encoder-precision bf16|bf16x3]
    python scripts/evaluate.py --tf-checkpoint logs/checkpoints/checkpoint-1000000 ...

--checkpoint reads this project's format (unreal_b200.train.checkpoint.save; only the variables are used),
--tf-checkpoint the reference's TF-1 checkpoint (tf_checkpoint.load_tf_checkpoint).  Env e samples with
RandomState(seed + e).  Maze only, like scripts/train_maze.py: a greedy maze episode is deterministic, so --mode greedy
with --envs 1 is the agent's learned path.  --encoder-precision picks the encoder arithmetic the policy runs with (a
checkpoint stores variables only, not the mode it was trained in); the summary names it when it is not the default.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from unreal_b200 import _lib
from unreal_b200.model.model import UnrealModel
from unreal_b200.train import checkpoint, tf_checkpoint
from unreal_b200.train.evaluator import Evaluator

ACTIONS = 4     # maze_environment.py:11-13


def _model(use_pc, use_rp, dev, encoder_precision='bf16'):
  return UnrealModel(ACTIONS, 0, -1, True, use_pc, True, use_rp, 0.05, 0.001, dev, {'segnet_mode': 0}, (84, 84), False, 0,
                     0.0, 0.0, num_envs=1, seed=0, encoder_precision=encoder_precision)


def _reject(msg):
  raise _lib.UnrealError("checkpoint rejected: " + msg)


def load_checkpoint(path, dev, encoder_precision='bf16'):
  """This project's checkpoint -> UnrealModel with its variables; every name and shape is checked before anything is
  loaded (as checkpoint.validate does for a whole agent)."""
  d = torch.load(path, map_location="cpu", weights_only=True)
  if not isinstance(d, dict) or d.get("format") != checkpoint.FORMAT:
    _reject("not an unreal_b200 checkpoint (format %r)" % (d.get("format") if isinstance(d, dict) else None,))
  var = d.get("variables")
  if not isinstance(var, dict) or not all(isinstance(v, torch.Tensor) for v in var.values()):
    _reject("no variables")
  net = _model("W_pc_fc1" in var, "W_rp_fc1" in var, dev, encoder_precision)
  want = {k: tuple(v.shape) for k, v in net.named_vars().items()}
  if set(var) != set(want):
    _reject("variables %s do not match a %d-action maze model's %s" % (sorted(var), ACTIONS, sorted(want)))
  for k, shape in want.items():
    if tuple(var[k].shape) != shape or var[k].dtype != torch.float32:
      _reject("variable %s is %s %s, the model's is %s float32" % (k, tuple(var[k].shape), var[k].dtype, shape))
  net.load_vars({k: v.numpy() for k, v in var.items()})
  return net


def load_tf(prefix, dev, encoder_precision='bf16'):
  names = tf_checkpoint.read_tf_checkpoint(prefix)
  leaf = {k.rsplit("/", 1)[-1] for k in names}
  net = _model("W_pc_fc1" in leaf, "W_rp_fc1" in leaf, dev, encoder_precision)
  tf_checkpoint.load_tf_checkpoint(net, prefix)
  return net


def main(argv=None):
  p = argparse.ArgumentParser()
  src = p.add_mutually_exclusive_group(required=True)
  src.add_argument("--checkpoint", help="unreal_b200 checkpoint (checkpoint.save)")
  src.add_argument("--tf-checkpoint", help="prefix of a TF-1 checkpoint of the reference (<prefix>.index + data)")
  p.add_argument("--envs", type=int, default=256)
  p.add_argument("--episodes", type=int, default=4, help="episodes per env")
  p.add_argument("--mode", default="sample", choices=["sample", "greedy"])
  p.add_argument("--max-steps", type=int, default=2000, help="step cap of an episode")
  p.add_argument("--seed", type=int, default=0, help="env e samples with RandomState(seed + e)")
  p.add_argument("--encoder-precision", default="bf16", choices=["bf16", "bf16x3"],
                 help="bf16x3: split-bf16 operands in the encoder's forward convolutions (fp32-grade products)")
  args = p.parse_args(argv)
  dev = torch.device("cuda", 0)
  if args.checkpoint:
    net = load_checkpoint(args.checkpoint, dev, args.encoder_precision)
  else:
    net = load_tf(args.tf_checkpoint, dev, args.encoder_precision)
  ev = Evaluator(net, 'maze', '', num_envs=args.envs, seeds=args.seed + np.arange(args.envs), mode=args.mode,
                 max_episode_steps=args.max_steps, device=dev)
  summary = ev.run(args.episodes)["summary"]
  summary["checkpoint"] = args.checkpoint or args.tf_checkpoint
  summary["seed"] = args.seed
  if args.encoder_precision != "bf16":
    summary["encoder_precision"] = args.encoder_precision
  sys.stdout.write(json.dumps(summary) + "\n")
  sys.stdout.flush()
  return summary


if __name__ == "__main__":
  main()
