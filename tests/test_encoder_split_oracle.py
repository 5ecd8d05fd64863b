"""CPU: the split-bf16 encoder (UnrealModel(encoder_precision='bf16x3'), restated by tests/encoder_split_oracle.py) against
the vectors of the reference's own model.py (tests/golden/model_reference_golden*.npz, fp32 arithmetic throughout).

With every operand in bf16 the sampled gradient entries of conv1 are 12-17 % off on maze-A4; with the encoder's forward
operands as hi + lo pairs (and everything else, the backward pass included, as the bf16 path rounds it) every sampled
gradient of the encoder is within 1e-2 on both fixtures, and so is every variable on maze-A4."""
import os

import numpy as np
import pytest
import torch

from oracle import model_oracle as M
from encoder_split_oracle import SplitEncoderOracle

HERE = os.path.dirname(os.path.abspath(__file__))


def _fixture(name):
  g = np.load(os.path.join(HERE, "golden", name))
  A, G, seed, T, Lp, Lv = (int(x) for x in g["meta"])
  f32 = lambda k: torch.from_numpy(np.asarray(g[k], dtype=np.float32))          # noqa: E731
  img = lambda k: torch.from_numpy(g[k].astype(np.float32) / 255.0)             # noqa: E731
  ones = lambda n: torch.ones(n, 1)                                             # noqa: E731
  feed = {"base": dict(images=img("base_frames")[:, None], lar=f32("base_lar")[:, None], a=f32("base_a")[:, None],
                       adv=f32("base_adv")[:, None], R=f32("base_R")[:, None], mask=ones(T), c0=f32("base_c0"), h0=f32("base_h0")),
          "pc": dict(images=img("pc_frames")[:, None], lar=f32("pc_lar")[:, None], a=f32("pc_a")[:, None], R=f32("pc_R")[:, None],
                     mask=ones(Lp)),
          "vr": dict(images=img("vr_frames")[:, None], lar=f32("vr_lar")[:, None], R=f32("vr_R")[:, None], mask=ones(Lv)),
          "rp": dict(images=img("rp_train_frames")[None], c=f32("rp_c_target"))}
  return g, A, G, seed, feed


def sampled_errors(grads, g, A, G):
  """Relative L2 error of the 64 sampled gradient entries of every variable, as the GPU reference-vector test computes it."""
  out = {}
  for name, _, _ in M.variable_specs(A, G):
    have = grads[name].reshape(-1).double().numpy()[g["grad_idx_" + name]]
    want = g["grad_val_" + name]
    out[name] = float(np.linalg.norm(have - want) / max(np.linalg.norm(want), 1e-3 * float(g["grad_norm_" + name])))
  return out


ENCODER = ("W_base_conv1", "b_base_conv1", "W_base_conv2", "b_base_conv2")


# indoor-A3-G2: the encoder's four variables are within 1e-2, but the biases of fc1 and pc_fc1 stay at 1.2 % -- bf16
# rounding of the layers after the encoder (fc1's input and output, the LSTM, pc_fc1), which the split does not touch
@pytest.mark.parametrize("fixture,others_tol", [("model_reference_golden.npz", 1e-2), ("model_reference_golden_a3g2.npz", 1.5e-2)],
                         ids=["maze-A4", "indoor-A3-G2"])
def test_split_encoder_oracle_against_the_reference_vectors(fixture, others_tol):
  g, A, G, seed, feed = _fixture(fixture)
  p = M.init_params(A, G, seed=seed)
  errs = {}
  for split in (False, True):
    o = SplitEncoderOracle(p, A, G, 0.05, 0.001, emulate_bf16=True, encoder_split=split)
    _, _, grads = o.loss_and_grads(feed)
    errs[split] = sampled_errors(grads, g, A, G)
  for name in errs[True]:
    print("%-16s bf16 %.4f  bf16x3 %.4f" % (name, errs[False][name], errs[True][name]))
  assert max(errs[True][k] for k in ENCODER) <= 1e-2, errs[True]
  assert max(errs[True].values()) <= others_tol, errs[True]
  # the split is what closes the gap: conv1's filter gradient with bf16 operands is several times further off
  assert errs[False]["W_base_conv1"] >= 3 * errs[True]["W_base_conv1"]


def test_split_off_is_the_oracle_itself():
  g, A, G, seed, feed = _fixture("model_reference_golden.npz")
  p = M.init_params(A, G, seed=seed)
  _, _, ref = M.ModelOracle(p, A, G, 0.05, 0.001, emulate_bf16=True).loss_and_grads(feed)
  _, _, got = SplitEncoderOracle(p, A, G, 0.05, 0.001, emulate_bf16=True).loss_and_grads(feed)
  assert all(torch.equal(ref[k], got[k]) for k in ref)
