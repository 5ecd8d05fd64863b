"""UnrealModel(encoder_precision='bf16x3'): conv1 and conv2 forward on split-bf16 operands (a = a_hi + a_lo, three
tcgen05 passes a_hi.b_hi + a_hi.b_lo + a_lo.b_hi into one fp32 accumulator).

  * the split kernels alone against fp64 convolutions of the fp32 operands, against the bf16 kernels, and with zero lo
    operands bit for bit equal to the bf16 kernels;
  * the model against the split-emulating oracle (tests/encoder_split_oracle.py) and against the vectors of the
    reference's own model.py, which the split brings from 2e-1 to 3e-2 on sampled gradient entries;
  * every encoder user in split mode: cell tables against dense frames, the Trainer's CUDA graphs against its eager run,
    the fused Evaluator against the generic loop.
"""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
HERE = os.path.dirname(os.path.abspath(__file__))


def _model(seed=0, n=3, A=4, G=0, precision='bf16x3'):
  from unreal_b200.environment.environment import Environment
  from unreal_b200.model.model import UnrealModel
  Environment.action_size = -1
  return UnrealModel(A, G, -1, True, True, True, True, 0.05, 0.001, DEV, {'segnet_mode': 0}, (84, 84), True, 0, 0.0, 0.0,
                     num_envs=n, seed=seed, encoder_precision=precision)


def _conv64(x, w, b, stride):
  """relu(conv2d(x, w) + b) in float64; x NHWC, w HWIO -> NHWC."""
  y = torch.nn.functional.conv2d(x.double().permute(0, 3, 1, 2), w.double().permute(3, 2, 0, 1), b.double(), stride=stride)
  return torch.relu(y).permute(0, 2, 3, 1)


def _operands(s, seed):
  g = torch.Generator(device=DEV).manual_seed(seed)
  w1 = (torch.rand(8, 8, 3, 16, device=DEV, generator=g) - 0.5) * 0.3
  b1 = (torch.rand(16, device=DEV, generator=g) - 0.5) * 0.1
  w2 = (torch.rand(4, 4, 16, 32, device=DEV, generator=g) - 0.5) * 0.3
  b2 = (torch.rand(32, device=DEV, generator=g) - 0.5) * 0.1
  return g, w1, b1, w2, b2


def _cells(s):
  from oracle import unreal_oracle as O
  free = [(x, y) for y in range(7) for x in range(7) if not O.WALLS[y, x]]
  idx = torch.arange(s, device=DEV) % len(free)
  frames = torch.from_numpy(np.stack([O.maze_render(x, y) for x, y in free]).astype(np.float32)).to(DEV)
  return torch.tensor(free, dtype=torch.int32, device=DEV)[idx].contiguous(), frames[idx]


def _samples(s):
  """Sample count of a parameter: a number, or one of the multi-item sizes of test_gpu_model (several work items per
  CTA of the persistent conv kernels, derived from the SM count)."""
  from test_gpu_model import conv_multi_item_sizes, items_per_cta
  if isinstance(s, int):
    return s
  n = dict(zip(("past-one-wave", "8-items-per-cta"), conv_multi_item_sizes()))[s]
  assert items_per_cta(n) >= (8 if s == "8-items-per-cta" else 2)
  return n


SIZES = [1, 3, 129, "past-one-wave", "8-items-per-cta", 20480]


def _frames(kind, s, g):
  if kind == "u8":
    u8 = torch.randint(0, 256, (s, 84, 84, 3), device=DEV, dtype=torch.uint8, generator=g)
    return u8, u8.float() / 255.0
  f = torch.rand(s, 84, 84, 3, device=DEV, generator=g)
  return f, f


# ---- the kernels ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("s", SIZES)
@pytest.mark.parametrize("source", ["f32", "u8", "cells"])
def test_split_conv1_is_30x_closer_to_fp64_than_bf16(source, s):
  from unreal_b200 import kernels as K
  s = _samples(s)
  g, w1, b1, _, _ = _operands(s, 11 + s)
  w_hi, w_lo = K.split_bf16(w1)
  t_hi, t_lo = K.conv1_w_planes(w_hi), K.conv1_w_planes(w_lo)
  if source == "cells":
    pos, x32 = _cells(s)
    hi, lo = K.conv1_fwd_maze_split(pos, t_hi, t_lo, b1)
    base = K.conv1_fwd_maze(pos, t_hi, b1)
  else:
    x, x32 = _frames(source, s, g)
    xh, xl = K.s2d_frames_split(x)
    assert torch.equal(xh, K.s2d_frames(x))                                     # the hi planes are today's planes
    hi, lo = K.conv1_fwd_split(xh, xl, t_hi, t_lo, b1)
    base = K.conv_fwd(xh, 1, t_hi, b1)
  ref = _conv64(x32, w1, b1, 4)
  err_split = float((hi.double() + lo.double() - ref).abs().max())
  err_bf16 = float((base.double() - ref).abs().max())
  print("conv1 %s S=%d: |split - fp64| %.3g  |bf16 - fp64| %.3g" % (source, s, err_split, err_bf16))
  assert err_split * 30 <= err_bf16, (err_split, err_bf16)
  # reconstruction: hi + lo is the fp32 result to ~2^-16 of its scale, lo is a rounding residual of hi
  assert err_split <= 2 ** -14 * float(ref.abs().max())
  assert bool((lo.float().abs() <= hi.float().abs() * 2 ** -8 + 1e-30).all())


@pytest.mark.parametrize("s", SIZES)
def test_split_conv2_is_30x_closer_to_fp64_than_bf16(s):
  """conv2 writes h2 as bf16 in both modes, so both are compared with the correctly rounded fp64 result: the split
  kernel misses it only where the fp32 error crosses a rounding boundary."""
  from unreal_b200 import kernels as K
  s = _samples(s)
  g, _, _, w2, b2 = _operands(s, 21 + s)
  h1 = torch.relu(torch.randn(s, 20, 20, 16, device=DEV, generator=g))
  h_hi, h_lo = K.split_bf16(h1)
  w_hi, w_lo = K.split_bf16(w2)
  got = K.conv2_fwd_split(h_hi, h_lo, K.conv_taps(w_hi, 2), K.conv_taps(w_lo, 2), b2)
  base = K.conv_fwd(h_hi, 2, K.conv_taps(w_hi, 2), b2)
  ref = _conv64(h1, w2, b2, 2).to(torch.bfloat16).double()
  err_split = float((got.double() - ref).abs().mean())
  err_bf16 = float((base.double() - ref).abs().mean())
  print("conv2 S=%d: mean |split - rn(fp64)| %.3g  mean |bf16 - rn(fp64)| %.3g" % (s, err_split, err_bf16))
  assert err_split * 30 <= err_bf16, (err_split, err_bf16)


@pytest.mark.parametrize("s", SIZES)
def test_split_kernels_with_zero_lo_equal_the_bf16_kernels(s):
  from unreal_b200 import kernels as K
  s = _samples(s)
  g, w1, b1, w2, b2 = _operands(s, 31 + s)
  t1 = K.conv1_w_planes(w1.to(torch.bfloat16))
  z1 = torch.zeros_like(t1)
  x = torch.rand(s, 84, 84, 3, device=DEV, generator=g)
  xpp = K.s2d_frames(x)
  assert torch.equal(K.conv1_fwd_split(xpp, None, t1, z1, b1)[0], K.conv_fwd(xpp, 1, t1, b1))
  pos, _ = _cells(s)
  assert torch.equal(K.conv1_fwd_maze_split(pos, t1, z1, b1)[0], K.conv1_fwd_maze(pos, t1, b1))
  h1 = K.conv_fwd(xpp, 1, t1, b1)
  t2 = K.conv_taps(w2.to(torch.bfloat16), 2)
  assert torch.equal(K.conv2_fwd_split(h1, torch.zeros_like(h1), t2, torch.zeros_like(t2), b2), K.conv_fwd(h1, 2, t2, b2))


def test_s2d_lo_planes_reconstruct_the_frames():
  from unreal_b200 import kernels as K
  g = torch.Generator(device=DEV).manual_seed(5)
  for kind in ("f32", "u8"):
    x, x32 = _frames(kind, 7, g)
    hi, lo = K.s2d_frames_split(x)
    assert torch.equal(hi, K.s2d_frames(x)), kind
    # x'' [s, q, Y*21+X, e] = frame[4Y+dy, 4X+dx, c] with dy*12 + dx*3 + c = q*8 + e
    want = x32.view(7, 21, 4, 21, 4, 3).permute(0, 1, 3, 2, 4, 5).reshape(7, 441, 6, 8).permute(0, 2, 1, 3)
    rec = hi.float() + lo.float()
    assert float((rec - want).abs().max()) <= 2 ** -16 * float(want.abs().max()), kind


# ---- the model -----------------------------------------------------------------------------------------------------
def test_encoder_precision_is_a_construction_time_choice():
  from unreal_b200 import _lib
  m = _model(n=2)
  assert m.encoder_precision == 'bf16x3' and _model(n=2, precision='bf16').encoder_precision == 'bf16'
  with pytest.raises(AttributeError):
    m.encoder_precision = 'bf16'
  with pytest.raises(_lib.UnrealError):
    _model(n=2, precision='fp32')
  from test_gpu_model import _feed, _to
  feed = _to(_feed(3, 2, 2, seed=1), DEV)
  for attr in ("fused_conv", "fused_encoder"):
    m = _model(n=2)
    setattr(m, attr, False)
    m.refresh_shadow()
    with pytest.raises(_lib.UnrealError):
      m.loss_and_grads(feed)


@pytest.mark.parametrize("maze", [False, True])
def test_split_model_matches_the_split_oracle(maze):
  """As test_gpu_model.test_loss_and_gradients_match_oracle (emulating oracle), with the split encoder on both sides."""
  from encoder_split_oracle import SplitEncoderOracle
  from test_gpu_model import _feed, _to
  m = _model(seed=1, n=3)
  feed = _feed(5, 3, 4, seed=2, maze_frames=maze)
  total, parts, grad = m.loss_and_grads(_to(feed, DEV))
  got = {k: v.cpu() for k, v in m._views(grad).items()}
  params = {k: v.detach().cpu().clone() for k, v in m.named_vars().items()}
  o = SplitEncoderOracle(params, 4, 0, 0.05, 0.001, emulate_bf16=True, encoder_split=True)
  _, rparts, rgrads = o.loss_and_grads(feed)
  for k in ("policy", "value", "pc", "vr", "rp"):
    assert abs(float(parts[k]) - float(rparts[k])) <= 2e-3 * max(1.0, abs(float(rparts[k]))), k
  for k, rg in rgrads.items():
    err = float((got[k] - rg).abs().max())
    assert err <= 3e-2 * float(rg.abs().max()) + 1e-6, (k, err, float(rg.abs().max()))


@pytest.mark.parametrize("fixture", ["model_reference_golden.npz", "model_reference_golden_a3g2.npz"], ids=["maze-A4", "indoor-A3-G2"])
def test_split_model_against_vectors_from_the_references_own_model_py(fixture):
  """test_gpu_model.test_cuda_model_against_vectors_from_the_references_own_model_py in split mode: every variable's 64
  sampled gradient entries within 3e-2 (2e-1 in bf16 mode) and its norm within 2e-2 (1e-1)."""
  from oracle import model_oracle as M
  from test_encoder_split_oracle import sampled_errors, _fixture
  g, A_, G_, seed, feed = _fixture(fixture)
  m = _model(n=1, A=A_, G=G_)
  m.load_vars({k: v.numpy() for k, v in M.init_params(A_, G_, seed=seed).items()})
  f32 = lambda k: torch.from_numpy(np.asarray(g[k], dtype=np.float32)).to(DEV)          # noqa: E731
  img = lambda k: torch.from_numpy(g[k].astype(np.float32) / 255.0).to(DEV)             # noqa: E731

  def close(got, want, tol=3e-2):
    got, want = np.asarray(got.detach().float().cpu(), np.float64), np.asarray(want)
    assert np.abs(got - want).max() <= tol * max(1.0, np.abs(want).max()), (np.abs(got - want).max(), np.abs(want).max())
  m.reset_state()
  for t in range(3):
    pi, v, _ = m.run_base_policy_and_value(None, {'image': img("act_frames")[t][None]}, f32("act_lar")[t][None])
    close(pi[0], g["act_pi"][t]); close(v[0], g["act_v"][t])
  one = {'image': img("one_frame")}
  close(m.run_base_value(None, one, f32("one_lar"))[0], g["base_value"])
  close(m.run_pc_q_max(None, one, f32("one_lar"))[0], g["pc_q_max"])
  close(m.run_vr_value(None, one, f32("one_lar"))[0], g["vr_value"])
  close(m.run_rp_c(None, img("rp_frames")[None])[0], g["rp_c"])
  total, parts, grad = m.loss_and_grads(_to_dev(feed))
  close(total, g["total_loss"])
  got = {k: v.detach().cpu() for k, v in m._views(grad).items()}
  errs = sampled_errors(got, g, A_, G_)
  for name, _, _ in M.variable_specs(A_, G_):
    norm = float(np.linalg.norm(got[name].double().numpy()))
    nerr = abs(norm - float(g["grad_norm_" + name])) / float(g["grad_norm_" + name])
    print("bf16x3 %-16s sampled rel L2 err %.4f  norm rel err %.4f" % (name, errs[name], nerr))
    assert errs[name] <= 3e-2, (name, errs[name])
    assert nerr <= 2e-2, (name, nerr)


def _to_dev(feed):
  return {k: {kk: vv.to(DEV) for kk, vv in v.items()} for k, v in feed.items()}


def test_split_cell_tables_equal_the_dense_encoder_on_rendered_frames():
  """Split mode: the 49-cell tables (render-fused conv1, two passes) against the dense encoder on the rendered f32 frames
  of the same cells (s2d planes with an all-zero lo, three passes): the same forward values, gradients to the bf16
  rounding of the per-cell sums."""
  from test_gpu_model import _feed, _to
  from unreal_b200 import kernels as K
  from oracle import unreal_oracle as O
  m = _model(seed=5, n=6)
  T, N, L = 5, 6, 4
  rs = np.random.RandomState(9)
  cells = np.array([(x, y) for y in range(7) for x in range(7) if not O.WALLS[y, x]], np.int32)
  feed_c = _to(_feed(T, N, L, seed=31, maze_frames=True), DEV)
  pick = lambda *lead: torch.from_numpy(cells[rs.randint(0, len(cells), size=lead)]).to(DEV)   # noqa: E731
  feed_c["base"]["images"] = pick(T, N); feed_c["pc"]["images"] = pick(L, N); feed_c["vr"]["images"] = pick(L, N)
  feed_c["rp"]["images"] = pick(N, 3)
  feed_f = {k: dict(v) for k, v in feed_c.items()}
  for k in feed_f:
    c = feed_f[k]["images"]
    feed_f[k]["images"] = K.maze_render(c.reshape(-1, 2).contiguous(), dtype=torch.float32).view(*c.shape[:-1], 84, 84, 3)
  out = {}
  for name, feed in (("cells", feed_c), ("frames", feed_f)):
    total, parts, grad = m.loss_and_grads(feed)
    out[name] = ({k: float(v) for k, v in parts.items()}, {k: v.clone() for k, v in m._views(grad).items()})
  for k in out["frames"][0]:
    a, b = out["frames"][0][k], out["cells"][0][k]
    assert abs(a - b) <= 1e-5 * max(1.0, abs(a)), (k, a, b)
  for k, ref in out["frames"][1].items():
    assert float((out["cells"][1][k] - ref).abs().max()) <= 1e-2 * float(ref.abs().max()) + 1e-7, k
  res = {}
  for name, feed in (("cells", feed_c), ("frames", feed_f)):
    m.reset_state()
    pi, v, _ = m.run_base_policy_and_value(None, {'image': feed["base"]["images"][0]}, feed["base"]["lar"][0])
    res[name] = (pi.clone(), v.clone())
  for a, b in zip(res["cells"], res["frames"]):
    assert torch.allclose(a, b, rtol=1e-4, atol=1e-5)


# ---- the users: Trainer and Evaluator ------------------------------------------------------------------------------
def _trainer(env, n, seed, graphs):
  from unreal_b200.train.rmsprop_applier import RMSPropApplier
  from unreal_b200.train.trainer import Trainer
  net = _model(seed=seed, n=n, A=4 if env == 'maze' else 3)
  ap = RMSPropApplier(7e-4, decay=0.99, momentum=0.0, epsilon=0.1, clip_norm=40.0)
  kw = dict(obs_cells=True) if env == 'maze' else dict(env_args={'producer': 'table', 'seed': 2})
  tr = Trainer(0, net, 7e-4, None, ap, env, '', True, True, True, True, 0.05, 0.001, 20, 20, 0.99, 0.9, 40,
               10 ** 7, "cuda:0", {'segnet_mode': 0}, (84, 84), True, 0, np.random.RandomState(1), 50.0, 0.0, 0.0,
               num_envs=n, seeds=np.arange(n) + 11, use_graphs=graphs, **kw)
  tr.prepare()
  return tr


@pytest.mark.parametrize("env", ["maze", "synthetic"], ids=["cells", "framed"])
def test_split_trainer_graphs_equal_eager(env):
  n = 5
  tr_e, tr_g = _trainer(env, n, 2, False), _trainer(env, n, 2, True)
  for tr in (tr_e, tr_g):
    while not tr.experience.is_full():
      tr.process(None, 0)
  for it in range(4):
    de, _ = tr_e.process(None, 0)
    dg, _ = tr_g.process(None, 0)
    assert de == dg
    assert torch.equal(tr_e.last_feed['base']['a'], tr_g.last_feed['base']['a']), it
    for k in ('pc', 'vr', 'rp'):
      assert torch.equal(tr_e.last_feed[k]['start'], tr_g.last_feed[k]['start']), (it, k)
  assert tr_g._ugraph is not None, "the update graph must have been captured"
  assert torch.allclose(tr_e.local_network.flat, tr_g.local_network.flat, rtol=1e-3, atol=1e-5)
  for k in ("total", "grad_norm"):
    assert torch.allclose(tr_e.last_losses[k].float(), tr_g.last_losses[k].float(), rtol=2e-3, atol=1e-4), k
  tr_e.stop(); tr_g.stop()


@pytest.mark.parametrize("mode", ["sample", "greedy"])
def test_split_fused_evaluator_equals_generic(mode):
  from unreal_b200.train.evaluator import Evaluator
  net = _model(seed=7, n=1)
  out = {}
  for fused in (True, False):
    ev = Evaluator(net, device=DEV, num_envs=64, mode=mode, max_episode_steps=300, use_graphs=True, fused=fused)
    assert ev.path == ('fused' if fused else 'generic')
    out[fused] = ev.run(2)
  for k in ("score", "length", "finished"):
    assert torch.equal(out[True][k], out[False][k]), k
