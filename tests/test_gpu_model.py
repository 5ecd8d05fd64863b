"""UnrealModel on the tcgen05 path against oracle/model_oracle.py (PyTorch-CPU fp32 restatement of
model/model.py, itself held at 1e-9 to vectors produced by the reference's own model.py over a TF-1 op shim: see the
oracle's header) and, in `test_cuda_model_against_vectors_from_the_references_own_model_py`, against those vectors directly.

Two comparisons, tolerances stated where they are used:
  * against the oracle with `emulate_bf16=True` (it rounds exactly the tensors the CUDA path keeps
    in bf16): forward values differ only by fp32 accumulation order -> 2e-3 relative;
  * against the plain fp32 oracle: bf16 operand rounding (2^-9 per element) -> 3e-2 relative.
Gradients additionally round dY to bf16 at each layer; they are compared per variable with
max|diff| <= 3e-2 * max|ref| against the emulating oracle, and in
relative L2 norm (<= 1e-1) against the plain fp32 one, whose forward pass itself differs.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

A = 4


def _feed(T, N, L, seed, maze_frames=False):
  rs = np.random.RandomState(seed)

  def images(*lead):
    if maze_frames:
      from oracle import unreal_oracle as O
      cells = [(x, y) for y in range(7) for x in range(7) if not O.WALLS[y, x]]
      out = np.zeros(lead + (84, 84, 3), np.float32)
      flat = out.reshape(-1, 84, 84, 3)
      for i in range(flat.shape[0]):
        x, y = cells[rs.randint(len(cells))]
        flat[i] = O.maze_render(x, y).astype(np.float32)
      return torch.from_numpy(out)
    return torch.from_numpy(rs.rand(*lead, 84, 84, 3).astype(np.float32)).to(torch.bfloat16).float()

  def lar(*lead):
    a = rs.randint(0, A, size=lead)
    out = np.zeros(lead + (A + 1,), np.float32)
    np.put_along_axis(out, a[..., None], 1.0, axis=-1)
    out[..., A] = rs.randint(-1, 2, size=lead)
    return torch.from_numpy(out)

  def onehot(*lead):
    a = rs.randint(0, A, size=lead)
    out = np.zeros(lead + (A,), np.float32)
    np.put_along_axis(out, a[..., None], 1.0, axis=-1)
    return torch.from_numpy(out)

  def mask(t, n):
    m = np.ones((t, n), np.float32)
    m[t - 2:, 0] = 0          # env 0 ended two steps early
    return torch.from_numpy(m)

  f32 = lambda *s: torch.from_numpy(rs.randn(*s).astype(np.float32))  # noqa: E731
  rp_c = np.zeros((N, 3), np.float32); rp_c[np.arange(N), rs.randint(0, 3, N)] = 1
  return {
      "base": dict(images=images(T, N), lar=lar(T, N), a=onehot(T, N), adv=f32(T, N), R=f32(T, N), mask=mask(T, N),
                   c0=f32(N, 256) * 0.1, h0=f32(N, 256) * 0.1),
      "pc": dict(images=images(L, N), lar=lar(L, N), a=onehot(L, N),
                 R=torch.from_numpy(rs.rand(L, N, 20, 20).astype(np.float32)), mask=mask(L, N)),
      "vr": dict(images=images(L, N), lar=lar(L, N), R=f32(L, N), mask=mask(L, N)),
      "rp": dict(images=images(N, 3), c=torch.from_numpy(rp_c)),
  }


def _to(feed, dev):
  return {k: {kk: vv.to(dev) for kk, vv in v.items()} for k, v in feed.items()}


def _model(dev, seed=0, n=3):
  from unreal_b200.model.model import UnrealModel
  return UnrealModel(A, 0, -1, True, True, True, True, 0.05, 0.001, dev, {'segnet_mode': 0}, (84, 84), True, 0,
                     0.0, 0.0, num_envs=n, seed=seed)


def _oracle(model, emulate):
  from oracle import model_oracle as M
  params = {k: v.detach().cpu().clone() for k, v in model.named_vars().items()}
  return M.ModelOracle(params, A, 0, 0.05, 0.001, emulate_bf16=emulate)


def test_parameter_layout():
  dev = torch.device("cuda", 0)
  m = _model(dev)
  assert m.num_parameters == 1898877 and len(m.get_vars()) == 20
  shapes = [tuple(v.shape) for v in m.get_vars()]
  assert shapes[0] == (8, 8, 3, 16) and shapes[6] == (517, 1024) and shapes[-2] == (7776, 3)


def test_im2col_col2im_match_unfold_fold():
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  g = torch.Generator(device=dev).manual_seed(0)
  for (s, h, w, c, kh, kw, st, dt) in [(3, 84, 84, 3, 8, 8, 4, torch.float32), (3, 84, 84, 3, 8, 8, 4, torch.uint8),
                                       (2, 20, 20, 16, 4, 4, 2, torch.bfloat16), (2, 20, 20, 5, 4, 4, 2, torch.float32)]:
    if dt == torch.uint8:
      x = torch.randint(0, 256, (s, h, w, c), device=dev, dtype=torch.uint8, generator=g)
      xf = (x.float() / 255.0)
    else:
      x = torch.rand(s, h, w, c, device=dev, generator=g).to(dt)
      xf = x.float()
    cols = K.im2col(x, kh, kw, st)
    oh, ow = (h - kh) // st + 1, (w - kw) // st + 1
    ref = torch.nn.functional.unfold(xf.permute(0, 3, 1, 2), (kh, kw), stride=st)       # [S, C*KH*KW, L]
    ref = ref.view(s, c, kh, kw, oh * ow).permute(0, 4, 2, 3, 1).reshape(s * oh * ow, kh * kw * c)
    assert torch.equal(cols.float(), ref.to(torch.bfloat16).float())
    back = K.col2im(cols, s, h, w, c, kh, kw, st)
    folded = torch.nn.functional.fold(
        cols.float().view(s, oh * ow, kh, kw, c).permute(0, 4, 2, 3, 1).reshape(s, c * kh * kw, oh * ow),
        (h, w), (kh, kw), stride=st).permute(0, 2, 3, 1)
    assert torch.allclose(back, folded, rtol=1e-5, atol=1e-5)


def test_acting_helpers_match_oracle():
  dev = torch.device("cuda", 0)
  m = _model(dev, seed=3, n=3)
  o = _oracle(m, True)
  feed = _feed(2, 3, 2, seed=5)
  img, lar = feed["base"]["images"], feed["base"]["lar"]
  c = torch.zeros(3, 256); h = torch.zeros(3, 256)
  for t in range(2):
    pi, v, _ = m.run_base_policy_and_value(None, {'image': img[t].to(dev)}, lar[t].to(dev))
    rpi, rv, (c, h) = o.base_forward(img[t:t + 1], lar[t:t + 1], c, h)
    assert torch.allclose(pi.cpu(), rpi[0], rtol=2e-3, atol=2e-4)
    assert torch.allclose(v.cpu(), rv[0], rtol=2e-3, atol=2e-3)
  # bootstrap value does not advance the state (model.py:687-704)
  before = [s.clone() for s in m.base_lstm_state_out]
  bv = m.run_base_value(None, {'image': img[0].to(dev)}, lar[0].to(dev))
  assert all(torch.equal(a, b) for a, b in zip(before, m.base_lstm_state_out))
  rbv = o.base_forward(img[0:1], lar[0:1], c, h)[1][0]
  assert torch.allclose(bv.cpu(), rbv, rtol=2e-3, atol=2e-3)
  qmax = m.run_pc_q_max(None, {'image': img[1].to(dev)}, lar[1].to(dev))
  rq = o.pc_forward(img[1:2], lar[1:2])[1][0]
  assert torch.allclose(qmax.cpu(), rq, rtol=2e-3, atol=2e-3)
  vr = m.run_vr_value(None, {'image': img[1].to(dev)}, lar[1].to(dev))
  assert torch.allclose(vr.cpu(), o.vr_forward(img[1:2], lar[1:2])[0], rtol=2e-3, atol=2e-3)
  # masked state reset / masked advance
  m.reset_state(torch.tensor([1, 0, 0], device=dev, dtype=torch.uint8))
  assert float(m.base_lstm_state_out[0][0].abs().max()) == 0 and float(m.base_lstm_state_out[0][1].abs().max()) > 0


@pytest.mark.parametrize("n,a", [(1, 4), (77, 3), (4099, 7)])
def test_acting_cell_with_the_heads_inside_equals_cell_then_heads(n, a):
  """unreal_lstm_cell_act_heads (the acting step's cell + policy / value heads in one launch) against unreal_lstm_cell_act_g16
  followed by the head kernel: the same state update bit for bit (active rows advanced, inactive rows untouched), the same
  pi / v to fp32 summation order, also for the inactive rows (heads of the h they hold)."""
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  g = torch.Generator(device=dev).manual_seed(n + a)
  gates = torch.randn(n, 1024, device=dev, generator=g).to(torch.bfloat16)
  c0 = torch.randn(n, 256, device=dev, generator=g); h0 = torch.randn(n, 256, device=dev, generator=g) * 0.5
  wp = torch.randn(256, a, device=dev, generator=g) * 0.1; bp = torch.randn(a, device=dev, generator=g) * 0.1
  wv = torch.randn(256, device=dev, generator=g) * 0.1; bv = torch.randn(1, device=dev, generator=g)
  act = (torch.rand(n, device=dev, generator=g) < 0.7).to(torch.uint8)
  for active in (None, act):
    c1, h1 = c0.clone(), h0.clone()
    hout = torch.empty(n, 256, device=dev)
    K.lstm_cell_act(gates, c1, h1, hout, active)
    ref = K.a3c_head(hout, wp, bp, wv, bv, want_pi=True, want_v=True)
    c2, h2 = c0.clone(), h0.clone()
    vrow = torch.full((n,), -7.0, device=dev)
    pi, v = K.lstm_cell_act_heads(gates, c2, h2, wp, bp, wv, bv, active, v_out=vrow)
    assert v.data_ptr() == vrow.data_ptr()
    assert torch.equal(c1, c2) and torch.equal(h1, h2)
    if active is not None:
      keep = act == 0
      assert torch.equal(c2[keep], c0[keep]) and torch.equal(h2[keep], h0[keep])
    assert torch.allclose(pi, ref["pi"], rtol=1e-5, atol=1e-6) and torch.allclose(v, ref["v"], rtol=1e-5, atol=1e-5)
    assert torch.allclose(pi.sum(-1), torch.ones(n, device=dev), atol=1e-5)


@pytest.mark.parametrize("maze", [False, True])
def test_loss_and_gradients_match_oracle(maze):
  dev = torch.device("cuda", 0)
  m = _model(dev, seed=1, n=3)
  feed = _feed(5, 3, 4, seed=2, maze_frames=maze)
  total, parts, grad = m.loss_and_grads(_to(feed, dev))
  got = {k: v.cpu() for k, v in m._views(grad).items()}
  for emulate, ftol, gtol in ((True, 2e-3, 3e-2), (False, 3e-2, 1e-1)):
    o = _oracle(m, emulate)
    rtotal, rparts, rgrads = o.loss_and_grads(feed)
    for k in ("policy", "value", "pc", "vr", "rp"):
      assert abs(float(parts[k]) - float(rparts[k])) <= ftol * max(1.0, abs(float(rparts[k]))), (k, emulate)
    for k, rg in rgrads.items():
      if emulate:     # element-wise: worst element against the variable's largest gradient
        err = float((got[k] - rg).abs().max())
        assert err <= gtol * float(rg.abs().max()) + 1e-6, (k, emulate, err, float(rg.abs().max()))
      else:           # against pure fp32 the forward itself differs (bf16 operands): L2-relative
        err = float((got[k] - rg).norm() / rg.norm().clamp_min(1e-12))
        assert err <= gtol, (k, emulate, err)


@pytest.mark.parametrize("fixture", ["model_reference_golden.npz", "model_reference_golden_a3g2.npz"], ids=["maze-A4", "indoor-A3-G2"])
def test_cuda_model_against_vectors_from_the_references_own_model_py(fixture):
  """The CUDA model against tests/golden/model_reference_golden.npz DIRECTLY -- vectors produced by the reference's own
  model/model.py (unmodified, over the TF-1 op shim of tests/golden/make_model_golden.py), float64: the acting outputs
  (three run_base_policy_and_value steps with the carried LSTM state, run_base_value, run_pc_q_max, run_vr_value, run_rp_c),
  every loss term of the Trainer-shaped feed, sampled gradient entries of all 20 variables, and the global gradient norm
  the reference's RMSPropApplier reported.  Tolerances are the bf16 operand rounding of the tensor-core path: 3e-2 relative on
  values and loss terms; gradients: the variable's norm within 1e-1, its 64 sampled entries within 2e-1 (L2, relative)."""
  import os
  g = np.load(os.path.join(os.path.dirname(__file__), "golden", fixture))
  A_, G_, seed, T, Lp, Lv = (int(x) for x in g["meta"])
  from oracle import model_oracle as M
  from unreal_b200.model.model import UnrealModel
  dev = torch.device("cuda", 0)
  m = UnrealModel(A_, G_, -1, True, True, True, True, 0.05, 0.001, dev, {'segnet_mode': 0}, (84, 84), True, 0, 0.0, 0.0,
                  num_envs=1, seed=0)
  m.load_vars({k: v.numpy() for k, v in M.init_params(A_, G_, seed=seed).items()})
  f32 = lambda k: torch.from_numpy(np.asarray(g[k], dtype=np.float32)).to(dev)          # noqa: E731
  img = lambda k: torch.from_numpy(g[k].astype(np.float32) / 255.0).to(dev)             # noqa: E731
  def close(got, want, tol=3e-2):
    got, want = np.asarray(got.detach().float().cpu() if isinstance(got, torch.Tensor) else got, np.float64), np.asarray(want)
    assert np.abs(got - want).max() <= tol * max(1.0, np.abs(want).max()), (np.abs(got - want).max(), np.abs(want).max())
  m.reset_state()
  for t in range(3):
    pi, v, _ = m.run_base_policy_and_value(None, {'image': img("act_frames")[t][None]}, f32("act_lar")[t][None])
    close(pi[0], g["act_pi"][t]); close(v[0], g["act_v"][t])
  c, h = m.base_lstm_state_out
  close(c, g["act_state_c"]); close(h, g["act_state_h"])
  one = {'image': img("one_frame")}
  close(m.run_base_value(None, one, f32("one_lar"))[0], g["base_value"])
  close(m.run_pc_q_max(None, one, f32("one_lar"))[0], g["pc_q_max"])
  close(m.run_vr_value(None, one, f32("one_lar"))[0], g["vr_value"])
  close(m.run_rp_c(None, img("rp_frames")[None])[0], g["rp_c"])
  ones = lambda n: torch.ones(n, 1, device=dev)                                        # noqa: E731
  feed = {"base": dict(images=img("base_frames")[:, None], lar=f32("base_lar")[:, None], a=f32("base_a")[:, None],
                       adv=f32("base_adv")[:, None], R=f32("base_R")[:, None], mask=ones(T), c0=f32("base_c0"), h0=f32("base_h0")),
          "pc": dict(images=img("pc_frames")[:, None], lar=f32("pc_lar")[:, None], a=f32("pc_a")[:, None], R=f32("pc_R")[:, None],
                     mask=ones(Lp)),
          "vr": dict(images=img("vr_frames")[:, None], lar=f32("vr_lar")[:, None], R=f32("vr_R")[:, None], mask=ones(Lv)),
          "rp": dict(images=img("rp_train_frames")[None], c=f32("rp_c_target"))}
  total, parts, grad = m.loss_and_grads(feed)
  close(total, g["total_loss"])
  for k, name in (("policy", "policy_loss"), ("value", "value_loss"), ("pc", "pc_loss"), ("vr", "vr_loss"), ("rp", "rp_loss")):
    close(parts[k], g[name])
  got = {k: v.detach().cpu().double().reshape(-1).numpy() for k, v in m._views(grad).items()}
  sq = 0.0
  for name, _, _ in M.variable_specs(A_, G_):
    want, have = g["grad_val_" + name], got[name][g["grad_idx_" + name]]
    rel = np.linalg.norm(have - want) / max(np.linalg.norm(want), 1e-3 * float(g["grad_norm_" + name]))
    print("grad sample %-16s rel L2 err %.4f" % (name, rel))
    assert rel <= 2e-1, (name, rel)                # 64 sampled entries: noisier than the whole variable's 1e-1
    assert abs(np.linalg.norm(got[name]) - float(g["grad_norm_" + name])) <= 1e-1 * float(g["grad_norm_" + name]) + 1e-9, name
    sq += float((got[name] ** 2).sum())
  assert abs(np.sqrt(sq) - float(g["update_grad_norms"][0])) <= 5e-2 * float(g["update_grad_norms"][0])


def test_update_applies_rmsprop_like_the_oracle():
  """One learner step = K6 on the flat gradient: compare with the numpy RMSProp restatement."""
  from oracle import unreal_oracle as O
  from unreal_b200.train.rmsprop_applier import RMSPropApplier
  dev = torch.device("cuda", 0)
  m = _model(dev, seed=4, n=3)
  feed = _to(_feed(4, 3, 3, seed=6), dev)
  before = m.flat.detach().cpu().numpy().copy()
  _, _, grad = m.loss_and_grads(feed, 1.0 / 3)
  g = grad.detach().cpu().numpy().copy()
  applier = RMSPropApplier(7e-4, decay=0.99, momentum=0.0, epsilon=0.1, clip_norm=40.0)
  out = m.update(feed, 7e-4, applier)
  norm = np.sqrt((g.astype(np.float64) ** 2).sum())
  gc = g * (40.0 / max(norm, 40.0))
  ms = 1.0 + (gc * gc - 1.0) * (1 - 0.99)
  want = before - 7e-4 * gc / np.sqrt(ms + 0.1)
  after = m.flat.detach().cpu().numpy()
  assert np.allclose(after, want, rtol=1e-5, atol=1e-7)
  assert abs(float(out["grad_norm"]) - norm) <= 1e-4 * norm
  assert torch.equal(m.flat16.float(), m.flat.detach().to(torch.bfloat16).float())


def _sms():
  return torch.cuda.get_device_properties(0).multi_processor_count


def conv_multi_item_sizes():
  """Sample counts that run the persistent conv kernels (grid = min(items, 2 CTAs per SM)) through several work items
  per CTA, for the kernels with one item per sample (conv2 forward, the transposed convolutions; conv1 has 4 per
  sample): just past one wave, kStages + 2 = 8 items per CTA (ConvCfg<2,16>::kStages = 6: the stage ring wraps across
  items), and config 5's batch of 1024 envs x T = 20."""
  grid = 2 * _sms()
  sizes = (grid + 1, 8 * grid, 20480)
  assert items_per_cta(sizes[1]) >= 8 and items_per_cta(sizes[2]) >= 3
  return sizes


def items_per_cta(items):
  """Most work items one CTA of a persistent conv kernel runs."""
  grid = min(items, 2 * _sms())
  return -(-items // grid)


def _conv64(x, w_oihw, b=None, stride=1, transpose=False):
  """conv2d / conv_transpose2d in float64 on NHWC tensors (NCHW-ordered weights) -> NHWC float64."""
  import torch.nn.functional as F
  op = F.conv_transpose2d if transpose else F.conv2d
  y = op(x.double().permute(0, 3, 1, 2), w_oihw.double(), None if b is None else b.double(), stride=stride)
  return y.permute(0, 2, 3, 1)


@pytest.mark.parametrize("dtype", [torch.float32, torch.uint8])
def test_fused_conv_forward_matches_direct_convolution(dtype):
  """TMA-im2col convolutions (space-to-depth taps) against conv2d on the same bf16-rounded operands in float64: the
  kernels' fp32 sums and their bf16 output -> one bf16 ulp (2^-8 relative).  Every output row is compared, up to
  S = 20 480 (many items per CTA)."""
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  g = torch.Generator(device=dev).manual_seed(3)
  assert items_per_cta(20480) >= 3 and items_per_cta(4 * 20480) >= 3
  for s in (1, 5, 37) + conv_multi_item_sizes():
    if dtype == torch.uint8:
      x = torch.randint(0, 256, (s, 84, 84, 3), device=dev, dtype=torch.uint8, generator=g)
      xf = (x.float() / 255.0).to(torch.bfloat16).float()
    else:
      x = torch.rand(s, 84, 84, 3, device=dev, generator=g)
      xf = x.to(torch.bfloat16).float()
    w1 = ((torch.rand(8, 8, 3, 16, device=dev, generator=g) - 0.5) * 0.2).to(torch.bfloat16)
    b1 = (torch.rand(16, device=dev, generator=g) - 0.5) * 0.1
    w2 = ((torch.rand(4, 4, 16, 32, device=dev, generator=g) - 0.5) * 0.2).to(torch.bfloat16)
    b2 = (torch.rand(32, device=dev, generator=g) - 0.5) * 0.1
    xs = K.s2d_frames(x)
    want_s2d = xf.view(s, 21, 4, 21, 4, 3).permute(0, 1, 3, 2, 4, 5).reshape(s, 441, 6, 8).permute(0, 2, 1, 3)
    assert torch.equal(xs.float(), want_s2d)
    h1 = K.conv_fwd(xs, 1, K.conv1_w_planes(w1), b1)
    ref1 = torch.relu(_conv64(xf, w1.permute(3, 2, 0, 1), b1, stride=4))
    del xs, xf, x
    assert tuple(h1.shape) == (s, 20, 20, 16)
    assert torch.allclose(h1.double(), ref1, rtol=2.0 ** -7, atol=1e-3), s
    del ref1
    h2 = K.conv_fwd(h1, 2, K.conv_taps(w2, 2), b2)
    # transposed convolution (input gradient of conv2) through the zero-filling TMA boxes
    dy2 = (torch.randn(s * 81, 32, device=dev, generator=g) * 0.1).to(torch.bfloat16)
    dh1 = K.conv2_dgrad(dy2, K.conv2_dgrad_taps(w2))
    ref_dh1 = _conv64(dy2.view(s, 9, 9, 32), w2.permute(3, 2, 0, 1), stride=2, transpose=True)
    assert tuple(dh1.shape) == (s, 20, 20, 16)
    assert torch.allclose(dh1.double(), ref_dh1, rtol=2.0 ** -7, atol=1e-3), s
    del ref_dh1, dh1
    ref2 = torch.relu(_conv64(h1, w2.permute(3, 2, 0, 1), b2, stride=2))
    assert tuple(h2.shape) == (s, 9, 9, 32)
    assert torch.allclose(h2.double(), ref2, rtol=2.0 ** -7, atol=1e-3), s


def test_fused_conv1_wgrad_matches_autograd():
  """Tensor-core conv1 filter gradient (x'' planes x dY planes, reduction over pixels in TMEM)
  against torch autograd's conv2d weight gradient on the same bf16-rounded operands."""
  from unreal_b200 import kernels as K
  import torch.nn.functional as F
  dev = torch.device("cuda", 0)
  g = torch.Generator(device=dev).manual_seed(11)
  for s in (1, 3, 150):          # 150 frames = 600 items: several per CTA, accumulators persist across them
    x = torch.rand(s, 84, 84, 3, device=dev, generator=g)
    xf = x.to(torch.bfloat16).float()
    y = torch.rand(s * 400, 16, device=dev, generator=g).to(torch.bfloat16) - 0.3      # ReLU mask source
    dy = (torch.randn(s * 400, 16, device=dev, generator=g) * 0.1).to(torch.bfloat16)
    dyp, db = K.relu_grad(dy, y, planes=True)
    masked = (dy.float() * (y.float() > 0)).to(torch.bfloat16).float()
    assert torch.equal(dyp.permute(1, 0, 2).reshape(s * 400, 16).float(), masked)
    assert torch.allclose(db, masked.sum(0), rtol=1e-4, atol=1e-3)
    dw = K.conv1_wgrad(K.s2d_frames(x), dyp)
    w = torch.zeros(16, 3, 8, 8, device=dev, requires_grad=True)
    out = F.conv2d(xf.permute(0, 3, 1, 2), w, stride=4)                                   # [S,16,20,20]
    out.backward(masked.view(s, 20, 20, 16).permute(0, 3, 1, 2))
    ref = w.grad.permute(2, 3, 1, 0)                                                       # HWIO
    assert torch.allclose(dw, ref, rtol=1e-3, atol=1e-3 * float(ref.abs().max()))


def test_indoor_shaped_a3c_lstm_matches_oracle():
  """BASELINE configs[4] shape: MINOS-like observations -- uint8 RGB frames (/255 on load,
  indoor_environment.py:102-103), 3 actions (:16-20), a goal vector of G = 2 appended to
  last_action_reward (experience.py:34-46) -- through the A3C-LSTM tower only (no aux heads)."""
  from unreal_b200.model.model import UnrealModel
  from oracle import model_oracle as M
  dev = torch.device("cuda", 0)
  A_, G_, T, N = 3, 2, 4, 3
  m = UnrealModel(A_, G_, -1, True, False, False, False, 0.05, 0.001, dev, {'segnet_mode': 0}, (84, 84), True, 0, 0.0,
                  0.0, num_envs=N, seed=5)
  assert len(m.get_vars()) == 12                      # model_test.py: base only = 12 variables
  rs = np.random.RandomState(8)
  img8 = torch.from_numpy(rs.randint(0, 256, size=(T, N, 84, 84, 3)).astype(np.uint8))
  lar = np.zeros((T, N, A_ + 1 + G_), np.float32)
  np.put_along_axis(lar, rs.randint(0, A_, size=(T, N, 1)), 1.0, axis=-1)
  lar[..., A_] = rs.randint(-1, 2, size=(T, N)); lar[..., A_ + 1:] = rs.rand(T, N, G_)
  a = np.zeros((T, N, A_), np.float32); np.put_along_axis(a, rs.randint(0, A_, size=(T, N, 1)), 1.0, axis=-1)
  base = dict(lar=torch.from_numpy(lar), a=torch.from_numpy(a), adv=torch.from_numpy(rs.randn(T, N).astype(np.float32)),
              R=torch.from_numpy(rs.randn(T, N).astype(np.float32)), mask=torch.ones(T, N),
              c0=torch.zeros(N, 256), h0=torch.zeros(N, 256))
  feed_gpu = {"base": dict({k: v.to(dev) for k, v in base.items()}, images=img8.to(dev))}
  total, parts, grad = m.loss_and_grads(feed_gpu)
  params = {k: v.detach().cpu().clone() for k, v in m.named_vars().items()}
  o = M.ModelOracle(params, A_, G_, 0.05, 0.001, emulate_bf16=True)
  feed_cpu = {"base": dict(base, images=img8.float() / 255.0)}
  rtotal, rparts, rgrads = o.loss_and_grads(feed_cpu)
  for k in ("policy", "value"):
    assert abs(float(parts[k]) - float(rparts[k])) <= 2e-3 * max(1.0, abs(float(rparts[k]))), k
  got = {k: v.cpu() for k, v in m._views(grad).items()}
  for k, rg in rgrads.items():
    assert float((got[k] - rg).abs().max()) <= 3e-2 * float(rg.abs().max()) + 1e-6, k


def test_fused_conv2_wgrad_matches_autograd():
  """conv2 filter gradient through TMA boxes (MN-major SW64 operands, TMEM accumulators across
  samples) against torch autograd on the same bf16-rounded operands."""
  from unreal_b200 import kernels as K
  import torch.nn.functional as F
  dev = torch.device("cuda", 0)
  g = torch.Generator(device=dev).manual_seed(12)
  for s in (1, 2, 700):
    h1 = torch.rand(s, 20, 20, 16, device=dev, generator=g).to(torch.bfloat16)
    dy = (torch.randn(s * 81, 32, device=dev, generator=g) * 0.1).to(torch.bfloat16)
    dw = K.conv2_wgrad(h1, dy)
    w = torch.zeros(32, 16, 4, 4, device=dev, requires_grad=True)
    out = F.conv2d(h1.float().permute(0, 3, 1, 2), w, stride=2)                       # [S,32,9,9]
    out.backward(dy.float().view(s, 9, 9, 32).permute(0, 3, 1, 2))
    ref = w.grad.permute(2, 3, 1, 0)                                                   # HWIO [4,4,16,32]
    assert torch.allclose(dw, ref, rtol=1e-3, atol=1e-3 * float(ref.abs().max())), s


def test_fused_pc_deconv_forward_matches_conv_transpose():
  """The pixel-control head's merged 8-channel deconv forward (conv2's transposed-convolution tcgen05
  kernel at 8 channels, bias + ReLU epilogue) against torch conv_transpose2d in float64 on the same
  bf16-rounded operands, and against the GEMM + col2im path it replaces."""
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  g = torch.Generator(device=dev).manual_seed(21)
  for s in (1, 3, 500) + conv_multi_item_sizes():
    h = torch.rand(s, 9, 9, 32, device=dev, generator=g).to(torch.bfloat16)
    w8 = ((torch.rand(4, 4, 8, 32, device=dev, generator=g) - 0.5) * 0.2).to(torch.bfloat16)     # [kh,kw,out,in]
    b8 = (torch.rand(8, device=dev, generator=g) - 0.5) * 0.1
    y = K.pc_deconv_fwd(h, K.pc_deconv_taps(w8), b8)
    assert tuple(y.shape) == (s, 20, 20, 8) and y.dtype == torch.float32
    ref = torch.relu(_conv64(h, w8.permute(3, 2, 0, 1), b8, stride=2, transpose=True))
    assert torch.allclose(y.double(), ref, rtol=1e-4, atol=1e-5), (s, float((y - ref).abs().max()))
    del ref
    cols = K.gemm_bf16(h.view(s * 81, 32), w8.view(128, 32))
    old = K.col2im(cols, s, 20, 20, 8, 4, 4, 2, bias=b8, relu=True)
    assert torch.allclose(y, old, rtol=1e-4, atol=1e-5)


def test_conv2_dgrad_relu_equals_dgrad_then_relu_grad():
  """The fused transposed-convolution + ReLU-gradient epilogue writes exactly the planes the two-pass
  path (unreal_conv2_dgrad -> unreal_relu_grad(planes)) produces, and the same bias gradient."""
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  g = torch.Generator(device=dev).manual_seed(5)
  for s in (1, 3, 600) + conv_multi_item_sizes():
    dy = (torch.randn(s * 81, 32, device=dev, generator=g) * 0.1).to(torch.bfloat16)
    w = ((torch.rand(4, 4, 16, 32, device=dev, generator=g) - 0.5) * 0.2).to(torch.bfloat16)
    h1 = torch.relu(torch.randn(s, 20, 20, 16, device=dev, generator=g)).to(torch.bfloat16)     # about half zeros
    taps = K.conv2_dgrad_taps(w)
    dense = K.conv2_dgrad(dy, taps)
    want_planes, want_db = K.relu_grad(dense.view(s * 400, 16), h1.view(s * 400, 16), planes=True)
    planes, db = K.conv2_dgrad_relu(dy, taps, h1)
    assert torch.equal(planes, want_planes), s
    assert torch.allclose(db, want_db, rtol=1e-4, atol=1e-4 * float(want_db.abs().max() + 1e-6)), s
    # independently: conv_transpose2d in float64, masked by h1 > 0; the planes hold it rounded once to bf16, the bias
    # gradient is the sum of those rounded values over samples and pixels (fp32 partial sums and atomics)
    ref = (_conv64(dy.view(s, 9, 9, 32), w.permute(3, 2, 0, 1), stride=2, transpose=True) * (h1 > 0)).reshape(s * 400, 16)
    got = planes.permute(1, 0, 2).reshape(s * 400, 16).double()
    assert torch.allclose(got, ref, rtol=2.0 ** -8, atol=1e-5), (s, float((got - ref).abs().max()))
    assert torch.allclose(db.double(), got.sum(0), rtol=0, atol=1e-4 * float(got.abs().sum(0).max()) + 1e-6), s
    del ref, got, dense
    # the 21-pixel-pitch form conv1's wgrad copies in one piece per plane: same values, zero column 20
    p21, _ = K.conv2_dgrad_relu(dy, taps, h1, pitch21=True)
    p21 = p21.view(2, s, 20, 21, 8)
    assert torch.equal(p21[:, :, :, :20], want_planes.view(2, s, 20, 20, 8)) and not p21[:, :, :, 20].any()
    xpp = torch.rand(s, 6, 441, 8, device=dev, generator=g).to(torch.bfloat16)
    assert torch.allclose(K.conv1_wgrad(xpp, p21.view(2, s * 420, 8)), K.conv1_wgrad(xpp, want_planes), rtol=1e-4, atol=1e-4)


def test_fused_encoder_backward_equals_layerwise_backward():
  """EncoderFn (one autograd node, cross-layer fused backward) gives the same loss and gradients as the
  two ConvFn nodes with the dense gradient and the relu_grad pass between them."""
  dev = torch.device("cuda", 0)
  net_a, net_b = _model(dev, seed=4), _model(dev, seed=4)
  net_b.fused_encoder = False
  gpu = _to(_feed(5, 3, 4, seed=9), dev)
  ta, pa, ga = net_a.loss_and_grads(gpu)
  tb, pb, gb = net_b.loss_and_grads(gpu)
  assert abs(float(ta) - float(tb)) <= 1e-5 * max(1.0, abs(float(tb)))
  va, vb = net_a._views(ga), net_b._views(gb)
  for k in va:      # same operands, same roundings: only the order of the fp32 atomics differs
    assert torch.allclose(va[k], vb[k], rtol=2e-3, atol=2e-3 * float(vb[k].abs().max() + 1e-12)), k


def test_render_fused_conv1_equals_conv1_on_rendered_frames():
  """unreal_conv1_fwd_maze / unreal_conv1_wgrad_maze build the x'' tiles from the agent cells in shared memory:
  bit-identical outputs to the same kernels reading frames rendered by K1 (every free cell of the map)."""
  from oracle import unreal_oracle as O
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  g = torch.Generator(device=dev).manual_seed(3)
  cells = [(x, y) for y in range(7) for x in range(7) if not O.WALLS[y, x]]
  pos = torch.tensor(cells * 9, dtype=torch.int32, device=dev)           # 306 frames: several waves of work items
  s = pos.shape[0]
  w1 = ((torch.rand(8, 8, 3, 16, device=dev, generator=g) - 0.5) * 0.3).to(torch.bfloat16)
  b1 = (torch.rand(16, device=dev, generator=g) - 0.5) * 0.1
  taps = K.conv1_w_planes(w1)
  xpp = K.maze_render(pos, dtype=torch.bfloat16)
  want = K.conv_fwd(xpp, 1, taps, b1)
  got = K.conv1_fwd_maze(pos, taps, b1)
  assert torch.equal(got, want)
  # and every frame against the float64 convolution of the oracle's frame of its cell (0 / 1 pixels: the kernel's
  # operands are exact, so only its fp32 sums and the bf16 output rounding differ) -- here and at sample counts with
  # several conv1 items (4 per frame) per CTA, up to 20 480 frames
  frames = torch.from_numpy(np.stack([O.maze_render(x, y) for x, y in cells]).astype(np.float32)).to(dev)
  ref_cell = torch.relu(_conv64(frames, w1.permute(3, 2, 0, 1), b1, stride=4))          # [cells, 20, 20, 16]
  assert torch.allclose(got.double(), ref_cell.repeat(9, 1, 1, 1), rtol=2.0 ** -7, atol=1e-3)
  assert items_per_cta(4 * s) >= 3
  rs = np.random.RandomState(4)
  for n in conv_multi_item_sizes():
    idx = rs.randint(0, len(cells), size=n)
    h = K.conv1_fwd_maze(pos[:len(cells)][torch.from_numpy(idx).to(dev)].contiguous(), taps, b1)
    ref = ref_cell[torch.from_numpy(idx).to(dev)]
    assert torch.allclose(h.double(), ref, rtol=2.0 ** -7, atol=1e-3), (n, float((h.double() - ref).abs().max()))
    del h, ref
  dy = (torch.randn(2, s * 420, 8, device=dev, generator=g) * 0.1).to(torch.bfloat16)
  dy.view(2, s, 20, 21, 8)[:, :, :, 20] = 0
  a = K.conv1_wgrad_maze(pos, dy)
  b = K.conv1_wgrad(xpp, dy)
  assert torch.allclose(a, b, rtol=1e-5, atol=1e-5 * float(b.abs().max()))


def test_fused_heads_match_torch_heads():
  """unreal_a3c_head_loss / unreal_a3c_head_bwd (policy + value heads, softmax, A3C losses and their gradients in
  two sweeps over h) against the same arithmetic written in torch fp32 with autograd."""
  from unreal_b200 import kernels as K
  from unreal_b200.model.layers import A3CHeadLossFn
  dev = torch.device("cuda", 0)
  g = torch.Generator(device=dev).manual_seed(8)
  for m, a in ((5, 4), (1000, 3), (4097, 6)):
    h = torch.randn(m, 256, device=dev, generator=g, requires_grad=True)
    wp = (torch.randn(256, a, device=dev, generator=g) * 0.1).requires_grad_(True)
    bp = (torch.randn(a, device=dev, generator=g) * 0.1).requires_grad_(True)
    wv = (torch.randn(256, 1, device=dev, generator=g) * 0.1).requires_grad_(True)
    bv = (torch.randn(1, device=dev, generator=g) * 0.1).requires_grad_(True)
    act = torch.randint(0, a, (m,), device=dev, generator=g, dtype=torch.int32)
    adv = torch.randn(m, device=dev, generator=g); ret = torch.randn(m, device=dev, generator=g)
    mask = (torch.rand(m, device=dev, generator=g) < 0.8).float()
    beta = 0.01
    pol, val, ent = A3CHeadLossFn.apply(h, wp, bp, wv, bv, act, adv, ret, mask, beta, 0.25)
    (pol * 0.7 + val * 1.3).backward()
    got = [x.grad.clone() for x in (h, wp, bp, wv, bv)]
    for x in (h, wp, bp, wv, bv):
      x.grad = None
    pi = torch.softmax(h @ wp + bp, -1); v = (h @ wv + bv).squeeze(-1)
    lp = torch.log(pi.clamp(1e-20, 1.0)); H = -(pi * lp).sum(-1)
    onehot = torch.nn.functional.one_hot(act.long(), a).float()
    rpol = -((((lp * onehot).sum(-1)) * adv + H * beta) * mask).sum(); rval = 0.25 * (((ret - v) ** 2) * mask).sum()
    (rpol * 0.7 + rval * 1.3).backward()
    ref = [x.grad.clone() for x in (h, wp, bp, wv, bv)]
    assert torch.allclose(pol, rpol, rtol=1e-4, atol=1e-3) and torch.allclose(val, rval, rtol=1e-4, atol=1e-3)
    assert torch.allclose(ent, (H * mask).sum(), rtol=1e-4, atol=1e-3)
    for x, y, name in zip(got, ref, "h wp bp wv bv".split()):
      assert torch.allclose(x, y, rtol=1e-3, atol=1e-4 * float(y.abs().max() + 1e-6)), (m, a, name)
    out = K.a3c_head(h.detach(), wp.detach().contiguous(), bp.detach(), wv.detach().reshape(256).contiguous(), bv.detach(),
                     want_pi=True, want_v=True)
    assert torch.allclose(out["pi"], pi.detach(), rtol=1e-4, atol=1e-6) and torch.allclose(out["v"], v.detach(), rtol=1e-4, atol=1e-5)


def test_rp_head_on_the_device_path_matches_torch():
  """The reward-prediction head (model.py:479-488, :571-575) as tcgen05 GEMMs on the padded bf16 weight shadow +
  unreal_rp_loss (bias, softmax, clipped cross-entropy, d loss / d logits as the backward GEMMs' bf16 operand),
  against the same arithmetic in torch fp32 with autograd on the bf16-rounded operands.  Soft and one-hot targets,
  batch sizes off the 128-row tile, and run_rp_c's probabilities."""
  from unreal_b200 import kernels as K
  from unreal_b200.model.layers import RpHeadLossFn
  dev = torch.device("cuda", 0)
  g = torch.Generator(device=dev).manual_seed(21)
  for n in (3, 130, 1000):
    h2 = torch.relu(torch.randn(n, 7776, device=dev, generator=g)).to(torch.bfloat16).requires_grad_(True)
    w32 = (torch.randn(7776, 3, device=dev, generator=g) * 0.02).requires_grad_(True)
    b32 = (torch.randn(3, device=dev, generator=g) * 0.1).requires_grad_(True)
    w8 = torch.zeros(7776, 8, dtype=torch.bfloat16, device=dev)
    w8[:, :3] = w32.detach()
    cls = torch.randint(0, 3, (n,), device=dev, generator=g)
    c = torch.nn.functional.one_hot(cls, 3).float()
    if n == 130:
      c = torch.rand(n, 3, device=dev, generator=g)                  # the kernel takes the reference's general c
    loss = RpHeadLossFn.apply(h2, w8, w32, b32, c)
    (loss * 0.6).backward()
    got = [h2.grad.float().clone(), w32.grad.clone(), b32.grad.clone()]
    for x in (h2, w32, b32):
      x.grad = None
    hf = h2.detach().float().requires_grad_(True)
    wf = w8[:, :3].float().detach().requires_grad_(True)
    p = torch.softmax(hf @ wf + b32, -1)
    rloss = -(c * torch.log(p.clamp(1e-20, 1.0))).sum()
    (rloss * 0.6).backward()
    assert torch.allclose(loss, rloss.detach(), rtol=1e-4, atol=1e-3), n
    # dY is rounded to bf16 where it becomes a GEMM operand (2^-9 per element), dh2 is a bf16 tensor
    for x, y, name in zip(got, (hf.grad, wf.grad, b32.grad), ("h2", "W", "b")):
      assert float((x - y).abs().max()) <= 1e-2 * float(y.abs().max()) + 1e-7, (n, name)
    logits8 = K.gemm_bf16(h2.detach(), w8, b_mn_major=True)
    pr = K.rp_loss(logits8, b32.detach().contiguous(), want_p=True)["p"]
    assert torch.allclose(pr, p.detach(), rtol=1e-4, atol=1e-6)
    assert torch.allclose(logits8[:, 3:], torch.zeros_like(logits8[:, 3:]))


def test_cell_gather_and_segment_sum_match_torch():
  """unreal_cell_gather / unreal_cell_segment_sum (the two kernels of the maze-cell de-duplication) against torch
  index_select / index_add_: gather bit-exact, also into a column slice of a wider buffer; sums to fp32 order."""
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  g = torch.Generator(device=dev).manual_seed(3)
  for S in (1, 77, 4099, 200000):
    pos = torch.stack((torch.randint(0, 7, (S,), device=dev, generator=g), torch.randint(0, 7, (S,), device=dev, generator=g)),
                      dim=1).to(torch.int32).contiguous()
    idx = (pos[:, 1] * 7 + pos[:, 0]).long()
    table = torch.randn(49, 256, device=dev, generator=g).to(torch.bfloat16)
    assert torch.equal(K.cell_gather(table, pos), table[idx])
    wide = torch.zeros(S, 520, dtype=torch.bfloat16, device=dev)
    K.cell_gather(table, pos, out=wide[:, :256])
    assert torch.equal(wide[:, :256], table[idx]) and not wide[:, 256:].any()
    for dt in (torch.float32, torch.bfloat16):
      dy = torch.randn(S, 256, device=dev, generator=g).to(dt)
      want = torch.zeros(49, 256, device=dev, dtype=torch.float64).index_add_(0, idx, dy.double())
      got = K.cell_segment_sum(dy, pos)
      assert torch.allclose(got.double(), want, rtol=1e-5, atol=1e-4 * max(1.0, S ** 0.5) * 1e-1)


def test_cell_table_encoder_equals_dense_encoder():
  """UnrealModel.dedup_cells: conv1 -> conv2 -> fc1 of every sample as a row of the 49-cell table.  On the same feed of
  maze CELLS the losses must equal the dense (render-fused) encoder's -- the forward values are the same numbers -- and
  every variable's gradient must agree to the bf16 rounding of the per-cell gradient sums."""
  dev = torch.device("cuda", 0)
  m = _model(dev, seed=5, n=6)
  T, N, L = 5, 6, 4
  rs = np.random.RandomState(9)
  from oracle import unreal_oracle as O
  cells = np.array([(x, y) for y in range(7) for x in range(7) if not O.WALLS[y, x]], np.int32)
  feed = _to(_feed(T, N, L, seed=31, maze_frames=True), dev)
  pick = lambda *lead: torch.from_numpy(cells[rs.randint(0, len(cells), size=lead)]).to(dev)   # noqa: E731
  feed["base"]["images"] = pick(T, N); feed["pc"]["images"] = pick(L, N); feed["vr"]["images"] = pick(L, N)
  feed["rp"]["images"] = pick(N, 3)
  out = {}
  for dedup in (False, True):
    m.dedup_cells = dedup
    m.refresh_shadow()
    total, parts, grad = m.loss_and_grads(feed)
    out[dedup] = (float(total), {k: float(v) for k, v in parts.items()}, {k: v.clone() for k, v in m._views(grad).items()})
  for k in out[False][1]:
    a, b = out[False][1][k], out[True][1][k]
    assert abs(a - b) <= 1e-5 * max(1.0, abs(a)), (k, a, b)
  for k, ref in out[False][2].items():
    got = out[True][2][k]
    assert float((got - ref).abs().max()) <= 1e-2 * float(ref.abs().max()) + 1e-7, k
  # acting helpers read the no-grad table: same policy / value as the dense path
  lar = feed["base"]["lar"][0]
  res = {}
  for dedup in (False, True):
    m.dedup_cells = dedup
    m.refresh_shadow(); m.reset_state()
    pi, v, _ = m.run_base_policy_and_value(None, {'image': feed["base"]["images"][0]}, lar)
    q = m.run_pc_q_max(None, {'image': feed["base"]["images"][1]}, lar)
    res[dedup] = (pi.clone(), v.clone(), q.clone())
  for a, b in zip(res[False], res[True]):
    assert torch.allclose(a, b, rtol=1e-4, atol=1e-5)


def test_fused_pc_deconv_loss_equals_the_three_kernel_path():
  """unreal_pc_deconv_loss (pixel-control deconv forward + dueling / gather / L2 loss + its gradient in ONE kernel, the
  f32 head output never materialised) against PcHeadLossFn (deconv -> y8 f32 -> unreal_pc_loss -> unreal_pc_loss_grad16):
  same loss, same gradients for the input, both deconv filters and biases, including an upstream gradient != 1."""
  from unreal_b200.model.layers import PcFusedHeadLossFn, PcHeadLossFn
  dev = torch.device("cuda", 0)
  m = _model(dev, seed=9, n=2)
  p32 = m._views(m.flat)
  g = torch.Generator(device=dev).manual_seed(4)
  for s in (3, 129, 700):
    hp = torch.relu(torch.randn(s, 2592, device=dev, generator=g)).to(torch.bfloat16)
    act = torch.randint(0, A, (s,), device=dev, generator=g, dtype=torch.int32)
    tgt = torch.rand(s, 400, device=dev, generator=g)
    msk = (torch.rand(s, device=dev, generator=g) < 0.8).float()
    res = []
    for fn in (PcHeadLossFn, PcFusedHeadLossFn):
      x = hp.clone().requires_grad_(True)
      leaves = [p32[k].detach().clone().requires_grad_(True) for k in ("W_pc_deconv_v", "b_pc_deconv_v", "W_pc_deconv_a", "b_pc_deconv_a")]
      loss = fn.apply(x, m.pc_taps, m.pc_b8, m.pc_lin_taps, leaves[0], leaves[1], leaves[2], leaves[3], act, tgt, msk, A, 0.05)
      (loss * 0.37).backward()
      res.append((loss.detach(), x.grad.float(), [l.grad for l in leaves]))
    (l0, dx0, g0), (l1, dx1, g1) = res
    assert abs(float(l0) - float(l1)) <= 1e-5 * max(1.0, abs(float(l0))), s
    assert float((dx0 - dx1).abs().max()) <= 2.0 ** -7 * float(dx0.abs().max()) + 1e-9, s      # both round dh to bf16
    # the two paths round d loss / d y to bf16 at different points (before / after the upstream gradient is applied):
    # filter and bias gradients agree to the bf16 operand rounding, 2^-8 of the largest element
    for a_, b_, name in zip(g0, g1, ("Wv", "bv", "Wa", "ba")):
      assert float((a_ - b_).abs().max()) <= 2.0 ** -8 * float(a_.abs().max()) + 1e-9, (s, name)


def test_pc_tower_with_the_relu_gradient_in_the_backward_convolution_equals_two_nodes():
  """PcTowerFusedFn (pc_fc1 + deconv + loss as one autograd node; pc_fc1's ReLU mask and bias gradient applied by
  unreal_conv2_fwd_linear_masked's epilogue) against LinearFn -> PcFusedHeadLossFn with a unreal_relu_grad pass between
  them: same loss; the masked bf16 gradient is the same tensor, so every gradient agrees to summation order.  Sample
  counts below / at / above one wave of CTAs, an upstream gradient != 1."""
  from unreal_b200 import kernels as K
  from unreal_b200.model.layers import LinearFn, PcFusedHeadLossFn, PcTowerFusedFn
  dev = torch.device("cuda", 0)
  m = _model(dev, seed=10, n=2)
  p32 = m._views(m.flat)
  g = torch.Generator(device=dev).manual_seed(5)
  names = ("W_pc_fc1", "b_pc_fc1", "W_pc_deconv_v", "b_pc_deconv_v", "W_pc_deconv_a", "b_pc_deconv_a")
  for s in (1, 3, 296, 1000):
    h = torch.randn(s, 256, device=dev, generator=g)
    act = torch.randint(0, A, (s,), device=dev, generator=g, dtype=torch.int32)
    tgt = torch.rand(s, 400, device=dev, generator=g)
    msk = (torch.rand(s, device=dev, generator=g) < 0.8).float()
    res = []
    for fused in (False, True, 8, "planes"):
      x = h.clone().requires_grad_(True)
      lv = [p32[k].detach().clone().requires_grad_(True) for k in names]
      if fused:
        loss = PcTowerFusedFn.apply(x, m.v16["W_pc_fc1"], lv[0], lv[1], m.pc_taps, m.pc_b8,
                                    {8: m.pc_lin_taps8, "planes": m.pc_w_planes}.get(fused, m.pc_lin_taps), lv[2], lv[3],
                                    lv[4], lv[5], act, tgt, msk, A, 0.05)
      else:
        hp = LinearFn.apply(x, m.v16["W_pc_fc1"], lv[0], lv[1], True, True)
        loss = PcFusedHeadLossFn.apply(hp, m.pc_taps, m.pc_b8, m.pc_lin_taps, lv[2], lv[3], lv[4], lv[5], act, tgt, msk, A, 0.05)
      (loss * 0.37).backward()
      res.append((loss.detach(), x.grad.float(), [l.grad for l in lv]))
    (l0, dx0, g0), (l1, dx1, g1), (l2, dx2, g2), (l3, dx3, g3) = res
    assert float(l0) == float(l1) == float(l2) == float(l3), s
    assert float((dx0 - dx3).abs().max()) <= 2.0 ** -7 * float(dx0.abs().max()) + 1e-9, s
    for a_, b_, name in zip(g0, g3, names):
      assert float((a_ - b_).abs().max()) <= 2.0 ** -7 * float(a_.abs().max()) + 1e-9, (s, name, "planes")
    assert float((dx0 - dx1).abs().max()) <= 1e-5 * float(dx0.abs().max()) + 1e-9, s
    for a_, b_, name in zip(g0, g1, names):
      assert float((a_ - b_).abs().max()) <= 1e-5 * float(a_.abs().max()) + 1e-9, (s, name)
    # the 8-channel gradient: the UMMAs sum in another order, a bf16 rounding of d(pc_fc1 output) can move by one ulp
    assert float((dx0 - dx2).abs().max()) <= 2.0 ** -7 * float(dx0.abs().max()) + 1e-9, s
    for a_, b_, name in zip(g0, g2, names):
      assert float((a_ - b_).abs().max()) <= 2.0 ** -7 * float(a_.abs().max()) + 1e-9, (s, name)
  # the kernel alone: masked result and bias gradient against torch on the un-masked kernel's output
  s = 300
  dy16 = (torch.randn(s, 20, 20, 16, device=dev, generator=g) * 0.1).to(torch.bfloat16)
  y = torch.randn(s, 2592, device=dev, generator=g).to(torch.bfloat16)
  sc = torch.tensor([0.61], device=dev)
  dense = K.conv2_fwd_linear(dy16, m.pc_lin_taps, scale=sc).view(s, 2592)
  got, db = K.conv2_fwd_linear(dy16, m.pc_lin_taps, scale=sc, mask_y=y)
  want = torch.where(y > 0, dense, torch.zeros_like(dense))
  assert torch.equal(got.view(s, 2592), want)
  ref_db = want.float().sum(0)
  assert float((db - ref_db).abs().max()) <= 1e-5 * float(ref_db.abs().max()) + 1e-6


@pytest.mark.parametrize("s", [1, 5, 296, 297, 1500])
def test_pc_backward_kernels_on_the_8_channel_gradient_equal_the_16_channel_ones(s):
  """The pixel-control loss gradient without its 8 zero padding channels ([S,400,8] instead of conv2's [S,400,16]):
  unreal_pc_deconv_loss_c8 writes the same values; unreal_conv2_fwd_linear_masked (c_in = 8: 64-byte box rows under the
  64-byte swizzle) and unreal_conv2_wgrad_c8 give what the 16-channel kernels give on the zero-padded tensor -- the
  padding contributes exact zeros, so only the fp32 summation order inside the UMMAs can differ."""
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  m = _model(dev, seed=11, n=2)
  g = torch.Generator(device=dev).manual_seed(s)
  hp = torch.relu(torch.randn(s, 2592, device=dev, generator=g)).to(torch.bfloat16)
  act = torch.randint(0, A, (s,), device=dev, generator=g, dtype=torch.int32)
  tgt = torch.rand(s, 400, device=dev, generator=g)
  msk = (torch.rand(s, device=dev, generator=g) < 0.8).float()
  l16, dy16, db16 = K.pc_deconv_loss(hp, m.pc_taps, m.pc_b8, act, tgt, msk, A, 0.05)
  l8, dy8, db8 = K.pc_deconv_loss(hp, m.pc_taps, m.pc_b8, act, tgt, msk, A, 0.05, c8=True)
  assert tuple(dy8.shape) == (s, 400, 8) and torch.equal(dy8, dy16[:, :, :8]) and not bool(dy16[:, :, 8:].any())
  assert abs(float(l8) - float(l16)) <= 1e-9 * max(1.0, abs(float(l16)))
  assert float((db8 - db16).abs().max()) <= 1e-5 * float(db16.abs().max()) + 1e-9
  # a random 8-channel gradient (the loss gradient itself is sparse in the action channels)
  x8 = (torch.randn(s, 20, 20, 8, device=dev, generator=g) * 0.1).to(torch.bfloat16)
  x16 = torch.zeros(s, 20, 20, 16, device=dev, dtype=torch.bfloat16); x16[..., :8] = x8
  y = torch.randn(s, 2592, device=dev, generator=g).to(torch.bfloat16)
  sc = torch.tensor([0.61], device=dev)
  o16, b16 = K.conv2_fwd_linear(x16, m.pc_lin_taps, scale=sc, mask_y=y)
  o8, b8 = K.conv2_fwd_linear(x8, m.pc_lin_taps8, scale=sc, mask_y=y)
  ref = o16.float()
  assert float((o8.float() - ref).abs().max()) <= 2.0 ** -7 * float(ref.abs().max()) + 1e-9      # one bf16 rounding of a reordered sum
  assert float((b8 - b16).abs().max()) <= 2.0 ** -7 * float(b16.abs().max()) + 1e-6
  # and against an fp32 torch convolution of the same bf16 operands
  w8 = m.pc_w8.view(4, 4, 8, 32).float()                                    # HWIO
  conv = torch.nn.functional.conv2d(x8.float().permute(0, 3, 1, 2), w8.permute(3, 2, 0, 1), stride=2).permute(0, 2, 3, 1) * 0.61
  conv = torch.where(y.view(s, 9, 9, 32) > 0, conv, torch.zeros_like(conv))
  assert float((o8.float() - conv).abs().max()) <= 2.0 ** -7 * float(conv.abs().max()) + 1e-6
  dw16 = K.conv2_wgrad(x16, hp.view(s * 81, 32))
  dw8 = K.conv2_wgrad(x8, hp.view(s * 81, 32))
  assert tuple(dw8.shape) == (4, 4, 8, 32)
  assert float((dw8 - dw16[:, :, :8]).abs().max()) <= 1e-5 * float(dw16.abs().max()) + 1e-6
  assert not bool(dw16[:, :, 8:].any())
  # the plane-major layout (four parity planes of the 10 x 10 grid, one bulk copy per sample): same three results
  lp, dyp, dbp = K.pc_deconv_loss(hp, m.pc_taps, m.pc_b8, act, tgt, msk, A, 0.05, planes=True)
  assert tuple(dyp.shape) == (s, 4, 100, 8) and torch.equal(dyp, K.pc_planes_from_dense(dy8.view(s, 20, 20, 8)))
  assert abs(float(lp) - float(l16)) <= 1e-9 * max(1.0, abs(float(l16)))
  xp = K.pc_planes_from_dense(x8)
  op, bp = K.pc_planes_conv(xp, m.pc_w_planes, y, scale=sc)
  assert float((op.float() - conv).abs().max()) <= 2.0 ** -7 * float(conv.abs().max()) + 1e-6
  assert float((op.float() - ref).abs().max()) <= 2.0 ** -7 * float(ref.abs().max()) + 1e-9
  assert float((bp - b16).abs().max()) <= 2.0 ** -7 * float(b16.abs().max()) + 1e-6
  dwp = K.pc_planes_wgrad(xp, hp)
  assert float((dwp - dw16[:, :, :8]).abs().max()) <= 1e-5 * float(dw16.abs().max()) + 1e-6


@pytest.mark.parametrize("na", [3, 4])
def test_pc_loss_epilogue_with_a_static_action_count_equals_the_generic_one(na):
  """unreal_pc_deconv_loss with the action count as a compile-time constant (3 and 4, the reference's two action spaces) against
  the run-time loop over the 7 advantage channels: the same arithmetic in the same order -- identical gradient bits."""
  from unreal_b200 import _lib, kernels as K
  dev = torch.device("cuda", 0)
  g = torch.Generator(device=dev).manual_seed(40 + na)
  s = 777
  hp = torch.relu(torch.randn(s, 2592, device=dev, generator=g)).to(torch.bfloat16)
  w8 = torch.zeros(4, 4, 8, 32, device=dev, dtype=torch.bfloat16)
  w8[:, :, :1 + na] = (torch.randn(4, 4, 1 + na, 32, device=dev, generator=g) * 0.05).to(torch.bfloat16)
  b8 = torch.zeros(8, device=dev); b8[:1 + na] = torch.randn(1 + na, device=dev, generator=g) * 0.1
  taps = K.pc_deconv_taps(w8)
  act = torch.randint(0, na, (s,), device=dev, generator=g, dtype=torch.int32)
  tgt = torch.rand(s, 400, device=dev, generator=g)
  msk = (torch.rand(s, device=dev, generator=g) < 0.8).float()
  res = {}
  try:
    for static in (0, 1):
      _lib.set_tunable("pc_loss_static_a", static)
      res[static] = [K.pc_deconv_loss(hp, taps, b8, act, tgt, msk, na, 0.05, planes=pl, c8=c8) for pl, c8 in ((False, False), (False, True), (True, False))]
  finally:
    _lib.set_tunable("pc_loss_static_a", 1)
  for (l0, d0, b0), (l1, d1, b1) in zip(res[0], res[1]):
    assert torch.equal(d0, d1)
    assert abs(float(l0) - float(l1)) <= 1e-9 * max(1.0, abs(float(l0)))
    assert float((b0 - b1).abs().max()) <= 1e-5 * float(b0.abs().max()) + 1e-9
  assert not bool(res[1][0][1][:, :, 1 + na:].any())           # channels beyond 1 + A stay zero


def test_pc_q_max_epilogue_equals_the_materialised_head():
  """run_pc_q_max with the dueling combine + max over actions inside the deconv's epilogue (unreal_pc_deconv_qmax) against
  the path that materialises the [N,20,20,8] head output and reduces it with torch ops: same maps (fp32 order only)."""
  dev = torch.device("cuda", 0)
  m = _model(dev, seed=12, n=5)
  g = torch.Generator(device=dev).manual_seed(6)
  frames = torch.rand(5, 84, 84, 3, device=dev, generator=g)
  lar = torch.zeros(5, A + 1, device=dev); lar[:, 1] = 1.0; lar[:, A] = -1.0
  out = {}
  for fused in (False, True):
    m.fused_pc_loss = fused
    out[fused] = m.run_pc_q_max(None, {'image': frames}, lar).clone()
  assert tuple(out[True].shape) == (5, 20, 20)
  assert torch.allclose(out[True], out[False], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("na", [3, 4, 7])
def test_pc_deconv_qmax_matches_the_dueling_max_in_float64(na):
  """unreal_pc_deconv_qmax's epilogue (ReLU head, V + A - mean A, max over the `na` actions) against the same
  arithmetic on conv_transpose2d in float64, at sample counts with several items per CTA (up to 20 480)."""
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  g = torch.Generator(device=dev).manual_seed(40 + na)
  for s in (5,) + conv_multi_item_sizes():
    h = torch.rand(s, 9, 9, 32, device=dev, generator=g).to(torch.bfloat16)
    w8 = ((torch.rand(4, 4, 8, 32, device=dev, generator=g) - 0.5) * 0.2).to(torch.bfloat16)     # [kh,kw,out,in]
    b8 = (torch.rand(8, device=dev, generator=g) - 0.5) * 0.1
    q = K.pc_deconv_qmax(h, K.pc_deconv_taps(w8), b8, na)
    y = torch.relu(_conv64(h, w8.permute(3, 2, 0, 1), b8, stride=2, transpose=True))      # [S,20,20,8]: V, A_1..A_7
    adv = y[..., 1:1 + na]
    ref = y[..., 0] + adv.max(dim=3).values - adv.mean(dim=3)
    assert tuple(q.shape) == (s, 20, 20)
    assert torch.allclose(q.double(), ref, rtol=1e-4, atol=1e-5), (s, float((q.double() - ref).abs().max()))
    del y, adv, ref


def _bf16_close(got, want, ulps=1.0):
  """bf16 storage of a value computed in fp32: within `ulps` bf16 roundings (2^-8 relative each) of the fp32 reference."""
  return torch.allclose(got.float(), want, rtol=ulps * 2.0 ** -8, atol=1e-6)


def test_tile32_round_trip():
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  for n, c, dt in ((1, 256, torch.float32), (77, 256, torch.float32), (64, 1024, torch.bfloat16), (100, 1024, torch.bfloat16)):
    x = torch.randn(n, c, device=dev).to(dt)
    xt = K.tile32(x)
    assert xt.shape == ((n + 31) // 32 * 32, c) and torch.equal(K.untile32(xt, n), x)
    e = 16 // x.element_size()
    r, ch = n - 1, 3                      # chunk ch of row r sits at chunk index (r // 32 * chunks + ch) * 32 + r % 32
    at = ((r // 32) * (c // e) + ch) * 32 + r % 32
    assert torch.equal(xt.reshape(-1)[at * e:(at + 1) * e], x[r, ch * e:(ch + 1) * e])


@pytest.mark.parametrize("tiled", [False, True], ids=["row-major", "tiled"])
@pytest.mark.parametrize("n", [1, 100, 128, 1161, 4096])
def test_lstm_step_fwd_equals_gemm_plus_cell(n, tiled):
  """unreal_lstm_step_fwd (the BasicLSTMCell in the step GEMM's epilogue, model.py:110, :343-351) against an fp32 torch
  evaluation of the same step on the same bf16 operands, and against the two-kernel path it replaces; ragged row counts,
  the row-slice operand of the unroll, c / activations row-major and in the kernels' tiled layout, the acting variant
  (state in place, inactive rows untouched)."""
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  g = torch.Generator(device=dev).manual_seed(n)
  kx, kc = 264, 520
  xh3 = (torch.randn(2, n + 3, kc, device=dev, generator=g)).to(torch.bfloat16)      # [t, rows, kc]: step 0 feeds step 1
  xh3[:, :, 261:kx] = 0
  w = (torch.randn(kc, 1024, device=dev, generator=g) * 0.06).to(torch.bfloat16)
  bias = torch.randn(1024, device=dev, generator=g) * 0.1
  c0 = torch.randn(n, 256, device=dev, generator=g)
  xh = xh3[0, :n]
  z = xh.float() @ w.float() + bias
  i, j, f, o = z.split(256, dim=1)
  i, j, f, o = torch.sigmoid(i), torch.tanh(j), torch.sigmoid(f + 1.0), torch.sigmoid(o)
  c_ref = c0 * f + i * j
  h_ref = torch.tanh(c_ref) * o
  sentinel = 7.25
  nt = (n + 31) // 32 * 32 if tiled else n
  pad = 0 if tiled else 2
  c1b = torch.full((nt + pad, 256), sentinel, device=dev); h1 = torch.full((n + 2, 256), sentinel, device=dev)
  actsb = torch.full((nt + pad, 1024), sentinel, device=dev).to(torch.bfloat16)
  before = xh3[1].clone()
  K.lstm_step_fwd(xh, w, bias, K.tile32(c0) if tiled else c0, c1b[:nt], h_out=h1[:n], h16_out=xh3[1, :n, kx:], acts=actsb[:nt],
                  tiled=tiled)
  torch.cuda.synchronize()
  c1 = K.untile32(c1b, nt) if tiled else c1b
  acts = K.untile32(actsb, nt) if tiled else actsb
  assert torch.allclose(c1[:n], c_ref, rtol=1e-5, atol=2e-5), float((c1[:n] - c_ref).abs().max())
  assert torch.allclose(h1[:n], h_ref, rtol=1e-5, atol=2e-5)
  assert _bf16_close(acts[:n], torch.cat([i, j, f, o], dim=1))
  assert torch.equal(xh3[1, :n, kx:], h1[:n].to(torch.bfloat16)), "h' as bf16 in the next step's operand columns"
  # nothing outside the addressed rows / columns (tiled: the padding rows of the last 32-row block)
  assert (c1[n:] == sentinel).all() and (h1[n:] == sentinel).all() and (acts[n:].float() == sentinel).all()
  assert torch.equal(xh3[1, :, :kx], before[:, :kx]) and torch.equal(xh3[1, n:], before[n:])
  # the two-kernel path on f32 gates
  gates = K.gemm_bf16(xh, w, b_mn_major=True, bias=bias)
  c2 = torch.empty(n, 256, device=dev); h2 = torch.empty(n, 256, device=dev)
  h16 = torch.empty(n, 256, device=dev, dtype=torch.bfloat16)
  K.lstm_cell_fwd(gates, c0, c2, h2, h16)
  assert torch.allclose(c1[:n], c2, rtol=1e-5, atol=1e-5) and torch.allclose(h1[:n], h2, rtol=1e-5, atol=1e-5)
  if tiled:
    return
  # acting: persistent state in place, rows with active == 0 keep c / h and report their old h
  active = (torch.rand(n, device=dev, generator=g) < 0.6).to(torch.uint8)
  c_state = c0.clone(); h_state = torch.randn(n, 256, device=dev, generator=g); h_old = h_state.clone()
  h_rep = torch.full((n, 256), sentinel, device=dev)
  K.lstm_step_fwd(xh, w, bias, c_state, c_state, h_out=h_state, active=active, h_copy=h_rep)
  on = active.bool()[:, None]
  assert torch.equal(c_state, torch.where(on, c1[:n], c0)) and torch.equal(h_state, torch.where(on, h1[:n], h_old))
  assert torch.equal(h_rep, h_state)


@pytest.mark.parametrize("tiled", [False, True], ids=["row-major", "tiled"])
@pytest.mark.parametrize("last", [False, True], ids=["recurrent", "last-step"])
@pytest.mark.parametrize("n", [1, 100, 1161, 8192])
def test_lstm_step_bwd_equals_gemm_plus_cell_bwd(n, last, tiled):
  """unreal_lstm_step_bwd (recurrent dh GEMM with the cell's backward pass in its epilogue) against the two kernels it
  replaces (unreal_gemm_bf16 + unreal_lstm_cell_bwd_g16, themselves checked against autograd through the oracle tests) and
  against torch autograd of the cell on the same bf16 activations.  `last`: the unroll's last step (no product; dh2)."""
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  g = torch.Generator(device=dev).manual_seed(100 + n)
  w = (torch.randn(520, 1024, device=dev, generator=g) * 0.06).to(torch.bfloat16)
  wh = w[264:]
  dg_next = (torch.randn(n, 1024, device=dev, generator=g) * 0.1).to(torch.bfloat16)
  dh2 = torch.randn(n, 256, device=dev, generator=g) * 0.1
  z = torch.randn(n, 1024, device=dev, generator=g)
  acts = torch.cat([torch.sigmoid(z[:, :256]), torch.tanh(z[:, 256:512]), torch.sigmoid(z[:, 512:])], dim=1).to(torch.bfloat16)
  c_prev = torch.randn(n, 256, device=dev, generator=g)
  a = acts.float()
  c = c_prev * a[:, 512:768] + a[:, :256] * a[:, 256:512]
  dh = torch.randn(n, 256, device=dev, generator=g) * 0.1
  dc0 = torch.randn(n, 256, device=dev, generator=g) * 0.1
  sentinel = 3.5
  nt = (n + 31) // 32 * 32 if tiled else n
  T_ = (lambda x: K.tile32(x)) if tiled else (lambda x: x)
  dcb = torch.full((nt + 2, 256), sentinel, device=dev)
  dcb[:nt] = T_(dc0) if not tiled else torch.where(K.tile32(torch.ones(n, 256, device=dev)) > 0, K.tile32(dc0), dcb[:nt])
  dgates = torch.full((n + 2, 1024), sentinel, device=dev).to(torch.bfloat16)
  K.lstm_step_bwd(None if last else dg_next, wh, T_(acts), T_(c_prev), T_(c), dh, dcb[:nt], dgates[:n], dh2=dh2 if last else None,
                  tiled=tiled)
  torch.cuda.synchronize()
  dc = K.untile32(dcb[:nt], nt) if tiled else dcb
  assert (dc[n:nt] == sentinel).all() and (dcb[nt:] == sentinel).all() and (dgates[n:].float() == sentinel).all()
  # the kernels it replaces
  dh_rec = dh2 if last else K.gemm_bf16(dg_next, wh)
  dc_b = dc0.clone(); dg_b = torch.empty(n, 1024, device=dev, dtype=torch.bfloat16)
  K.lstm_cell_bwd(acts, c_prev, c, dh, dc_b, dg_b, dh_rec)
  assert torch.allclose(dc[:n], dc_b, rtol=1e-4, atol=1e-6), float((dc[:n] - dc_b).abs().max())
  assert _bf16_close(dgates[:n], dg_b.float(), ulps=2.0)
  # autograd of the cell in fp32 at the same activations: d/d(pre-activation) through sigmoid' = s (1 - s), tanh' = 1 - t^2
  dh_tot = dh + (dh2 if last else dg_next.float() @ wh.float().t())
  i, j, f, o = a[:, :256], a[:, 256:512], a[:, 512:768], a[:, 768:]
  tc = torch.tanh(c)
  dct = dc0 + dh_tot * o * (1 - tc * tc)
  want = torch.cat([dct * j * i * (1 - i), dct * i * (1 - j * j), dct * c_prev * f * (1 - f), dh_tot * tc * o * (1 - o)], dim=1)
  assert torch.allclose(dgates[:n].float(), want, rtol=2.0 ** -7, atol=1e-4)
  assert torch.allclose(dc[:n], dct * f, rtol=1e-4, atol=1e-5)


def test_fused_lstm_steps_equal_the_two_kernel_unroll():
  """UnrealModel.fused_lstm_step: the whole update (loss, gradient) with one launch per LSTM step against GEMM + cell
  kernels per step.  The two differ in ONE rounding: the two-kernel path stores the gate pre-activations as bf16 before
  the cell reads them (2^-9 relative on z), the fused path feeds the cell from the fp32 accumulator."""
  dev = torch.device("cuda", 0)
  feed = _to(_feed(6, 5, 4, seed=11), dev)
  out = {}
  for fused in (True, False):
    m = _model(dev, seed=5, n=5)
    m.fused_lstm_step = fused
    m.fused_lstm_min_rows = 1          # the unroll's one-launch steps at any batch size
    total, _, grad = m.loss_and_grads(feed)
    out[fused] = (float(total), grad.clone())
  assert abs(out[True][0] - out[False][0]) <= 2e-3 * abs(out[False][0])
  ga, gb = out[True][1], out[False][1]
  assert float((ga - gb).norm()) <= 2e-2 * float(gb.norm())
  # and each against the oracle that rounds what that path rounds (same bounds as test_loss_and_gradients_match_oracle)
  from oracle import model_oracle as M
  cpu_feed = {k: {kk: vv.cpu() for kk, vv in v.items()} for k, v in feed.items()}
  for fused in (True, False):
    m = _model(dev, seed=5, n=5)
    params = {k: v.detach().cpu().clone() for k, v in m.named_vars().items()}
    o = M.ModelOracle(params, A, 0, 0.05, 0.001, emulate_bf16=True, round_gates=not fused)
    rtotal, _, rgrads = o.loss_and_grads(cpu_feed)
    assert abs(out[fused][0] - float(rtotal)) <= 2e-3 * max(1.0, abs(float(rtotal))), fused
    got = {k: v.cpu() for k, v in m._views(out[fused][1]).items()}
    for k, rg in rgrads.items():
      err = float((got[k] - rg).abs().max())
      assert err <= 3e-2 * float(rg.abs().max()) + 1e-6, (fused, k, err, float(rg.abs().max()))
