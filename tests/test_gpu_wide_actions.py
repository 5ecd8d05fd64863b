"""8 to 15 actions: the 16-channel pixel-control head (unreal_pc_deconv_loss16 / unreal_pc_deconv_qmax16) and the 15-wide
policy / value head kernels, from the kernels up through UnrealModel, FrameTrainer and Evaluator.

  * kernels against float64 (transposed convolution + dueling loss; torch heads), at S = 64, just past one wave and 20 480;
  * outputs inside NaN guard bands;
  * the model against oracle/model_oracle.py with the tolerances of tests/test_gpu_model.py's A = 4 comparisons;
  * which kernels run (profiler), the errors, and a registered 12-action env end to end."""
import numpy as np
import pytest
import torch

DEV = torch.device("cuda", 0)


def _sms():
  return torch.cuda.get_device_properties(0).multi_processor_count


# ---- 1. the 16-channel pixel-control kernels against float64 ----------------------------------------------------------
def _pc_case(s, a, seed):
  g = torch.Generator(device=DEV).manual_seed(seed)
  hp = torch.randn(s, 9, 9, 32, device=DEV, generator=g).to(torch.bfloat16)
  w16 = torch.zeros(4, 4, 16, 32, device=DEV)
  w16[:, :, :1 + a] = torch.randn(4, 4, 1 + a, 32, device=DEV, generator=g) * 0.1
  w16 = w16.to(torch.bfloat16)
  b16 = torch.zeros(16, device=DEV)
  b16[:1 + a] = torch.randn(1 + a, device=DEV, generator=g) * 0.3       # both signs: both halves of the ReLU
  act = torch.randint(0, a, (s,), device=DEV, generator=g, dtype=torch.int32)
  tgt = torch.rand(s, 400, device=DEV, generator=g) * 2.0
  mask = (torch.rand(s, device=DEV, generator=g) < 0.8).float()          # masked samples
  return hp, w16, b16, act, tgt, mask


def _pc_ref(hp, w16, b16, act, tgt, mask, a, lam):
  """float64: pre-ReLU deconv output [S,20,20,16], loss, d loss / d pre, q-max."""
  s = hp.shape[0]
  w = w16.double().permute(3, 2, 0, 1)                  # [kh,kw,out,in] -> [in,out,kh,kw]
  pre = torch.nn.functional.conv_transpose2d(hp.double().permute(0, 3, 1, 2), w, b16.double(), stride=2)
  pre = pre.permute(0, 2, 3, 1).contiguous().requires_grad_(True)
  y = torch.relu(pre)
  adv = y[..., 1:1 + a]
  q = y[..., 0:1] + adv - adv.mean(-1, keepdim=True)
  qa = q.gather(-1, act.long().view(s, 1, 1, 1).expand(s, 20, 20, 1))[..., 0]
  loss = lam * 0.5 * (((tgt.double().view(s, 20, 20) - qa) ** 2) * mask.double().view(s, 1, 1)).sum()
  loss.backward()
  return pre.detach(), loss.detach(), pre.grad, q.detach().max(-1).values


@pytest.mark.gpu
@pytest.mark.parametrize("a", [8, 11, 15])
def test_pc_deconv_loss16_and_qmax16_match_float64(a):
  from unreal_b200 import kernels as K
  lam = 0.05
  for s in (64, 2 * _sms() + 1, 20480):
    hp, w16, b16, act, tgt, mask = _pc_case(s, a, seed=s + a)
    taps = K.conv2_dgrad_taps(w16)
    loss, dy16, db16 = K.pc_deconv_loss(hp, taps, b16, act, tgt, mask, a, lam)
    qmax = K.pc_deconv_qmax(hp, taps, b16, a)
    pre, rloss, rgrad, rq = _pc_ref(hp, w16, b16, act, tgt, mask, a, lam)
    assert dy16.shape == (s, 400, 16) and db16.shape == (16,)
    assert abs(float(loss) - float(rloss)) <= 1e-4 * abs(float(rloss)), (s, float(loss), float(rloss))
    got = dy16.view(s, 20, 20, 16).double()
    # elements whose pre-activation sits within fp32 accumulation noise of 0 may take the other side of the ReLU
    settled = pre.abs() > 1e-4
    err = ((got - rgrad).abs() - 2.0 ** -8 * rgrad.abs())[settled]
    assert float(err.max()) <= 1e-5 * float(rgrad.abs().max()), s
    assert not got[..., 1 + a:].any(), "channels past the actions carry no gradient"
    assert ((rgrad != 0) & settled).any() and ((pre < 0) & settled).any()
    rdb = got.sum((0, 1, 2))                                          # db sums the rounded values
    assert torch.allclose(db16.double(), rdb, rtol=0, atol=1e-4 * float(got.abs().sum((0, 1, 2)).max()) + 1e-6), s
    assert torch.allclose(db16.double(), rgrad.sum((0, 1, 2)), rtol=0, atol=2.0 ** -7 * float(rgrad.abs().sum((0, 1, 2)).max())), s
    assert torch.allclose(qmax.double(), rq, rtol=1e-4, atol=1e-4 * float(rq.abs().max())), s


@pytest.mark.gpu
def test_pc16_kernels_write_inside_nan_guard_bands():
  from unreal_b200 import _lib, kernels as K
  s, a, pad = 2 * _sms() + 3, 13, 1024
  hp, w16, b16, act, tgt, mask = _pc_case(s, a, seed=5)
  taps = K.conv2_dgrad_taps(w16)
  dyb = torch.full((pad + s * 6400 + pad,), float("nan"), dtype=torch.bfloat16, device=DEV)
  dbb = torch.full((pad + 16 + pad,), float("nan"), device=DEV); dbb[pad:pad + 16] = 0
  qb = torch.full((pad + s * 400 + pad,), float("nan"), device=DEV)
  loss = torch.zeros(1, dtype=torch.float64, device=DEV)
  sp = _lib.stream_ptr()
  _lib.call("unreal_pc_deconv_loss16", hp.data_ptr(), taps.data_ptr(), b16.data_ptr(), act.data_ptr(), tgt.data_ptr(),
            mask.data_ptr(), a, 0.05, s, loss.data_ptr(), dyb[pad:].data_ptr(), dbb[pad:].data_ptr(), sp)
  _lib.call("unreal_pc_deconv_qmax16", hp.data_ptr(), taps.data_ptr(), b16.data_ptr(), a, s, qb[pad:].data_ptr(), sp)
  torch.cuda.synchronize()
  for buf, n in ((dyb, s * 6400), (dbb, 16), (qb, s * 400)):
    assert bool(buf[:pad].isnan().all()) and bool(buf[pad + n:].isnan().all())
    assert not bool(buf[pad:pad + n].isnan().any())
  ref_loss, ref_dy, ref_db = K.pc_deconv_loss(hp, taps, b16, act, tgt, mask, a, 0.05)
  assert torch.equal(dyb[pad:pad + s * 6400].view(s, 400, 16), ref_dy)
  assert torch.equal(qb[pad:pad + s * 400].view(s, 20, 20), K.pc_deconv_qmax(hp, taps, b16, a))


# ---- 2. the 15-wide head kernels against float64 ------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("a", [8, 12, 15])
def test_wide_head_kernels_match_float64(a):
  from unreal_b200 import kernels as K
  for m in (64, 64 * _sms() + 1, 20480):        # 64 rows per pass of the persistent loss grid
    g = torch.Generator(device=DEV).manual_seed(m + a)
    h = torch.randn(m, 256, device=DEV, generator=g)
    wp = torch.randn(256, a, device=DEV, generator=g) * 0.1; bp = torch.randn(a, device=DEV, generator=g) * 0.1
    wv = torch.randn(256, device=DEV, generator=g) * 0.1; bv = torch.randn(1, device=DEV, generator=g)
    act = torch.randint(0, a, (m,), device=DEV, generator=g, dtype=torch.int32)
    adv = torch.randn(m, device=DEV, generator=g); ret = torch.randn(m, device=DEV, generator=g)
    mask = (torch.rand(m, device=DEV, generator=g) < 0.8).float()
    beta, coef = 0.01, 0.25
    out = K.a3c_head(h, wp, bp, wv, bv, act, adv, ret, mask, beta, coef, want_pi=True, want_v=True, want_sums=True,
                     want_grads=True)
    go2 = torch.tensor([0.7, 1.3], device=DEV)
    dh, dwp, dbp, dwv, dbv = K.a3c_head_bwd(h, wp, wv, out["dz"], out["dv"], go2)
    # float64 reference with autograd
    hd, wpd, bpd, wvd, bvd = (x.double().requires_grad_(True) for x in (h, wp, bp, wv, bv))
    z = hd @ wpd + bpd
    z.retain_grad()
    pi = torch.softmax(z, -1); v = hd @ wvd + bvd
    v.retain_grad()
    lp = torch.log(pi.clamp(1e-20, 1.0)); H = -(pi * lp).sum(-1)
    md, advd, retd = mask.double(), adv.double(), ret.double()
    pol = -((lp.gather(1, act.long().view(m, 1))[:, 0] * advd + beta * H) * md).sum()
    val = coef * (((retd - v) ** 2) * md).sum()
    (pol * 0.7 + val * 1.3).backward()
    close = lambda x, y, r=1e-4: torch.allclose(x.double(), y, rtol=r, atol=r * float(y.abs().max()) + 1e-7)  # noqa: E731
    assert close(out["pi"], pi.detach()) and close(out["v"], v.detach())
    sums = out["sums"]
    assert close(sums[0], pol.detach()) and close(sums[1], val.detach()) and close(sums[2], (H * md).sum().detach())
    assert close(out["dz"] * 0.7, z.grad, 1e-3) and close(out["dv"] * 1.3, v.grad, 1e-3)
    for x, y, name in ((dh, hd.grad, "dh"), (dwp, wpd.grad, "dwp"), (dbp, bpd.grad, "dbp"), (dwv, wvd.grad, "dwv"),
                       (dbv, bvd.grad, "dbv")):
      assert close(x, y, 1e-3), (m, a, name)


@pytest.mark.gpu
def test_wide_heads_write_inside_nan_guard_bands():
  from unreal_b200 import _lib, kernels as K
  m, a, pad = 1001, 15, 256
  g = torch.Generator(device=DEV).manual_seed(3)
  h = torch.randn(m, 256, device=DEV, generator=g)
  wp = torch.randn(256, a, device=DEV, generator=g) * 0.1; bp = torch.zeros(a, device=DEV)
  wv = torch.randn(256, device=DEV, generator=g) * 0.1; bv = torch.zeros(1, device=DEV)
  act = torch.randint(0, a, (m,), device=DEV, generator=g, dtype=torch.int32)
  adv = torch.randn(m, device=DEV, generator=g); ret = torch.randn(m, device=DEV, generator=g)
  nan = lambda n: torch.full((pad + n + pad,), float("nan"), device=DEV)  # noqa: E731
  pi, v, dz, dv, dh = nan(m * a), nan(m), nan(m * a), nan(m), nan(m * 256)
  sums = torch.zeros(3, dtype=torch.float64, device=DEV)
  sp = _lib.stream_ptr()
  _lib.call("unreal_a3c_head_loss", h.data_ptr(), wp.data_ptr(), bp.data_ptr(), wv.data_ptr(), bv.data_ptr(), act.data_ptr(),
            adv.data_ptr(), ret.data_ptr(), None, m, a, 0.01, 0.25, pi[pad:].data_ptr(), v[pad:].data_ptr(), sums.data_ptr(),
            dz[pad:].data_ptr(), dv[pad:].data_ptr(), sp)
  go2 = torch.ones(2, device=DEV)
  grads = [nan(256 * a), nan(a), nan(256), nan(1)]
  for t in grads:
    t[pad:-pad] = 0
  _lib.call("unreal_a3c_head_bwd", h.data_ptr(), wp.data_ptr(), wv.data_ptr(), dz[pad:].data_ptr(), dv[pad:].data_ptr(),
            go2.data_ptr(), m, a, dh[pad:].data_ptr(), *[t[pad:].data_ptr() for t in grads], sp)
  torch.cuda.synchronize()
  for buf in [pi, v, dz, dv, dh] + grads:
    assert bool(buf[:pad].isnan().all()) and bool(buf[-pad:].isnan().all())
    assert not bool(buf[pad:-pad].isnan().any())


# ---- 3. the model against the oracle -------------------------------------------------------------------------------
def _wide_model(a, g, n, seed, **kw):
  from unreal_b200.model.model import UnrealModel
  return UnrealModel(a, g, -1, True, True, True, True, 0.05, 0.001, DEV, {'segnet_mode': 0}, (84, 84), True, 0, 0.0, 0.0,
                     num_envs=n, seed=seed, **kw)


def _wide_feed(a, g, T, N, L, seed):
  """Trainer-shaped feed with u8 frames: (GPU feed, CPU feed with the frames as floats / 255)."""
  rs = np.random.RandomState(seed)

  def images(*lead):
    return torch.from_numpy(rs.randint(0, 256, size=lead + (84, 84, 3)).astype(np.uint8))

  def onehot(*lead):
    out = np.zeros(lead + (a,), np.float32)
    np.put_along_axis(out, rs.randint(0, a, size=lead + (1,)), 1.0, axis=-1)
    return torch.from_numpy(out)

  def lar(*lead):
    out = np.zeros(lead + (a + 1 + g,), np.float32)
    out[..., :a] = onehot(*lead).numpy()
    out[..., a] = rs.randint(-1, 2, size=lead)
    out[..., a + 1:] = rs.rand(*(lead + (g,)))
    return torch.from_numpy(out)

  def mask(t, n):
    m = np.ones((t, n), np.float32)
    m[t - 2:, 0] = 0
    return torch.from_numpy(m)

  f32 = lambda *s: torch.from_numpy(rs.randn(*s).astype(np.float32))  # noqa: E731
  rp_c = np.zeros((N, 3), np.float32); rp_c[np.arange(N), rs.randint(0, 3, N)] = 1
  feed = {
      "base": dict(images=images(T, N), lar=lar(T, N), a=onehot(T, N), adv=f32(T, N), R=f32(T, N), mask=mask(T, N),
                   c0=f32(N, 256) * 0.1, h0=f32(N, 256) * 0.1),
      "pc": dict(images=images(L, N), lar=lar(L, N), a=onehot(L, N),
                 R=torch.from_numpy(rs.rand(L, N, 20, 20).astype(np.float32)), mask=mask(L, N)),
      "vr": dict(images=images(L, N), lar=lar(L, N), R=f32(L, N), mask=mask(L, N)),
      "rp": dict(images=images(N, 3), c=torch.from_numpy(rp_c)),
  }
  gpu = {k: {kk: vv.to(DEV) for kk, vv in v.items()} for k, v in feed.items()}
  cpu = {k: {kk: (vv.float() / 255.0 if kk == "images" else vv) for kk, vv in v.items()} for k, v in feed.items()}
  return gpu, cpu


@pytest.mark.gpu
@pytest.mark.parametrize("g", [0, 2])
@pytest.mark.parametrize("a", [8, 12, 15])
def test_wide_model_loss_and_gradients_match_oracle(a, g):
  """Tolerances of test_gpu_model.py's A = 4 comparison, except that pc_fc1's two gradients are compared in L2 norm (1e-1)
  also against the emulating oracle: a pc_fc1 unit within accumulation noise of its ReLU threshold moves single elements
  of those gradients by several per cent of their maximum.  The 8-channel head of A = 4 on these u8 feeds shows the same
  (up to 0.16 of the maximum element-wise, 1.2e-2 in L2, measured on a B200); no other variable is affected."""
  from oracle import model_oracle as M
  m = _wide_model(a, g, 3, seed=a + g)
  assert m.pc_grad_layout == "c16"
  gpu, cpu = _wide_feed(a, g, 5, 3, 4, seed=a * 10 + g)
  total, parts, grad = m.loss_and_grads(gpu)
  got = {k: v.cpu() for k, v in m._views(grad).items()}
  params = {k: v.detach().cpu().clone() for k, v in m.named_vars().items()}
  for emulate, ftol, gtol in ((True, 2e-3, 3e-2), (False, 3e-2, 1e-1)):
    o = M.ModelOracle({k: v.clone() for k, v in params.items()}, a, g, 0.05, 0.001, emulate_bf16=emulate)
    rtotal, rparts, rgrads = o.loss_and_grads(cpu)
    for k in ("policy", "value", "pc", "vr", "rp"):
      assert abs(float(parts[k]) - float(rparts[k])) <= ftol * max(1.0, abs(float(rparts[k]))), (k, emulate)
    assert abs(float(total) - float(rtotal)) <= ftol * max(1.0, abs(float(rtotal)))
    for k, rg in rgrads.items():
      if emulate and k not in ("W_pc_fc1", "b_pc_fc1"):
        err = float((got[k] - rg).abs().max())
        assert err <= gtol * float(rg.abs().max()) + 1e-6, (k, emulate, err, float(rg.abs().max()))
      else:           # L2-relative at the fp32 oracle's tolerance
        err = float((got[k] - rg).norm() / rg.norm().clamp_min(1e-12))
        assert err <= 1e-1, (k, emulate, err)


@pytest.mark.gpu
@pytest.mark.parametrize("a", [8, 12, 15])
def test_wide_acting_helpers_match_oracle(a):
  from oracle import model_oracle as M
  m = _wide_model(a, 0, 3, seed=a)
  params = {k: v.detach().cpu().clone() for k, v in m.named_vars().items()}
  o = M.ModelOracle(params, a, 0, 0.05, 0.001, emulate_bf16=True)
  gpu, cpu = _wide_feed(a, 0, 2, 3, 2, seed=a)
  img, lar = cpu["base"]["images"], cpu["base"]["lar"]
  c = torch.zeros(3, 256); h = torch.zeros(3, 256)
  for t in range(2):
    pi, v, _ = m.run_base_policy_and_value(None, {'image': gpu["base"]["images"][t]}, gpu["base"]["lar"][t])
    rpi, rv, (c, h) = o.base_forward(img[t:t + 1], lar[t:t + 1], c, h)
    assert pi.shape == (3, a)
    assert torch.allclose(pi.cpu(), rpi[0], rtol=2e-3, atol=2e-4)
    assert torch.allclose(v.cpu(), rv[0], rtol=2e-3, atol=2e-3)
  qmax = m.run_pc_q_max(None, {'image': gpu["base"]["images"][1]}, gpu["base"]["lar"][1])
  rq = o.pc_forward(img[1:2], lar[1:2])[1][0]
  assert torch.allclose(qmax.cpu(), rq, rtol=2e-3, atol=2e-3)


# ---- 4. dispatch ---------------------------------------------------------------------------------------------------
def _kernel_names(prof):
  import re
  names = []
  for e in prof.events():
    n = re.sub(r"\s+", "", e.name)
    for pat in (r"conv2_dgrad_tcgen05_kernel(?:<|ILi)(\d+)(?:,|ELi)(\d+)(?:,|ELi)(\d+)(?:,|E)(?:Lb)?(true|false|1|0)",
                r"(a3c_head_loss_kernel)(?:<|ILi)(\d+)", r"(a3c_head_bwd_kernel)(?:<|ILi)(\d+)",
                r"(pc_planes_conv_tcgen05_kernel)"):
      mt = re.search(pat, n)
      if mt:
        names.append(tuple(x.replace("true", "1").replace("false", "0") for x in mt.groups()))
  return names


def _profile_update(a):
  from torch.profiler import profile, ProfilerActivity
  m = _wide_model(a, 0, 3, seed=1)
  gpu, _ = _wide_feed(a, 0, 5, 3, 4, seed=2)
  m.loss_and_grads(gpu)                      # warm-up
  torch.cuda.synchronize()
  with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
    m.loss_and_grads(gpu)
    torch.cuda.synchronize()
  ops = [e.name for e in prof.events()]
  return set(_kernel_names(prof)), ops


@pytest.mark.gpu
def test_dispatch_by_action_count():
  k4, ops4 = _profile_update(4)
  k12, ops12 = _profile_update(12)
  # A = 4: the 8-channel fused deconv + loss (compile-time A = 4), the plane-major backward, the 7-wide heads
  assert ("8", "8", "4", "0") in k4 and ("pc_planes_conv_tcgen05_kernel",) in k4
  assert ("a3c_head_loss_kernel", "7") in k4 and ("a3c_head_bwd_kernel", "7") in k4
  assert not any(k[:2] == ("16", "8") for k in k4) and ("a3c_head_loss_kernel", "15") not in k4
  # A = 12: the 16-channel export and the 15-wide heads; nothing of the 8-channel head, no torch softmax / extra matmuls
  assert ("16", "8", "0", "1") in k12
  assert ("a3c_head_loss_kernel", "15") in k12 and ("a3c_head_bwd_kernel", "15") in k12
  assert not any(k[0] == "8" for k in k12 if len(k) == 4) and ("pc_planes_conv_tcgen05_kernel",) not in k12
  assert not any("softmax" in n for n in ops12)
  mm = lambda ops: sum(n in ("aten::mm", "aten::matmul", "aten::addmm", "aten::bmm") for n in ops)  # noqa: E731
  assert mm(ops12) == mm(ops4)


# ---- 5. errors -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_wide_action_errors():
  from unreal_b200 import _lib, kernels as K
  with pytest.raises(_lib.UnrealError, match="15 actions"):
    _wide_model(16, 0, 2, seed=0)
  gpu, _ = _wide_feed(12, 0, 3, 2, 2, seed=1)
  for attr, value in (("fused_pc_loss", False), ("pc_grad_layout", "planes"), ("pc_grad_layout", "c8"),
                      ("fused_pc_relu", False)):
    m = _wide_model(12, 0, 2, seed=0)
    setattr(m, attr, value)
    with pytest.raises(_lib.UnrealError, match="c16"):
      m.loss(gpu)
  m = _wide_model(12, 0, 2, seed=0)
  m.fused_pc_loss = False
  with pytest.raises(_lib.UnrealError, match="c16"):
    m.run_pc_q_max(None, {'image': gpu["base"]["images"][0]}, gpu["base"]["lar"][0])
  hp, w16, b16, act, tgt, mask = _pc_case(8, 12, seed=0)
  taps = K.conv2_dgrad_taps(w16)
  with pytest.raises(_lib.UnrealError, match="action count"):
    K.pc_deconv_loss(hp, taps, b16, act, tgt, mask, 16, 0.05)
  with pytest.raises(_lib.UnrealError, match="action count"):
    K.pc_deconv_qmax(hp, taps, b16, 16)
  with pytest.raises(_lib.UnrealError, match="action count"):
    K.pc_deconv_loss(hp, taps, b16, act, tgt, mask, 7, 0.05)
  with pytest.raises(_lib.UnrealError):
    K.pc_deconv_loss(hp, taps, b16, act, tgt, mask, 12, 0.05, planes=True)


def test_new_exports_reject_out_of_range_action_counts_without_a_gpu():
  """Argument checks run before any device work: a = 16 (or 7) into the 16-channel exports, a = 16 into the heads."""
  import __graft_entry__ as ge
  ge.build()
  from unreal_b200 import _lib
  L = _lib.lib
  p = 4096                                    # any aligned non-null address: the call must fail before touching it
  for a in (16, 7):
    assert L.unreal_pc_deconv_loss16(p, p, p, p, p, p, a, 0.05, 4, p, p, p, None) != 0
    assert b"action count" in L.unreal_last_error()
    assert L.unreal_pc_deconv_qmax16(p, p, p, a, 4, p, None) != 0
    assert b"action count" in L.unreal_last_error()
  assert L.unreal_a3c_head_loss(p, p, p, p, p, None, None, None, None, 4, 16, 0.0, 0.25, None, None, None, None, None,
                                None) != 0
  assert b"action count" in L.unreal_last_error()
  assert L.unreal_a3c_head_bwd(p, p, p, None, None, p, 4, 16, p, None, None, None, None, None) != 0
  assert b"action count" in L.unreal_last_error()


# ---- 6. a registered 12-action env end to end ----------------------------------------------------------------------
def _register_wide():
  from unreal_b200.environment import frame_environment as FE
  from unreal_b200.environment.environment import Environment
  Environment.register('wide12', lambda name, args, tt, ti: FE.BatchedFrameEnvironment(
      FE.TableFrameProducer(args['num_envs'], args['device'], 12, seed=4 + ti), args['device']), action_size=12)
  Environment.action_size = -1


def _wide_trainer_run(graphs, n=6, updates=3):
  from unreal_b200.train.frame_trainer import FrameTrainer
  from unreal_b200.train.rmsprop_applier import RMSPropApplier
  from unreal_b200.train.trainer import Trainer
  net = _wide_model(12, 0, n, seed=2)
  ap = RMSPropApplier(7e-4, decay=0.99, momentum=0.0, epsilon=0.1, clip_norm=40.0)
  tr = Trainer(0, net, 7e-4, None, ap, 'wide12', '', True, True, True, True, 0.05, 0.001, 20, 20, 0.99, 0.9, 40, 10 ** 8,
               DEV, {'segnet_mode': 0}, (84, 84), True, 0, np.random.RandomState(1), 50.0, 0.0, 0.0, num_envs=n,
               seeds=np.arange(n) + 3, use_graphs=graphs)
  assert isinstance(tr, FrameTrainer)
  tr.prepare()
  while not tr.experience.is_full():
    tr.process(None, 0)
  before = net.flat.detach().clone()
  losses = []
  for _ in range(updates):
    tr.process(None, 0)
    losses.append({k: float(v) for k, v in tr.last_losses.items()})
  torch.cuda.synchronize()
  assert all(np.isfinite(list(l.values())).all() for l in losses), losses
  assert float((net.flat.detach() - before).abs().max()) > 0
  tr.stop()
  return net


@pytest.mark.gpu
def test_registered_twelve_action_env_trains_and_evaluates():
  from unreal_b200.environment.environment import Environment
  from unreal_b200.train.evaluator import Evaluator
  _register_wide()
  try:
    eager, eager2, graphed = _wide_trainer_run(False), _wide_trainer_run(False), _wide_trainer_run(True)
    spread = float((eager.flat - eager2.flat).abs().max())
    diff = float((graphed.flat - eager.flat).abs().max())
    assert diff <= max(4 * spread, 1e-7) or torch.allclose(graphed.flat, eager.flat, rtol=1e-3, atol=1e-5), (diff, spread)
    for mode in ("sample", "greedy"):
      ev = Evaluator(graphed, env_type='wide12', num_envs=16, mode=mode, max_episode_steps=30, device=DEV, use_graphs=False)
      out = ev.run(2)
      assert out["summary"]["episodes"] == 32
      assert (out["length"] >= 1).all() and (out["length"] <= 30).all()
  finally:
    Environment._registry.pop('wide12', None)
    Environment.action_size = -1
