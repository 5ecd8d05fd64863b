"""K7 GEMM (tcgen05) against a float64 torch matmul of the same bf16-rounded operands.

Tolerance: operands are exactly representable, products are exact in fp32 and the accumulation
is fp32, so the only differences to the float64 reference are fp32 summation rounding
(<= K * 2^-24 relative to sum |a||b|) and, for bf16 outputs, the final rounding (2^-9).
"""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ref(a, b, a_mn, b_mn, bias=None, add=None, relu=False):
  A = a.double().t() if a_mn else a.double()
  B = b.double() if b_mn else b.double().t()
  c = A @ B
  if bias is not None:
    c = c + bias.double()
  if add is not None:
    c = c + add.double()
  if relu:
    c = c.clamp_min(0)
  return c


def _mk(shape, seed, dev):
  g = torch.Generator(device=dev).manual_seed(seed)
  return (torch.randn(*shape, device=dev, generator=g) * 0.5).to(torch.bfloat16)


CASES = [
    # m, n, k, a_mn, b_mn
    (128, 128, 64, False, False),
    (256, 128, 256, False, False),
    (1000, 256, 2592, False, False),     # fc1 with a K-major weight shadow
    (1000, 256, 2592, False, True),      # fc1 with TF's [in,out] layout (model.py:337-340)
    (300, 1024, 264, False, True),       # LSTM input projection
    (777, 2592, 256, False, True),       # pc_fc1 (model.py:424)
    (4000, 16, 192, False, False),       # conv1 as im2col GEMM
    (810, 32, 256, False, False),        # conv2
    (810, 80, 32, False, False),         # deconv taps
    (555, 2592, 256, False, False),      # dgrad through fc1: dY [S,256] x W[2592,256]^T
    (2592, 256, 5000, True, True),       # wgrad fc1: X^T dY
    (16, 192, 4000, True, True),         # wgrad conv1 (small M padded by TMA)
    (264, 1024, 640, True, True),
    (96, 64, 200, True, False),
]


@pytest.mark.parametrize("m,n,k,a_mn,b_mn", CASES)
def test_gemm_matches_float64(m, n, k, a_mn, b_mn):
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  a = _mk((k, m) if a_mn else (m, k), 1, dev)
  b = _mk((k, n) if b_mn else (n, k), 2, dev)
  c = K.gemm_bf16(a, b, a_mn_major=a_mn, b_mn_major=b_mn)
  torch.cuda.synchronize()
  ref = _ref(a, b, a_mn, b_mn)
  scale = (a.double().abs().t() if a_mn else a.double().abs()) @ (b.double().abs() if b_mn else b.double().abs().t())
  err = ((c.double() - ref).abs() / scale.clamp_min(1e-6)).max().item()
  assert err <= k * 2.0 ** -23, err


def test_gemm_epilogue_bias_add_relu_bf16():
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  m, n, k = 700, 2592, 256
  a, b = _mk((m, k), 3, dev), _mk((k, n), 4, dev)
  bias = torch.randn(n, device=dev)
  add = torch.randn(m, n, device=dev)
  ref = _ref(a, b, False, True, bias, add, True)
  c32 = K.gemm_bf16(a, b, b_mn_major=True, bias=bias, add=add, relu=True)
  assert torch.allclose(c32.double(), ref, rtol=1e-4, atol=1e-4)
  c16 = K.gemm_bf16(a, b, b_mn_major=True, bias=bias, add=add, relu=True, out_dtype=torch.bfloat16)
  assert torch.allclose(c16.double(), ref, rtol=2.0 ** -7, atol=1e-2)


def test_gemm_strided_views_and_ragged_k():
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  m, n, k = 333, 1024, 261                      # LSTM input: 256 + A + 1 columns of a 264-wide buffer
  abuf = _mk((m, 264), 5, dev)
  wbuf = _mk((261 + 256, n), 6, dev)            # [in, out] kernel of BasicLSTMCell: x rows then h rows
  a = abuf[:, :k]
  b = wbuf[:k]
  out_buf = torch.zeros(m, n + 8, device=dev)
  c = K.gemm_bf16(a, b, out=out_buf[:, :n], b_mn_major=True)
  ref = _ref(a, b, False, True)
  assert torch.allclose(c.double(), ref, rtol=1e-4, atol=1e-4)
  assert float(out_buf[:, n:].abs().max()) == 0.0


def test_gemm_split_k_and_accumulate():
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  kk, m, n = 20000, 2592, 256
  x, dy = _mk((kk, m), 7, dev), _mk((kk, n), 8, dev)
  ref = _ref(x, dy, True, True)
  c = K.gemm_bf16(x, dy, a_mn_major=True, b_mn_major=True, split_k=7)
  assert torch.allclose(c.double(), ref, rtol=1e-3, atol=1e-2)
  K.gemm_bf16(x, dy, out=c, a_mn_major=True, b_mn_major=True, accumulate=True, split_k=3)
  assert torch.allclose(c.double(), 2 * ref, rtol=1e-3, atol=2e-2)


def test_gemm_rejects_bad_arguments():
  from unreal_b200 import _lib, kernels as K
  dev = torch.device("cuda", 0)
  a, b = _mk((64, 60), 1, dev), _mk((64, 60), 2, dev)    # ld 60 is not a multiple of 8
  with pytest.raises(_lib.UnrealError):
    K.gemm_bf16(a, b)
  with pytest.raises(_lib.UnrealError):
    K.gemm_bf16(_mk((64, 64), 1, dev), _mk((64, 72), 2, dev))
  # the TMA-store epilogue reads the bias as float4: a bias 4 bytes off a 16-byte boundary is refused, not launched
  a, b = _mk((256, 64), 1, dev), _mk((64, 64), 2, dev)
  bias = torch.zeros(65, device=dev)[1:]
  with pytest.raises(_lib.UnrealError):
    K.gemm_bf16(a, b, bias=bias)


# ---- every kernel instantiation, forced through the tunables, at shapes that run each CTA's tile loop >= 3 times ----
# unreal_gemm_bf16 picks one of 26 builds: gemm_tcgen05_kernel<BN, A_MN, B_MN, DEEP> (14 with 4 epilogue warps, 4 with
# 8) and gemm2sm_tcgen05_kernel<BN, A_MN, B_MN> (8, CTA pairs on 256-row tiles).  Small or natural-dispatch problems reach
# only a few of them, with one tile per CTA; the tests below force each build and check it against float64.
_TUNABLE_DEFAULTS = {"gemm_bn": 0, "gemm_2sm": -1, "gemm_2sm_bn": 0, "gemm_deep_epilogue": -1, "gemm_tma_store": 1}


@pytest.fixture
def tunables():
  """force(**kv) sets GEMM tunables for this test; the defaults are restored afterwards whatever happens."""
  from unreal_b200 import _lib

  def force(**kv):
    for k, v in dict(_TUNABLE_DEFAULTS, **kv).items():
      assert k in _TUNABLE_DEFAULTS, k
      _lib.set_tunable(k, v)
  try:
    force()
    yield force
  finally:
    for k, v in _TUNABLE_DEFAULTS.items():
      _lib.set_tunable(k, v)


BUILDS = ([("1cta", bn, amn, bmn) for bn in (32, 64, 128, 256) for amn in (False, True) for bmn in (False, True)
           if not (bn == 32 and bmn)] +                                   # BN 32 with an MN-major B is raised to 64
          [("deep", bn, False, bmn) for bn in (128, 256) for bmn in (False, True)] +    # deep: K-major A only
          [("pair", bn, amn, bmn) for bn in (128, 256) for amn in (False, True) for bmn in (False, True)])
assert len(BUILDS) == 26


def _build_id(b):
  return "%s-%d-%s-%s" % (b[0], b[1], "Amn" if b[2] else "Ak", "Bmn" if b[3] else "Bk")


def _force_build(force, build, tma):
  kind, bn = build[:2]
  if kind == "pair":
    force(gemm_2sm=1, gemm_2sm_bn=bn, gemm_tma_store=tma)
  else:
    force(gemm_bn=bn, gemm_2sm=0, gemm_deep_epilogue=1 if kind == "deep" else 0, gemm_tma_store=tma)


def _kernel_of(build):
  """The instantiation a forced build launches: (kernel, BN, A_MN, B_MN[, DEEP])."""
  kind, bn, amn, bmn = build
  if kind == "pair":
    return ("gemm2sm_tcgen05_kernel", bn, amn, bmn)
  return ("gemm_tcgen05_kernel", bn, amn, bmn, kind == "deep")


def _stages(build):
  kind, bn = build[:2]
  if kind == "deep":
    return 3 if bn >= 256 else 5
  if kind == "pair":
    return 6 if bn == 256 else 8
  return 4 if bn >= 256 else (6 if bn >= 128 else 8)


def _sms():
  return torch.cuda.get_device_properties(0).multi_processor_count


def _multi_tile_shape(build):
  """(m, n, k): two column tiles, the second ragged (n % 32 != 0: the epilogue's scalar bias branch); enough 128-row
  tiles that every CTA -- or CTA pair -- runs at least 3 of them; m = 256 q + 64, so the last 256-row tile of a pair
  has no rows for its second CTA; k = 64 kStages + 1 wraps the shared-memory stage ring inside every tile."""
  bn = build[1]
  n = bn + bn // 2 + 8                 # rows of whole 16-byte chunks: C is stored with TMA in both dtypes
  num_n = 2
  sms = _sms()
  q = -(-3 * sms // (2 * num_n))
  m = 256 * q + 64
  tiles = -(-m // 128) * num_n if build[0] != "pair" else -(-m // 256) * num_n
  ctas = sms if build[0] != "pair" else sms // 2
  assert tiles >= 3 * ctas, (m, n, tiles)
  return m, n, 64 * _stages(build) + 1


def _edge_shapes(build):
  n = _multi_tile_shape(build)[1]
  # n - 3: rows that are not whole 16-byte chunks, which the epilogue writes with element stores
  edges = [(1, n, 24), (127, n, 8), (129, n, 24), (257, n, 8), (129, n - 3, 24)]
  if build[0] != "pair":           # the pair kernel needs n > 128
    edges += [(129, 24, 24), (129, 20, 24)]
  return edges


def _operand(rows, cols, seed, dev, pad=8):
  """bf16 [rows, cols] view of a buffer whose leading dimension is padded with NaN: a kernel that reads past the
  matrix (TMA boxes are clipped at `cols` and must zero-fill) produces NaN."""
  ld = (cols + 7) // 8 * 8 + pad
  buf = torch.full((rows, ld), float("nan"), device=dev, dtype=torch.bfloat16)
  buf[:, :cols] = _mk((rows, cols), seed, dev)
  return buf[:, :cols]


def _guarded_out(m, n, dtype, dev, fill=None):
  """C as [m, n] view of a NaN buffer with 8 padding columns (ldc > n) and 16 padding rows."""
  ldc = (n + 7) // 8 * 8 + 8
  buf = torch.full((m + 16, ldc), float("nan"), device=dev, dtype=dtype)
  c = buf[:m, :n]
  if fill is not None:
    c.copy_(fill)
  return buf, c


def _assert_guard_bands(buf, m, n, what):
  assert bool(torch.isnan(buf[:m, n:]).all()) and bool(torch.isnan(buf[m:]).all()), "%s wrote outside C" % what


def _assert_close(c, ref, scale, k, bf16, splits, what):
  """|C - ref| <= K * 2^-23 * (|A||B| + |bias| + |add| + |C0|) elementwise, times the number of partial sums added on the
  atomic paths, plus one bf16 rounding of |ref| for bf16 outputs.  K is the reduction the kernel runs: k rounded up to
  its 64-wide blocks (the padding is zero-filled by TMA)."""
  kk = (k + 63) // 64 * 64
  tol = kk * 2.0 ** -23 * scale * splits
  if bf16:
    tol = tol + 2.0 ** -8 * ref.abs()
  err = (c.double() - ref).abs()
  bad = ~(err <= tol)                     # NaN counts as bad
  if bool(bad.any()):
    i = int(bad.flatten().nonzero()[0])
    r, col = divmod(i, ref.shape[1])
    raise AssertionError("%s: %d of %d elements off, first at [%d, %d]: got %r want %r (tol %.3g)" % (
        what, int(bad.sum()), bad.numel(), r, col, float(c[r, col]), float(ref[r, col]), float(tol[r, col])))


def _run_case(m, n, k, a_mn, b_mn, out_dtype, epilogues, dev, seed=0, what=""):
  """One product through every listed epilogue, each into a guarded C, against float64."""
  from unreal_b200 import kernels as K
  a = _operand(k, m, seed + 1, dev) if a_mn else _operand(m, k, seed + 1, dev)
  b = _operand(k, n, seed + 2, dev) if b_mn else _operand(n, k, seed + 2, dev)
  g = torch.Generator(device=dev).manual_seed(seed + 3)
  bias = torch.randn(n, device=dev, generator=g)
  addbuf = torch.randn(m, (n + 7) // 8 * 8 + 8, device=dev, generator=g)     # row pitch of _guarded_out's C
  base = _ref(a, b, a_mn, b_mn)
  absa = a.double().abs().t() if a_mn else a.double().abs()
  scale0 = absa @ (b.double().abs() if b_mn else b.double().abs().t())
  bf16 = out_dtype == torch.bfloat16
  kb = (k + 63) // 64
  for epi in epilogues:
    use_bias = epi in ("bias", "bias_add_relu", "accumulate", "split2", "splitmax")
    use_add = epi in ("add", "bias_add_relu", "accumulate", "split2", "splitmax")
    relu = epi == "bias_add_relu"
    split = {"split2": 2, "splitmax": kb}.get(epi, 1)
    acc = epi == "accumulate"
    c0 = torch.randn(m, n, device=dev, generator=g) if acc else (torch.zeros(m, n, device=dev) if split > 1 else None)
    if bf16 and c0 is not None:
      continue                          # accumulation needs an f32 C
    buf, c = _guarded_out(m, n, out_dtype, dev, c0)
    add = addbuf[:, :n] if use_add else None            # the addend is read with C's row stride (ldc)
    K.gemm_bf16(a, b, out=c, a_mn_major=a_mn, b_mn_major=b_mn, bias=bias if use_bias else None, add=add, relu=relu,
                accumulate=acc, split_k=split, out_dtype=out_dtype)
    torch.cuda.synchronize()
    ref, scale = base, scale0
    if use_bias:
      ref, scale = ref + bias.double(), scale + bias.double().abs()
    if use_add:
      ref, scale = ref + add.double(), scale + add.double().abs()
    if c0 is not None:
      ref, scale = ref + c0.double(), scale + c0.double().abs()
    if relu:
      ref = ref.clamp_min(0)
    tag = "%s %s [%d,%d,%d] %s" % (what, epi, m, n, k, out_dtype)
    _assert_guard_bands(buf, m, n, tag)
    _assert_close(c, ref, scale, k, bf16, split if split > 1 else 1, tag)


_EPILOGUES = ("bias", "add", "bias_add_relu", "accumulate", "split2", "splitmax")


@pytest.mark.parametrize("tma", [1, 0], ids=["tma-store", "element-store"])
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("build", BUILDS, ids=[_build_id(b) for b in BUILDS])
def test_gemm_forced_build_matches_float64(build, out_dtype, tma, tunables):
  """Each build at >= 3 tiles per CTA (both TMEM accumulators, mbarrier phases and the stage ring wrapping across tiles)
  and at the edge shapes, with every epilogue: bias, addend, bias + addend + ReLU and, for f32 outputs, accumulation
  into a nonzero C and split-K (2 and one split per K block) with bias and addend applied once."""
  if build[0] == "deep" and not tma:
    pytest.skip("the deep-epilogue build stores with TMA only")
  dev = torch.device("cuda", 0)
  _force_build(tunables, build, tma)
  epis = _EPILOGUES if out_dtype == torch.float32 else _EPILOGUES[:3]
  m, n, k = _multi_tile_shape(build)
  _run_case(m, n, k, build[2], build[3], out_dtype, epis, dev, seed=10, what=_build_id(build))
  for i, (m, n, k) in enumerate(_edge_shapes(build)):
    _run_case(m, n, k, build[2], build[3], out_dtype, epis, dev, seed=20 + 3 * i, what=_build_id(build))


def _launched_gemm_kernels(prof):
  """(kernel, BN, A_MN, B_MN[, DEEP]) of every GEMM kernel in the trace, in launch order."""
  import re
  demangled = re.compile(r"(gemm2sm_tcgen05_kernel|gemm_tcgen05_kernel)<\s*(\d+)\s*,\s*(true|false)\s*,\s*(true|false)"
                         r"\s*(?:,\s*(true|false)\s*)?>")
  mangled = re.compile(r"(gemm2sm_tcgen05_kernel|gemm_tcgen05_kernel)ILi(\d+)ELb([01])ELb([01])E(?:Lb([01])E)?")
  found = []
  for e in prof.events():
    mt = demangled.search(e.name) or mangled.search(e.name)
    if mt is None:
      continue
    flag = lambda s: s in ("true", "1")          # noqa: E731
    key = (mt.group(1), int(mt.group(2)), flag(mt.group(3)), flag(mt.group(4)))
    if mt.group(1) == "gemm_tcgen05_kernel":
      key += (flag(mt.group(5)) if mt.group(5) is not None else False,)
    found.append((e.time_range.start, key))
  return [key for _, key in sorted(found)]


def test_gemm_forced_builds_launch_all_26_instantiations(tunables):
  """The forced matrix really reaches every instantiation: under torch.profiler, each forced build launches exactly
  the kernel it names.  A change to the dispatch or the tunables that silently reroutes a build fails here."""
  from torch.profiler import profile, ProfilerActivity
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  cases = []
  for build in BUILDS:
    m, n, k = 257, _multi_tile_shape(build)[1], 72
    a = _operand(k, m, 1, dev) if build[2] else _operand(m, k, 1, dev)
    b = _operand(k, n, 2, dev) if build[3] else _operand(n, k, 2, dev)
    cases.append((build, a, b))
  outs = []
  torch.cuda.synchronize()
  with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for build, a, b in cases:
      _force_build(tunables, build, 1)
      outs.append(K.gemm_bf16(a, b, a_mn_major=build[2], b_mn_major=build[3]))
      torch.cuda.synchronize()
  launched = _launched_gemm_kernels(prof)
  want = [_kernel_of(b) for b, _, _ in cases]
  assert launched == want, (launched, want)
  assert len(set(launched)) == 26
  for (build, a, b), c in zip(cases, outs):
    ref = _ref(a, b, build[2], build[3])
    scale = (a.double().abs().t() if build[2] else a.double().abs()) @ (b.double().abs() if build[3] else b.double().abs().t())
    _assert_close(c, ref, scale, a.shape[0] if build[2] else a.shape[1], False, 1, _build_id(build))


def test_gemm_odd_ldc_falls_back_to_element_stores(tunables):
  """A C whose row pitch is not 16-byte aligned cannot be a TMA tensor: the epilogue stores elements / atomics instead,
  inside the same guard bands."""
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  m, n, k = 1000, 300, 200
  a, b = _operand(m, k, 1, dev), _operand(k, n, 2, dev)
  bias = torch.randn(n, device=dev)
  ref0 = _ref(a, b, False, True)
  scale0 = a.double().abs() @ b.double().abs()
  for dtype in (torch.float32, torch.bfloat16):
    for acc in ((False, True) if dtype == torch.float32 else (False,)):
      buf = torch.full((m + 16, n + 3), float("nan"), device=dev, dtype=dtype)
      c = buf[:m, :n]
      c0 = torch.randn(m, n, device=dev) if acc else None
      if acc:
        c.copy_(c0)
      K.gemm_bf16(a, b, out=c, b_mn_major=True, bias=bias, accumulate=acc, relu=not acc, out_dtype=dtype)
      torch.cuda.synchronize()
      ref, scale = ref0 + bias.double(), scale0 + bias.double().abs()
      if acc:
        ref, scale = ref + c0.double(), scale + c0.double().abs()
      else:
        ref = ref.clamp_min(0)
      _assert_guard_bands(buf, m, n, "ldc %d %s" % (n + 3, dtype))
      _assert_close(c, ref, scale, k, dtype == torch.bfloat16, 1, "ldc %d %s acc %d" % (n + 3, dtype, acc))


# ---- the model's call sites at production batch sizes, natural dispatch ------------------------------------------------
def _site(name, s):
  """(m, n, k, a_mn, b_mn, out dtype, bias, relu, split_k) of one unreal_gemm_bf16 call of model/layers.py at S samples
  (1024 envs x T = 20 is S = 20 480)."""
  from unreal_b200.model.layers import split_k_for
  return {
      "fc1_fwd": (s, 256, 2592, False, True, torch.bfloat16, True, True, 1),          # LinearFn.forward, h2 -> fc1
      "fc1_dgrad": (s, 2592, 256, False, False, torch.bfloat16, False, False, 1),     # LinearFn.backward, dx
      "fc1_wgrad": (2592, 256, s, True, True, torch.float32, False, False, split_k_for(2592, 256, s)),
      "pc_fc1_fwd": (s, 2592, 256, False, True, torch.bfloat16, True, True, 1),       # PcTowerFusedFn.forward
      "pc_fc1_dgrad": (s, 256, 2592, False, False, torch.float32, False, False, 1),   # dx of the f32 LSTM output
      "pc_fc1_wgrad": (256, 2592, s, True, True, torch.float32, False, False, split_k_for(256, 2592, s)),
      "lstm_wgrad": (520, 1024, s, True, True, torch.float32, False, False, split_k_for(520, 1024, s)),
  }[name]


@pytest.mark.parametrize("s", [1024, 20480])
@pytest.mark.parametrize("site", ["fc1_fwd", "fc1_dgrad", "fc1_wgrad", "pc_fc1_fwd", "pc_fc1_dgrad", "pc_fc1_wgrad",
                                  "lstm_wgrad"])
def test_gemm_model_call_sites_at_production_sizes(site, s, tunables):
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  m, n, k, a_mn, b_mn, dtype, use_bias, relu, split = _site(site, s)
  a = _operand(k, m, 1, dev, pad=0) if a_mn else _operand(m, k, 1, dev, pad=0)
  b = _operand(k, n, 2, dev, pad=0) if b_mn else _operand(n, k, 2, dev, pad=0)
  bias = torch.randn(n, device=dev) if use_bias else None
  buf, c = _guarded_out(m, n, dtype, dev, torch.zeros(m, n, device=dev) if split > 1 else None)
  K.gemm_bf16(a, b, out=c, a_mn_major=a_mn, b_mn_major=b_mn, bias=bias, relu=relu, split_k=split, out_dtype=dtype)
  torch.cuda.synchronize()
  ref = _ref(a, b, a_mn, b_mn, bias, None, relu)
  scale = (a.double().abs().t() if a_mn else a.double().abs()) @ (b.double().abs() if b_mn else b.double().abs().t())
  if bias is not None:
    scale = scale + bias.double().abs()
  _assert_guard_bands(buf, m, n, site)
  _assert_close(c, ref, scale, k, dtype == torch.bfloat16, split, "%s S=%d split %d" % (site, s, split))


@pytest.mark.parametrize("gates_dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_gemm_lstm_step_at_1024_envs(gates_dtype, tunables):
  """LstmFn's per-step product (layers.py, unfused steps): [N, 520] step operands of the [T, N, 520] buffer x the
  concatenated kernel [520, 1024] + bias, at N = 1024 envs."""
  from unreal_b200 import kernels as K
  dev = torch.device("cuda", 0)
  t, n_env = 3, 1024
  xh = _mk((t, n_env, 520), 1, dev)
  w = _mk((520, 1024), 2, dev)
  bias = torch.randn(1024, device=dev)
  gates = torch.full((t, n_env + 16, 1024), float("nan"), device=dev, dtype=gates_dtype)
  for i in range(t):
    K.gemm_bf16(xh[i], w, out=gates[i, :n_env], b_mn_major=True, bias=bias, out_dtype=gates_dtype)
  torch.cuda.synchronize()
  for i in range(t):
    ref = _ref(xh[i], w, False, True, bias)
    scale = xh[i].double().abs() @ w.double().abs() + bias.double().abs()
    _assert_close(gates[i, :n_env], ref, scale, 520, gates_dtype == torch.bfloat16, 1, "lstm step %d" % i)
    assert bool(torch.isnan(gates[i, n_env:]).all())
