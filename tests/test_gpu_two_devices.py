"""One process, two devices.  The opt-in above 48 KB of dynamic shared memory is a function attribute of the device that
was current when it was set, and the maze layout lives in each device's constant memory: the library's lazy set-up has
to happen once per device, not once per process.  Every kernel family that opts in runs on device 0 and then, on the
same inputs, on device 1, where it must launch and give device 0's results; the maze steps on device 1 with a map that
was set while device 0 was current."""
import pytest
import torch

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two CUDA devices in one process")]

_GEMM_TUNABLES = {"gemm_bn": 0, "gemm_2sm": -1, "gemm_2sm_bn": 0}

MAP = ("S-----+"
       "-++++-+"
       "----+--"
       "+-+-+-+"
       "--+---+"
       "-+++-+-"
       "-----+G")


def _inputs(s=600, seed=0):
  """Seeded CPU tensors for every family below (s samples: more than the two CTAs per SM the persistent kernels launch)."""
  g = torch.Generator().manual_seed(seed)
  rn = lambda *shape: torch.randn(*shape, generator=g)
  bf = lambda *shape, scale=1.0: (rn(*shape) * scale).to(torch.bfloat16)
  n = 1100                                                    # LSTM rows: 9 row blocks of 128, the last ragged
  z = rn(n, 1024)
  return {
      "a": bf(1024, 1024), "b": bf(512, 1024),
      "frames": torch.randint(0, 256, (s, 84, 84, 3), generator=g, dtype=torch.uint8),
      "pos": torch.randint(0, 7, (s, 2), generator=g, dtype=torch.int32),
      "w1": bf(8, 8, 3, 16, scale=0.05), "b1": rn(16) * 0.1,
      "w2": bf(4, 4, 16, 32, scale=0.05), "b2": rn(32) * 0.1,
      "dy1": bf(2, s * 400, 8), "dy2": bf(s * 81, 32), "dyp": bf(s, 4, 100, 8),
      "hp": torch.relu(rn(s, 2592)).to(torch.bfloat16), "w8": bf(4, 4, 8, 32, scale=0.05), "b8": rn(8) * 0.1,
      "act": torch.randint(0, 4, (s,), generator=g, dtype=torch.int32), "tgt": torch.rand(s, 400, generator=g),
      "msk": torch.ones(s), "scale": torch.tensor([0.7]),
      "xh": bf(n, 520), "wx": bf(520, 1024, scale=0.06), "bias": rn(1024) * 0.1, "c0": rn(n, 256),
      "dg_next": bf(n, 1024, scale=0.1), "dh": rn(n, 256) * 0.1, "dc": rn(n, 256) * 0.1,
      "acts": torch.cat([torch.sigmoid(z[:, :256]), torch.tanh(z[:, 256:512]), torch.sigmoid(z[:, 512:])], 1).to(torch.bfloat16),
      "seq8": torch.randint(0, 256, (150, 3, 84, 84, 3), generator=g, dtype=torch.uint8),
      "seg": rn(4099, 256), "seg_pos": torch.randint(0, 7, (4099, 2), generator=g, dtype=torch.int32),
  }


def _run(dev, x):
  """Every family that opts into large dynamic shared memory, on `dev` (the current device): name -> output on the CPU."""
  from unreal_b200 import _lib, kernels as K
  x = {k: v.to(dev) for k, v in x.items()}
  out = {}
  try:
    for build, kv in (("1cta", {"gemm_bn": 256, "gemm_2sm": 0}), ("pair", {"gemm_2sm": 1, "gemm_2sm_bn": 256})):
      for k, v in dict(_GEMM_TUNABLES, **kv).items():
        _lib.set_tunable(k, v)
      out["gemm_" + build] = K.gemm_bf16(x["a"], x["b"])
  finally:
    for k, v in _GEMM_TUNABLES.items():
      _lib.set_tunable(k, v)
  xpp = K.s2d_frames(x["frames"])
  w1p = K.conv1_w_planes(x["w1"])
  out["conv1"] = h1 = K.conv_fwd(xpp, 1, w1p, x["b1"])
  out["conv1_maze"] = K.conv1_fwd_maze(x["pos"], w1p, x["b1"])
  out["conv2"] = K.conv_fwd(h1, 2, K.conv_taps(x["w2"], 2), x["b2"])
  out["sum:conv1_wgrad"] = K.conv1_wgrad(xpp, x["dy1"])
  out["sum:conv2_wgrad"] = K.conv2_wgrad(h1, x["dy2"])
  out["conv2_dgrad"] = K.conv2_dgrad(x["dy2"], K.conv2_dgrad_taps(x["w2"]))
  loss, dy16, db8 = K.pc_deconv_loss(x["hp"], K.pc_deconv_taps(x["w8"]), x["b8"], x["act"], x["tgt"], x["msk"], 4, 0.05)
  out.update({"sum:pc_loss": loss, "pc_loss_dy": dy16, "sum:pc_loss_db": db8})
  dpc, db = K.pc_planes_conv(x["dyp"], K.pc_w_planes(x["w8"]), x["hp"], x["scale"])
  out.update({"pc_planes_conv": dpc, "sum:pc_planes_conv_db": db})
  out["sum:pc_planes_wgrad"] = K.pc_planes_wgrad(x["dyp"], x["hp"])
  n = x["xh"].shape[0]
  c1, h1s = torch.empty(n, 256, device=dev), torch.empty(n, 256, device=dev)
  acts = torch.empty(n, 1024, device=dev, dtype=torch.bfloat16)
  K.lstm_step_fwd(x["xh"], x["wx"], x["bias"], x["c0"], c1, h_out=h1s, acts=acts)
  out.update({"lstm_fwd_c": c1, "lstm_fwd_h": h1s, "lstm_fwd_acts": acts})
  a = x["acts"].float()
  c = x["c0"] * a[:, 512:768] + a[:, :256] * a[:, 256:512]
  dc, dgates = x["dc"].clone(), torch.empty(n, 1024, device=dev, dtype=torch.bfloat16)
  K.lstm_step_bwd(x["dg_next"], x["wx"][264:], x["acts"], x["c0"], c, x["dh"], dc, dgates)
  out.update({"lstm_bwd_dc": dc, "lstm_bwd_dgates": dgates})
  out["pc84_u8"] = K.pixel_change_stream(x["seq8"])
  out["pc84_f32"] = K.pixel_change_stream(x["seq8"].float() / 255.0)
  out["sum:cell_segment_sum"] = K.cell_segment_sum(x["seg"], x["seg_pos"])
  torch.cuda.synchronize(dev)
  return {k: v.cpu() for k, v in out.items()}


def test_kernel_families_on_a_second_device():
  """Kernels without float atomics give device 0's bits; those that add with red.global.add (filter gradients, bias
  gradients, the loss, segment sums) add in a run-dependent order and agree to fp32 summation rounding."""
  x = _inputs()
  got = []
  for d in (0, 1):
    dev = torch.device("cuda", d)
    with torch.cuda.device(dev):
      got.append(_run(dev, x))
  ref, dev1 = got
  assert ref.keys() == dev1.keys()
  for k in ref:
    a, b = ref[k], dev1[k]
    assert bool(torch.isfinite(a.double()).all()), "%s: non-finite on device 0" % k
    if k.startswith("sum:"):
      err = float((a.double() - b.double()).abs().max())
      assert err <= 1e-5 * float(a.double().abs().max()), "%s: device 1 differs from device 0 by %g" % (k, err)
    else:
      assert torch.equal(a, b), "%s: device 1 differs from device 0" % k


def test_maze_map_set_on_one_device_applies_on_another():
  """A map set while device 0 is current steps and renders on device 1 as on device 0, and maze_layout() reports it."""
  from unreal_b200 import kernels as K
  t, n = 8, 300
  actions = torch.randint(0, 4, (t, n), generator=torch.Generator().manual_seed(1), dtype=torch.int32)
  try:
    with torch.cuda.device(0):
      K.maze_set_map(MAP)
    got = []
    for d in (0, 1):
      dev = torch.device("cuda", d)
      with torch.cuda.device(dev):
        st = K.MazeState(n, dev)
        obs = torch.empty(t, n, 84, 84, 3, device=dev)
        rec = torch.empty(t, n, dtype=torch.int64, device=dev)
        rew, term = K.maze_window(st, actions.to(dev), obs=obs, frame_rec=rec, auto_reset=True)
        torch.cuda.synchronize(dev)
        got.append({"obs": obs.cpu(), "reward": rew.cpu(), "terminal": term.cpu(), "rec": rec.cpu(), "pos": st.pos.cpu(),
                    "layout": K.maze_layout()})
    ref, dev1 = got
    for k in ref:
      assert (ref[k] == dev1[k]) if k == "layout" else torch.equal(ref[k], dev1[k]), "%s: device 1 differs" % k
    start, goal, walls = dev1["layout"]
    assert (start, goal) == ((0, 0), (6, 6))
    assert walls == bytes(1 if c == "+" else 0 for c in MAP)
    # the map is not the reference's: walls are drawn where MAP has them (channel 0 of the cell's 12 x 12 block)
    wall_px = dev1["obs"][0, :, 12 * 1 + 5, 12 * 1 + 5, 0]
    assert bool((wall_px == 1.0).all())
  finally:
    with torch.cuda.device(0):
      K.maze_set_map(None)
