"""Pins the numpy oracle against fixtures produced by the REFERENCE's own code
(tests/golden/make_golden.py).  CPU only."""
import hashlib
import os

import numpy as np
import pytest

from oracle import unreal_oracle as O
from fake_net import FakeNet

PC_PROBE = np.array([0, 19, 21, 63, 105, 147, 168, 189, 210, 231, 252, 294, 336, 378, 380, 399])


def _load(golden_dir, name):
  with np.load(os.path.join(golden_dir, name)) as z:   # NpzFile re-inflates on every [] access
    return {k: z[k] for k in z.files}


def test_maze_rollout_matches_reference(golden_dir):
  g = _load(golden_dir, "maze_golden.npz")
  env = O.MazeOracle()
  assert np.array_equal(env.last_state['image'].astype(np.uint8), g["initial_frame"])
  init = env.last_state['image']
  assert init[:, :, 0].sum() == 2160 and init[:, :, 1].sum() == 144 and init[:, :, 2].sum() == 0
  rs = np.random.RandomState(0xA3C)
  p = np.full(4, 0.25, np.float32)
  h_tr = hashlib.sha256()
  h_pc = hashlib.sha256()
  for i in range(len(g["actions"])):
    a = rs.choice(4, p=p)
    image, r, t, pc = env.process(a)
    assert (a, env.x, env.y, r, int(t)) == (g["actions"][i], g["x"][i], g["y"][i], g["reward"][i],
                                            g["terminal"][i])
    h_tr.update(bytes([int(a), env.x, env.y, r & 0xff, int(t)]))
    h_pc.update(pc.astype(np.float32).tobytes())
    if i < 64:
      assert np.array_equal(pc, g["first_pc"][i])
    if t:
      env.reset()
  assert h_tr.digest() == g["sha_transitions"].tobytes()
  assert h_pc.digest() == g["sha_pc_f32"].tobytes()
  assert h_tr.hexdigest().startswith("e93ee1fe3b3c931b")   # SURVEY.md 8(c)
  assert h_pc.hexdigest().startswith("f2871154166d891a")


def test_all_cell_action_pairs_and_closed_form(golden_dir):
  g = _load(golden_dir, "maze_golden.npz")
  tab, pcs = g["pair_table"], g["pair_pc"]
  assert len(tab) == 34 * 4
  distinct = set()
  for (x, y, a, nx, ny, r, t), pc in zip(tab, pcs):
    assert O.maze_step(int(x), int(y), int(a)) == (nx, ny, r, bool(t))
    lit = O.pixel_change(O.maze_render(int(nx), int(ny)), O.maze_render(int(x), int(y)))
    assert np.array_equal(lit, pc)                      # literal restatement, float64 exact
    cf = O.maze_pixel_change_closed_form(int(x), int(y), int(nx), int(ny))
    assert cf.dtype == np.float32
    assert np.array_equal(cf, pc.astype(np.float32))    # closed form == reference in fp32
    distinct.add(cf.tobytes())
  assert len(distinct) == 43                            # SURVEY.md 8(a) a6
  # out-of-range action: no move, reward 0
  assert O.maze_step(0, 2, 7) == (0, 2, 0, False)


@pytest.mark.parametrize("name", ["h2000", "h64", "h16", "h40neg"])
def test_ring_indices_match_reference(golden_dir, name):
  g = _load(golden_dir, "experience_golden.npz")
  H, L, seed, n, every = [int(v) for v in g[name + "_cfg"]]
  rewards, terms, log = g[name + "_reward"], g[name + "_terminal"], g[name + "_log"]
  ring = O.RingOracle(H, np.random.RandomState(seed))
  k = 0
  for i in range(n):
    ring.add(dict(reward=int(rewards[i]), terminal=bool(terms[i]), serial=i))
    if ring.is_full() and i % every == 0:
      start, cnt = ring.sample_sequence_index(L)
      assert (i, 0, start, cnt, ring.top, len(ring.pos_idx), len(ring.neg_idx)) == tuple(log[k])
      k += 1
      s = ring.sample_rp_index()
      assert (i, 1, s, s + 3 + ring.top, ring.top, len(ring.pos_idx), len(ring.neg_idx)) == tuple(log[k])
      k += 1
  assert k == len(log)


@pytest.mark.parametrize("name", ["h2000", "h100"])
def test_rollout_targets_match_reference(golden_dir, name):
  g = _load(golden_dir, "trainer_%s.npz" % name)
  H, n_iter, n_step, seed, net_seed, n_fill = [int(v) for v in g["cfg"]]
  rs = np.random.RandomState(seed)
  w = O.RolloutOracle(H, rs, FakeNet(net_seed), n_step_TD=n_step)
  fills = 0
  while not w.ring.is_full():
    w.fill_step()
    fills += 1
  assert fills == n_fill
  bi = pi = vi = 0
  for it in range(n_iter):
    b = w.process_base()
    assert len(b['pos']) == g["base_len"][it]
    for k in range(len(b['pos'])):
      assert tuple(b['pos'][k]) == tuple(g["base_pos"][bi])
      assert np.array_equal(b['lar'][k], g["base_lar"][bi])
      assert np.array_equal(b['a'][k], g["base_a"][bi])
      assert b['R'][k] == g["base_R"][bi] and b['adv'][k] == g["base_adv"][bi]
      bi += 1
    p = w.process_pc()
    assert len(p['pos']) == g["pc_len"][it]
    for k in range(len(p['pos'])):
      assert tuple(p['pos'][k]) == tuple(g["pc_pos"][pi])
      assert np.array_equal(p['lar'][k], g["pc_lar"][pi])
      assert np.array_equal(p['a'][k], g["pc_a"][pi])
      m = np.asarray(p['R'][k], np.float64)
      assert np.sum(m, dtype=np.float64) == g["pc_R_sum"][pi]
      assert np.array_equal(m.reshape(-1)[PC_PROBE].astype(np.float32), g["pc_R_probe"][pi])   # stored as float32
      if pi < len(g["pc_R_head"]):
        assert np.array_equal(m.astype(np.float32), g["pc_R_head"][pi])
      pi += 1
    v = w.process_vr()
    assert len(v['pos']) == g["vr_len"][it]
    for k in range(len(v['pos'])):
      assert tuple(v['pos'][k]) == tuple(g["vr_pos"][vi])
      assert np.array_equal(v['lar'][k], g["vr_lar"][vi])
      assert v['R'][k] == g["vr_R"][vi]
      vi += 1
    r = w.process_rp()
    assert np.array_equal(np.array(r['pos']), g["rp_pos"][it])
    assert r['c'] == list(g["rp_c"][it])
  assert (w.ring.top, w.local_t) == tuple(g["final_top"])
  lrs = [O.anneal_learning_rate(7.0710678e-4, t, 13200000)
         for t in (0, 1, 6600000, 13199999, 13200000, 14000000)]
  assert lrs == list(g["lr_anneal"])


def test_nstep_segmented_equals_rollout_form():
  rs = np.random.RandomState(0)
  T, N = 20, 64
  r = rs.randint(-1, 2, size=(T, N)).astype(np.float32)
  v = rs.randn(T, N).astype(np.float32)
  boot = rs.randn(N).astype(np.float32)
  term = np.zeros((T, N), np.uint8)
  term[-1, ::3] = 1                        # reference rollouts: terminal only at the end
  R, adv = O.nstep_returns_segmented(r, v, term, boot, 0.99, np.float32)
  for n in range(N):
    b = np.float32(0) if term[-1, n] else boot[n]
    R1, adv1 = O.nstep_returns(r[:, n], v[:, n], b, 0.99, np.float32)
    assert np.array_equal(R[:, n], R1) and np.array_equal(adv[:, n], adv1)


def test_rmsprop_known_answer():
  """train/rmsprop_applier_test.py:9-53 (lr=2, decay=.9, momentum=0, eps=1; rms0=1)."""
  for dt, tol in ((np.float64, 1e-15), (np.float32, 1e-6)):
    var = [np.array([1.0, 2.0], dt)]
    rms = [np.ones(2, dt)]
    mom = [np.zeros(2, dt)]
    n0 = O.rmsprop_step(var, rms, mom, [np.array([2.0, 4.0], dt)], 2.0, 0.9, 0.0, 1.0, 40.0, dt)
    np.testing.assert_allclose(var[0], [-1.6375218935831484, -2.2761798705987903], rtol=tol)
    np.testing.assert_allclose(rms[0], [1.3, 2.5], rtol=tol)
    np.testing.assert_allclose(n0, np.sqrt(20.0), rtol=tol)
    O.rmsprop_step(var, rms, mom, [np.array([3.0, 6.0], dt)], 2.0, 0.9, 0.0, 1.0, 40.0, dt)
    np.testing.assert_allclose(var[0], [-5.061902766795246, -6.861144190004011], rtol=tol)
    np.testing.assert_allclose(rms[0], [2.07, 5.85], rtol=tol)


def test_global_norm_clip():
  g = [np.full(100, 3.0, np.float32), np.full(300, -4.0, np.float32)]
  clipped, norm = O.clip_by_global_norm(g, 40.0)
  np.testing.assert_allclose(norm, np.sqrt(100 * 9 + 300 * 16), rtol=1e-6)
  np.testing.assert_allclose(O.global_norm(clipped), 40.0, rtol=1e-6)
  small, n2 = O.clip_by_global_norm([np.ones(4, np.float32)], 40.0)
  assert np.array_equal(small[0], np.ones(4, np.float32)) and n2 == 2.0


def test_generic_frame_rollout_targets_match_reference(golden_dir):
  """SURVEY 8f-4: the REFERENCE's Trainer._fill_experience / _process_base / _pc / _vr / _rp and Experience, driven
  on a generic-frame env (frames as `uint8 / 255` float32, float rewards, episode ends: the lab / gym / indoor
  process() shape), against the oracle's RolloutOracle on the same frame stream: sampled frames by checksum,
  last_action_reward vectors, actions, n-step returns / advantages, PC and VR targets, RP classes, ring top."""
  import zlib
  g = _load(golden_dir, "trainer_frames_h120.npz")
  H, n_iter, n_step, seed, net_seed, n_fill, table_seed = [int(v) for v in g["cfg"]]
  crc = lambda img: zlib.crc32(np.ascontiguousarray(img, np.float32).tobytes())   # noqa: E731
  rs = np.random.RandomState(seed)
  w = O.RolloutOracle(H, rs, FakeNet(net_seed, 3), n_step_TD=n_step, action_size=3,
                      env=O.TableFrameEnvOracle(0, O.make_frame_table(table_seed)))
  fills = 0
  while not w.ring.is_full():
    w.fill_step()
    fills += 1
  assert fills == n_fill
  bi = pi = vi = 0
  ended = 0
  for it in range(n_iter):
    b = w.process_base()
    ended += int(b['terminal_end'])
    assert len(b['states']) == g["base_len"][it]
    for k in range(len(b['states'])):
      assert crc(b['states'][k]['image']) == g["base_crc"][bi]
      assert np.array_equal(b['lar'][k], g["base_lar"][bi]) and np.array_equal(b['a'][k], g["base_a"][bi])
      assert b['R'][k] == g["base_R"][bi] and b['adv'][k] == g["base_adv"][bi]
      bi += 1
    p = w.process_pc()
    assert len(p['states']) == g["pc_len"][it]
    for k in range(len(p['states'])):
      assert crc(p['states'][k]['image']) == g["pc_crc"][pi]
      assert np.array_equal(p['lar'][k], g["pc_lar"][pi]) and np.array_equal(p['a'][k], g["pc_a"][pi])
      m = np.asarray(p['R'][k], np.float64)
      assert np.sum(m, dtype=np.float64) == g["pc_R_sum"][pi]
      assert np.array_equal(m.reshape(-1)[PC_PROBE], g["pc_R_probe"][pi])
      pi += 1
    v = w.process_vr()
    assert len(v['states']) == g["vr_len"][it]
    for k in range(len(v['states'])):
      assert crc(v['states'][k]['image']) == g["vr_crc"][vi]
      assert np.array_equal(v['lar'][k], g["vr_lar"][vi]) and v['R'][k] == g["vr_R"][vi]
      vi += 1
    r = w.process_rp()
    assert [crc(s['image']) for s in r['states']] == list(g["rp_crc"][it])
    assert r['c'] == list(g["rp_c"][it])
  assert ended > 50, "the fixture covers rollouts that end in a terminal"
  assert (w.ring.top, w.local_t) == tuple(g["final_top"])


def test_generic_pixel_change_matches_reference(golden_dir):
  """Environment._calc_pixel_change (environment.py:88-99) of the REFERENCE on float32 `uint8 / 255` frames of
  several sizes / channel counts, against the oracle's restatement: bit-equal float32 maps."""
  g = _load(golden_dir, "pixel_change_golden.npz")
  n = len([k for k in g if k.startswith("pc")])
  assert n == 5
  for i in range(n):
    a = g["a%d" % i].astype(np.float32) / np.float32(255.0)
    b = g["b%d" % i].astype(np.float32) / np.float32(255.0)
    pc = O.pixel_change(a, b)
    assert pc.dtype == g["pc%d" % i].dtype and pc.shape == g["pc%d" % i].shape
    assert np.array_equal(pc, g["pc%d" % i]), i


def test_concat_action_and_reward_matches_reference(golden_dir):
  """ExperienceFrame.concat_action_and_reward (experience.py:34-46) with and without the state's objective vector."""
  g = _load(golden_dir, "lar_golden.npz")
  for i in range(len(g["action"])):
    a, r = int(g["action"][i]), float(g["reward"][i])
    assert np.array_equal(O.concat_action_and_reward(a, 3, r, g["objective"][i]), g["with_obj"][i])
    assert np.array_equal(O.concat_action_and_reward(a, 3, r), g["without"][i])
