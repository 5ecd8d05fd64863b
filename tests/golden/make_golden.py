#!/usr/bin/env python
"""Generate the golden fixtures in this directory FROM THE REFERENCE ITSELF.

Run only in the authoring container (needs the read-only reference tree):

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py [/root/reference]

It imports the reference's own modules unmodified:

* ``environment.maze_environment.MazeEnvironment``  (runs as is)
* ``train.experience.Experience / ExperienceFrame``  (runs as is)
* ``train.trainer.Trainer._process_base/_process_pc/_process_vr/_process_rp,
  choose_action, _anneal_learning_rate`` with ``tensorflow`` stubbed by
  ``MagicMock`` (the methods themselves are pure numpy) and the network replaced
  by ``fake_net.FakeNet``.  The maze needs the three-line ``MazeShim`` below
  because the fork's Trainer passes ``flag=`` and reads ``_last_full_state``
  (trainer.py:264, :285) which only IndoorEnvironment has (SURVEY.md section 0).

Nothing here is read at test time; the tests read the ``.npz`` files it writes.
The GPU box has no ``/root/reference``.
"""
import hashlib
import os
import sys
import types
from collections import deque
from unittest.mock import MagicMock

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = sys.argv[1] if len(sys.argv) > 1 else "/root/reference"
sys.dont_write_bytecode = True
sys.path.insert(0, REF)
sys.path.insert(0, HERE)

for m in ("tensorflow", "tensorflow.python", "tensorflow.python.client",
          "tensorflow.python.client.timeline", "tensorflow.contrib",
          "tensorflow.python.training", "tensorflow.python.training.training_ops",
          "tensorflow.python.training.slot_creator"):
  sys.modules[m] = MagicMock()

from environment.environment import Environment  # noqa: E402  (reference)
from environment.maze_environment import MazeEnvironment  # noqa: E402  (reference)
from train.experience import Experience, ExperienceFrame  # noqa: E402  (reference)
from train.trainer import Trainer  # noqa: E402  (reference)

from fake_net import FakeNet  # noqa: E402


def agent_pos(image):
  ys, xs = np.nonzero(image[:, :, 1])
  return int(xs.min()) // 12, int(ys.min()) // 12


# ---------------------------------------------------------------------------
# A. maze transitions, rewards, frames, pixel-change
# ---------------------------------------------------------------------------
def gen_maze():
  env = Environment.create_environment('maze', '')
  init = env.last_state['image']
  assert init.dtype == np.float64 and init.shape == (84, 84, 3)
  rs = np.random.RandomState(0xA3C)
  p = np.full(4, 0.25, np.float32)
  n = 6000
  act = np.zeros(n, np.uint8); xs = np.zeros(n, np.uint8); ys = np.zeros(n, np.uint8)
  rew = np.zeros(n, np.int8); term = np.zeros(n, np.uint8)
  h_tr = hashlib.sha256(); h_pc = hashlib.sha256()
  pcs = []
  for i in range(n):
    a = rs.choice(4, p=p)
    image, r, t, pc = env.process(a)
    act[i] = a; xs[i] = env.x; ys[i] = env.y; rew[i] = r; term[i] = t
    h_tr.update(bytes([int(a), env.x, env.y, r & 0xff, int(t)]))
    h_pc.update(pc.astype(np.float32).tobytes())
    if i < 64:
      pcs.append(pc.astype(np.float64))
    if t:
      env.reset()
  # every (free cell, action) pair: next cell, reward, terminal, pixel-change, frame sums
  rows = []
  pair_pc = []
  for y in range(7):
    for x in range(7):
      if env._is_wall(x, y):
        continue
      for a in range(4):
        env.reset()
        env.x, env.y = x, y
        env.last_state = {'image': env._get_current_image()}
        image, r, t, pc = env.process(a)
        assert agent_pos(image) == (env.x, env.y)
        rows.append((x, y, a, env.x, env.y, r, int(t)))
        pair_pc.append(pc)
  # out-of-range action is a no-op move with reward 0 (maze_environment.py:99-108)
  env.reset()
  image, r, t, pc = env.process(7)
  assert (env.x, env.y) == (0, 2) and r == 0 and not t and not pc.any()
  np.savez_compressed(
      os.path.join(HERE, "maze_golden.npz"),
      initial_frame=init.astype(np.uint8),
      actions=act, x=xs, y=ys, reward=rew, terminal=term,
      sha_transitions=np.frombuffer(h_tr.digest(), np.uint8),
      sha_pc_f32=np.frombuffer(h_pc.digest(), np.uint8),
      first_pc=np.stack(pcs),
      pair_table=np.array(rows, np.int16),
      pair_pc=np.stack(pair_pc))
  print("maze: sha tr", h_tr.hexdigest()[:16], "sha pc", h_pc.hexdigest()[:16],
        "episodes", int(term.sum()), "pairs", len(rows))


# ---------------------------------------------------------------------------
# B. replay ring: synthetic frame streams through the reference Experience
# ---------------------------------------------------------------------------
def gen_experience():
  out = {}
  cases = [  # (name, H, L, seed, n_frames, p_term, p_pos, sample_every)
      ("h2000", 2000, 21, 0xA3C, 6000, 0.02, 0.05, 20),
      ("h64", 64, 21, 7, 1500, 0.10, 0.20, 3),
      ("h16", 16, 5, 11, 600, 0.25, 0.02, 1),     # pos list often empty / single
      ("h40neg", 40, 9, 13, 600, 0.05, 0.97, 2),  # neg list often empty / single
  ]
  for name, H, L, seed, n, p_term, p_pos, every in cases:
    gen = np.random.RandomState(seed + 1000)
    rs = np.random.RandomState(seed)
    exp = Experience(H, rs)
    rewards = np.zeros(n, np.int8); terms = np.zeros(n, np.uint8)
    log = []   # rows: (frame_no, kind, v0, v1, top, npos, nneg) kind 0=seq 1=rp
    for i in range(n):
      u = gen.rand()
      reward = 1 if u < p_pos else (-1 if u < p_pos + 0.3 else 0)
      terminal = bool(gen.rand() < p_term)
      rewards[i] = reward; terms[i] = terminal
      fr = ExperienceFrame({'id': i}, reward, int(gen.randint(4)), terminal, None, 0, 0)
      fr.serial = None
      import io, contextlib
      with contextlib.redirect_stdout(io.StringIO()):   # "Terminal frames continued."
        exp.add_frame(fr)
      # tag with the absolute index the ring gave it (stays None when discarded)
      if exp._frames[-1] is fr:
        fr.serial = exp._top_frame_index + len(exp._frames) - 1
      if exp.is_full() and (i % every == 0):
        seq = exp.sample_sequence(L)
        start = seq[0].serial - exp._top_frame_index
        log.append((i, 0, start, len(seq), exp._top_frame_index,
                    len(exp._pos_reward_indices), len(exp._neg_reward_indices)))
        rp = exp.sample_rp_sequence()
        assert len(rp) == 4
        log.append((i, 1, rp[0].serial - exp._top_frame_index, rp[3].serial, exp._top_frame_index,
                    len(exp._pos_reward_indices), len(exp._neg_reward_indices)))
    out[name + "_cfg"] = np.array([H, L, seed, n, every], np.int64)
    out[name + "_reward"] = rewards
    out[name + "_terminal"] = terms
    out[name + "_log"] = np.array(log, np.int64)
    print("experience", name, "events", len(log), "final top", exp._top_frame_index,
          exp.get_debug_string())
  np.savez_compressed(os.path.join(HERE, "experience_golden.npz"), **out)


# ---------------------------------------------------------------------------
# C. Trainer targets: the reference's _process_* on the real maze + Experience
# ---------------------------------------------------------------------------
class MazeShim(MazeEnvironment):
  def process(self, action, flag=0):
    image, r, t, pc = MazeEnvironment.process(self, action)
    self._last_full_state = {'success': bool(t)}
    return {'image': image}, r, t, pc


def gen_trainer(name, H, n_iter, n_step_TD, seed, net_seed):
  rs = np.random.RandomState(seed)
  net = FakeNet(net_seed)
  me = types.SimpleNamespace(
      experience=Experience(H, rs), local_t_max=20, action_size=4, gamma=0.99, gamma_pc=0.9,
      n_step_TD=n_step_TD, environment=MazeShim(), local_network=net, use_lstm=True, segnet_mode=0,
      segnet_param_dict={'segnet_mode': 0}, thread_index=1, local_t=0, episode_reward=0,
      success_rates=deque(maxlen=50), sr_size=50, random_state=rs)
  me.choose_action = lambda pi: Trainer.choose_action(me, pi)
  n_fill = 0
  while not me.experience.is_full():
    Trainer._fill_experience(me, None)
    n_fill += 1
  out = {"cfg": np.array([H, n_iter, n_step_TD, seed, net_seed, n_fill], np.int64)}
  base_len = []; base_pos = []; base_lar = []; base_a = []; base_adv = []; base_R = []
  pc_len = []; pc_pos = []; pc_lar = []; pc_a = []; pc_R = []
  vr_len = []; vr_pos = []; vr_lar = []; vr_R = []
  rp_pos = []; rp_c = []
  import io, contextlib
  for it in range(n_iter):
    sd = {'placeholders': {}, 'values': {}}
    with contextlib.redirect_stdout(io.StringIO()):
      si, _, lar, a, adv, R, _ = Trainer._process_base(me, None, 0, None, None, sd)
    base_len.append(len(si))
    for k in range(len(si)):
      x, y = agent_pos(si[k])
      assert np.array_equal(si[k], me.environment._maze_image + _agent(x, y))
      base_pos.append((x, y)); base_lar.append(lar[k]); base_a.append(a[k])
      base_adv.append(adv[k]); base_R.append(R[k])
    si, lar, a, R = Trainer._process_pc(me, None)
    pc_len.append(len(si))
    for k in range(len(si)):
      pc_pos.append(agent_pos(si[k])); pc_lar.append(lar[k]); pc_a.append(a[k]); pc_R.append(R[k])
    si, lar, R = Trainer._process_vr(me, None)
    vr_len.append(len(si))
    for k in range(len(si)):
      vr_pos.append(agent_pos(si[k])); vr_lar.append(lar[k]); vr_R.append(R[k])
    si, c = Trainer._process_rp(me)
    rp_pos.append([agent_pos(s) for s in si]); rp_c.append(c[0])
  out.update(
      base_len=np.array(base_len), base_pos=np.array(base_pos, np.uint8),
      base_lar=np.array(base_lar, np.float64), base_a=np.array(base_a, np.float64),
      base_adv=np.array(base_adv, np.float64), base_R=np.array(base_R, np.float64),
      pc_len=np.array(pc_len), pc_pos=np.array(pc_pos, np.uint8), pc_lar=np.array(pc_lar, np.float64),
      pc_a=np.array(pc_a, np.float64),
      # full maps only for the first frames (size); float64 sums + 16 float32 probe cells for all
      pc_R_head=np.array(pc_R[:PC_FULL], np.float32),
      pc_R_sum=np.array([np.sum(m, dtype=np.float64) for m in pc_R]),
      pc_R_probe=np.array([np.asarray(m, np.float64).reshape(-1)[PC_PROBE] for m in pc_R], np.float32),
      vr_len=np.array(vr_len), vr_pos=np.array(vr_pos, np.uint8), vr_lar=np.array(vr_lar, np.float64),
      vr_R=np.array(vr_R, np.float64),
      rp_pos=np.array(rp_pos, np.uint8), rp_c=np.array(rp_c, np.float64),
      final_top=np.array([me.experience._top_frame_index, me.local_t]),
      lr_anneal=np.array([Trainer._anneal_learning_rate(
          types.SimpleNamespace(initial_learning_rate=7.0710678e-4, max_global_time_step=13200000), t)
          for t in (0, 1, 6600000, 13199999, 13200000, 14000000)]))
  np.savez_compressed(os.path.join(HERE, "trainer_%s.npz" % name), **out)
  print("trainer", name, "fill", n_fill, "iters", n_iter, "base steps", sum(base_len),
        "episodes ended", int(sum(1 for l in base_len if l < n_step_TD)),
        "dtype adv", np.asarray(base_adv).dtype)


# ---------------------------------------------------------------------------
# D. the same reference functions on a GENERIC-FRAME env (the lab / gym / indoor process() shape, SURVEY 8f-4):
#    frames come from the oracle's table-hashed frame source, everything under test is the reference's
# ---------------------------------------------------------------------------
def gen_trainer_frames(name, H, n_iter, n_step_TD, seed, net_seed, table_seed):
  import zlib
  sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
  from oracle import unreal_oracle as O

  class FrameShim(O.TableFrameEnvOracle):
    def process(self, action, flag=0):
      out = O.TableFrameEnvOracle.process(self, action)
      self._last_full_state = {'success': bool(out[2])}     # trainer.py:285 reads it on terminal
      return out

  crc = lambda img: zlib.crc32(np.ascontiguousarray(img, np.float32).tobytes())   # noqa: E731
  rs = np.random.RandomState(seed)
  net = FakeNet(net_seed, 3)
  me = types.SimpleNamespace(
      experience=Experience(H, rs), local_t_max=20, action_size=3, gamma=0.99, gamma_pc=0.9,
      n_step_TD=n_step_TD, environment=FrameShim(0, O.make_frame_table(table_seed)), local_network=net, use_lstm=True,
      segnet_mode=0, segnet_param_dict={'segnet_mode': 0}, thread_index=1, local_t=0, episode_reward=0,
      success_rates=deque(maxlen=50), sr_size=50, random_state=rs)
  me.choose_action = lambda pi: Trainer.choose_action(me, pi)
  n_fill = 0
  import io, contextlib
  while not me.experience.is_full():
    with contextlib.redirect_stdout(io.StringIO()):
      Trainer._fill_experience(me, None)
    n_fill += 1
  out = {"cfg": np.array([H, n_iter, n_step_TD, seed, net_seed, n_fill, table_seed], np.int64)}
  base_len = []; base_crc = []; base_lar = []; base_a = []; base_adv = []; base_R = []
  pc_len = []; pc_crc = []; pc_lar = []; pc_a = []; pc_sum = []; pc_probe = []
  vr_len = []; vr_crc = []; vr_lar = []; vr_R = []
  rp_crc = []; rp_c = []
  for it in range(n_iter):
    sd = {'placeholders': {}, 'values': {}}
    with contextlib.redirect_stdout(io.StringIO()):
      si, _, lar, a, adv, R, _ = Trainer._process_base(me, None, 0, None, None, sd)
    base_len.append(len(si))
    for k in range(len(si)):
      base_crc.append(crc(si[k])); base_lar.append(lar[k]); base_a.append(a[k]); base_adv.append(adv[k]); base_R.append(R[k])
    si, lar, a, R = Trainer._process_pc(me, None)
    pc_len.append(len(si))
    for k in range(len(si)):
      pc_crc.append(crc(si[k])); pc_lar.append(lar[k]); pc_a.append(a[k])
      pc_sum.append(np.sum(R[k], dtype=np.float64)); pc_probe.append(np.asarray(R[k], np.float64).reshape(-1)[PC_PROBE])
    si, lar, R = Trainer._process_vr(me, None)
    vr_len.append(len(si))
    for k in range(len(si)):
      vr_crc.append(crc(si[k])); vr_lar.append(lar[k]); vr_R.append(R[k])
    si, c = Trainer._process_rp(me)
    rp_crc.append([crc(s_) for s_ in si]); rp_c.append(c[0])
  out.update(
      base_len=np.array(base_len), base_crc=np.array(base_crc, np.uint32), base_lar=np.array(base_lar, np.float64),
      base_a=np.array(base_a, np.float64), base_adv=np.array(base_adv, np.float64), base_R=np.array(base_R, np.float64),
      pc_len=np.array(pc_len), pc_crc=np.array(pc_crc, np.uint32), pc_lar=np.array(pc_lar, np.float64),
      pc_a=np.array(pc_a, np.float64), pc_R_sum=np.array(pc_sum), pc_R_probe=np.array(pc_probe),
      vr_len=np.array(vr_len), vr_crc=np.array(vr_crc, np.uint32), vr_lar=np.array(vr_lar, np.float64),
      vr_R=np.array(vr_R, np.float64), rp_crc=np.array(rp_crc, np.uint32), rp_c=np.array(rp_c, np.float64),
      final_top=np.array([me.experience._top_frame_index, me.local_t]))
  np.savez_compressed(os.path.join(HERE, "trainer_%s.npz" % name), **out)
  print("trainer", name, "fill", n_fill, "iters", n_iter, "base steps", sum(base_len),
        "episodes ended", int(sum(1 for l in base_len if l < n_step_TD)))


# ---------------------------------------------------------------------------
# E. Environment._calc_pixel_change on generic frames (the lab / gym / indoor call, environment.py:88-99):
#    float32 `uint8 / 255` frames of several sizes and channel counts
# ---------------------------------------------------------------------------
def gen_pixel_change():
  env = Environment()
  rs = np.random.RandomState(77)
  out = {}
  for i, (h, w, c) in enumerate([(84, 84, 3), (100, 120, 3), (44, 44, 1), (84, 84, 4), (36, 52, 3)]):
    a = (rs.randint(0, 256, size=(h, w, c)).astype(np.float32) / 255.0).astype(np.float32)
    b = (rs.randint(0, 256, size=(h, w, c)).astype(np.float32) / 255.0).astype(np.float32)
    pc = env._calc_pixel_change(a, b)
    out["a%d" % i] = (a * 255.0 + 0.5).astype(np.uint8); out["b%d" % i] = (b * 255.0 + 0.5).astype(np.uint8)
    out["pc%d" % i] = pc
    print("pixel change", (h, w, c), "->", pc.shape, pc.dtype)
  np.savez_compressed(os.path.join(HERE, "pixel_change_golden.npz"), **out)


# ---------------------------------------------------------------------------
# F. ExperienceFrame.concat_action_and_reward with an objective vector (experience.py:34-46; the indoor state)
# ---------------------------------------------------------------------------
def gen_lar():
  rs = np.random.RandomState(3)
  acts = rs.randint(0, 3, size=64); rews = (rs.randint(-2, 3, size=64) * 0.25).astype(np.float64)
  objs = rs.rand(64, 2).astype(np.float32)
  with_obj = np.stack([ExperienceFrame.concat_action_and_reward(int(a), 3, float(r), {'image': None, 'objective': o})
                       for a, r, o in zip(acts, rews, objs)])
  without = np.stack([ExperienceFrame.concat_action_and_reward(int(a), 3, float(r), {'image': None})
                      for a, r in zip(acts, rews)])
  np.savez_compressed(os.path.join(HERE, "lar_golden.npz"), action=acts, reward=rews, objective=objs, with_obj=with_obj,
                      without=without)
  print("lar", with_obj.shape, with_obj.dtype, without.shape)


PC_FULL = 160          # keeps each trainer_*.npz under 1 MB
PC_PROBE = np.array([0, 19, 21, 63, 105, 147, 168, 189, 210, 231, 252, 294, 336, 378, 380, 399])


def _agent(x, y):
  im = np.zeros((84, 84, 3))
  im[12 * y:12 * y + 12, 12 * x:12 * x + 12, 1] = 1.0
  return im


if __name__ == "__main__":
  gen_maze()
  gen_experience()
  gen_trainer("h2000", 2000, 300, 20, 0xA3C, 99)
  gen_trainer("h100", 100, 400, 20, 5, 17)
  gen_trainer_frames("frames_h120", 120, 200, 20, 21, 33, 6)
  gen_pixel_change()
  gen_lar()
