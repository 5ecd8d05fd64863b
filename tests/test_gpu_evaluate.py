"""GPU: the evaluator (unreal_b200/train/evaluator.py) and its fused maze kernel (unreal_maze_eval_act).

  * the kernel against the numpy restatement on the oracle maze (tests/eval_restatement.py), plus what only the device
    has: the LSTM state rows zeroed on reset and untouched for inactive envs, the operand row it writes;
  * the fused path against the generic loop, both modes, graphs on / off, both acting-head kernels;
  * the generic path against the public acting step; isolation from a Trainer sharing the model;
  * a policy with a known answer; a framed env against a hand-written loop; the CLI round trip."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import unreal_oracle as O
import eval_restatement as R

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = torch.device("cuda", 0)


def _net(seed=3, actions=4, n=1, fused_heads=False):
  from unreal_b200.environment.environment import Environment
  from unreal_b200.model.model import UnrealModel
  Environment.action_size = -1
  net = UnrealModel(actions, 0, -1, True, True, True, True, 0.05, 0.001, DEV, {'segnet_mode': 0}, (84, 84), True, 0, 0.0, 0.0,
                    num_envs=n, seed=seed)
  net.fused_act_heads = fused_heads
  return net


def _evaluator(net, **kw):
  from unreal_b200.train.evaluator import Evaluator
  return Evaluator(net, device=DEV, **kw)


# ---- 1. the kernel against the restatement -------------------------------------------------------------------------
@pytest.mark.parametrize("greedy", [False, True], ids=["sample", "greedy"])
def test_kernel_matches_restatement(greedy):
  from unreal_b200 import kernels as K
  m, a, episodes, cap, steps, kx = 7, 4, 3, 9, 40, 264
  seeds = [5, 0, 77, 2 ** 31, 12, 3, 999]
  pi = R.random_pi(np.random.RandomState(11 + greedy), steps, m, a, ties=greedy)
  want = R.restate(O.MAZE_MAP, seeds, pi, episodes, cap, greedy, kl=kx - 256)
  K.maze_set_map(None)
  state = K.MazeState(m, DEV)
  streams = K.MtStreams(seeds, DEV)
  ep = dict(score=torch.zeros(m, device=DEV), length=torch.zeros(m, dtype=torch.int32, device=DEV),
            index=torch.zeros(m, dtype=torch.int32, device=DEV), active=torch.ones(m, dtype=torch.uint8, device=DEV))
  res = dict(score=torch.zeros(m, episodes, device=DEV), length=torch.zeros(m, episodes, dtype=torch.int32, device=DEV),
             finished=torch.zeros(m, episodes, dtype=torch.uint8, device=DEV))
  gen = torch.Generator(device=DEV).manual_seed(1)
  fc_tab = torch.randn(49, 256, device=DEV, generator=gen).to(torch.bfloat16)
  c = torch.randn(m, 256, device=DEV, generator=gen)
  xh = torch.randn(m, kx + 256, device=DEV, generator=gen).to(torch.bfloat16)
  pi_d = torch.from_numpy(pi).to(DEV)
  for t in range(steps):
    h = torch.randn(m, 256, device=DEV, generator=gen) * 3       # what the cell kernel left in the state this step
    c0, h0, xh0 = c.clone(), h.clone(), xh.clone()
    K.maze_eval_act(pi_d[t].contiguous(), greedy, streams, state, ep, res, c, h, fc_tab, xh, kx, cap)
    log = want["log"][t]
    stepped = torch.from_numpy(log[:, 0] == 1).to(DEV)
    done = torch.from_numpy(log[:, 6] == 1).to(DEV)
    assert torch.equal(ep["index"].cpu(), torch.from_numpy(log[:, 7])), t
    assert torch.equal(ep["active"].cpu(), torch.from_numpy((log[:, 7] < episodes).astype(np.uint8))), t
    for e in range(m):
      if not stepped[e]:           # inactive: nothing of the env is touched
        assert torch.equal(xh[e], xh0[e]) and torch.equal(c[e], c0[e]) and torch.equal(h[e], h0[e])
        continue
      assert tuple(state.pos[e].tolist()) == (int(log[e, 4]), int(log[e, 5])), (t, e)
      cell = int(log[e, 5]) * 7 + int(log[e, 4])
      assert torch.equal(xh[e, :256], fc_tab[cell])
      assert torch.equal(xh[e, 256:kx].float().cpu(), torch.from_numpy(want["lar"][t, e]))
      if done[e]:
        assert not c[e].any() and not h[e].any() and not xh[e, kx:].float().any()
        assert not torch.signbit(c[e]).any() and not torch.signbit(h[e]).any()
      else:
        assert torch.equal(c[e], c0[e]) and torch.equal(h[e], h0[e])
        assert torch.equal(xh[e, kx:], h0[e].to(torch.bfloat16))          # torch's round-to-nearest-even cast
      assert int(state.last_action[e]) == int(np.argmax(want["lar"][t, e, :a])) or done[e]
  for k in ("score", "length", "finished"):
    assert np.array_equal(res[k].cpu().numpy(), want[k]), k
  for e, rs in enumerate(want["streams"]):
    _, key, pos, _, _ = rs.get_state()
    assert int(streams.pos[e]) == int(pos)
    assert np.array_equal(streams.mt[:, e].cpu().numpy().view(np.uint32), key)


def test_kernel_operand_row_equals_the_acting_step_operand():
  """The row the kernel writes is what UnrealModel._step_gates builds: cell_gather + lar + the cast of h."""
  from unreal_b200 import kernels as K
  net = _net(seed=4, n=16)
  m = 16
  ev = _evaluator(net, num_envs=m, max_episode_steps=5, use_graphs=False)
  assert ev.path == 'fused'
  ev._start(2)
  with torch.no_grad():
    for _ in range(13):
      pos = ev.env.state.pos.clone()
      lar = K.rollout_lar(ev.env.state.last_action, ev.env.state.last_reward, 4)
      xh_ref = torch.zeros_like(ev.xh)
      active = ev.ep["active"].bool()
      net._step_gates(net._views(net.flat), pos, lar, ev.lstm_h, xh_ref)
      assert torch.equal(ev.xh[active], xh_ref[active])
      ev._fused_step()


# ---- 2. fused against generic --------------------------------------------------------------------------------------
@pytest.mark.parametrize("fused_heads", [False, True], ids=["cell+heads", "cell_act_heads"])
@pytest.mark.parametrize("graphs", [False, True], ids=["eager", "graphs"])
@pytest.mark.parametrize("mode", ["sample", "greedy"])
def test_fused_equals_generic(mode, graphs, fused_heads):
  net = _net(seed=7, fused_heads=fused_heads)
  out, streams = {}, {}
  for fused in (True, False):
    ev = _evaluator(net, num_envs=64, mode=mode, max_episode_steps=300, use_graphs=graphs, fused=fused)
    assert ev.path == ('fused' if fused else 'generic')
    out[fused] = ev.run(2)
    streams[fused] = (ev.streams.mt.clone(), ev.streams.pos.clone())
  for k in ("score", "length", "finished"):
    assert torch.equal(out[True][k], out[False][k]), k
  assert torch.equal(streams[True][0], streams[False][0]) and torch.equal(streams[True][1], streams[False][1])
  s = out[True]["summary"]
  assert s["episodes"] == 128 and s["env_steps"] == int(out[True]["length"].sum())
  assert (out[True]["length"] >= 1).all() and (out[True]["length"] <= 300).all()
  if mode == "greedy":     # deterministic: every env plays the same episode
    assert (out[True]["length"] == out[True]["length"][0, 0]).all()
    assert int(streams[True][1].min()) == 624


def test_second_run_replays_the_captured_chunk():
  net = _net(seed=8)
  ev = _evaluator(net, num_envs=32, max_episode_steps=40)
  first = ev.run(1)
  g = ev._graph
  again = _evaluator(net, num_envs=32, max_episode_steps=40, use_graphs=False)
  again.streams.mt.copy_(ev.streams.mt); again.streams.pos.copy_(ev.streams.pos)
  second = ev.run(1)
  assert ev._graph is g
  ref = again.run(1)
  for k in ("score", "length", "finished"):
    assert torch.equal(second[k], ref[k]), k
  assert first["summary"]["episodes"] == 32


# ---- 3. generic path against the public acting step ---------------------------------------------------------------
def test_generic_path_pi_equals_run_base_policy_and_value():
  from unreal_b200 import kernels as K
  net = _net(seed=9)
  net2 = _net(seed=1, n=16)
  net2.sync_from(net)
  net2.reset_state()
  ev = _evaluator(net, num_envs=16, max_episode_steps=300, use_graphs=False, fused=False)
  got = []
  act_step = net.act_step

  def recording(*args, **kw):
    pi, v = act_step(*args, **kw)
    got.append(pi.clone())
    return pi, v
  net.act_step = recording
  try:
    ev._start(1)
    with torch.no_grad():
      for t in range(50):
        lar = K.rollout_lar(ev.env.last_action, ev.env.last_reward, 4)
        obs = ev.env.last_state['image'].clone()
        active = ev.ep["active"].clone()
        idx0 = ev.ep["index"].clone()
        ev._generic_step()
        pi2, _, _ = net2.run_base_policy_and_value(None, {'image': obs}, lar, active)
        a = active.bool()
        assert torch.equal(got[-1][a], pi2[a]), t
        net2.reset_state((ev.ep["index"] != idx0).to(torch.uint8))
  finally:
    del net.act_step
  assert len(got) == 50


# ---- 4. isolation from a Trainer sharing the model ----------------------------------------------------------------
def _trainer_trial(with_eval):
  from unreal_b200.train.rmsprop_applier import RMSPropApplier
  from unreal_b200.train.trainer import Trainer
  n = 4
  net = _net(seed=6, n=n)
  ap = RMSPropApplier(7e-4, decay=0.99, momentum=0.0, epsilon=0.1, clip_norm=40.0)
  tr = Trainer(0, net, 7e-4, None, ap, 'maze', '', True, True, True, True, 0.05, 0.001, 20, 20, 0.99, 0.9, 40, 10 ** 7,
               "cuda:0", {'segnet_mode': 0}, (84, 84), True, 0, np.random.RandomState(1), 50.0, 0.0, 0.0, num_envs=n,
               seeds=np.arange(n) + 11, obs_cells=True, use_graphs=True)
  tr.prepare()
  while not tr.experience.is_full():
    tr.process(None, 0)
  ev = _evaluator(net, num_envs=8, max_episode_steps=50) if with_eval else None
  rets, losses = [], []
  for _ in range(3):
    if ev is not None:
      ev.run(1)
    rets.append(tr.process(None, 0))
    losses.append({k: v.clone() for k, v in tr.last_losses.items()})
  if ev is not None:
    ev.run(1)
  torch.cuda.synchronize()
  out = dict(rets=rets, losses=losses, flat=net.flat.detach().clone(), c=net._lstm_c.clone(), h=net._lstm_h.clone(),
             ring={k: v.clone() for k, v in tr.experience.ring.export_state().items()},
             mt=tr.streams.mt.clone(), pos=tr.streams.pos.clone(), env_pos=tr.environment.state.pos.clone(),
             act_xh={k: v.clone() for k, v in net._act_xh.items()})
  tr.stop()
  return out


def test_evaluation_leaves_a_trainer_untouched():
  """Everything of the Trainer that is deterministic -- returned (steps, score), LSTM state, acting operand, ring, RNG
  streams, env state -- is bit-identical with and without evaluations between its updates.  Parameters and losses
  are compared against the Trainer's own run-to-run difference (float atomics in the gradient reductions make two
  identical training runs differ in the last bits): two runs without evaluation give the reference spread."""
  a, b, b2 = _trainer_trial(True), _trainer_trial(False), _trainer_trial(False)
  assert a["rets"] == b["rets"] == b2["rets"]
  for k in ("c", "h", "mt", "pos", "env_pos"):
    assert torch.equal(a[k], b[k]), k
  for k in a["ring"]:
    assert torch.equal(a["ring"][k], b["ring"][k]), k
  assert set(a["act_xh"]) == set(b["act_xh"]) and all(torch.equal(a["act_xh"][k], b["act_xh"][k]) for k in a["act_xh"])
  spread = float((b["flat"] - b2["flat"]).abs().max())
  assert float((a["flat"] - b["flat"]).abs().max()) <= max(4 * spread, 1e-7)
  for la, lb in zip(a["losses"], b["losses"]):
    assert set(la) == set(lb)
    for k in la:
      assert torch.allclose(la[k].double(), lb[k].double(), rtol=1e-5, atol=1e-6), k


# ---- 5. a policy with a known answer ------------------------------------------------------------------------------
@pytest.mark.parametrize("fused", [True, False], ids=["fused", "generic"])
@pytest.mark.parametrize("mode", ["sample", "greedy"])
def test_repeated_action_policy(mode, fused):
  """pi one-hot on UP whatever the input: from S = (0,2) two moves to (0,0), then the boundary on every step, so every
  episode is capped with score -(cap - 2)."""
  net = _net(seed=2)
  v = {k: t.cpu().numpy() for k, t in net.named_vars().items()}
  v["W_base_fc_p"] = np.zeros_like(v["W_base_fc_p"])
  v["b_base_fc_p"] = np.array([60.0, 0.0, 0.0, 0.0], np.float32)
  net.load_vars(v)
  cap = 37
  ev = _evaluator(net, num_envs=8, mode=mode, max_episode_steps=cap, fused=fused)
  out = ev.run(2)
  walls, start, goal = O.maze_layout()
  x, y, score = start[0], start[1], 0
  for _ in range(cap):
    x, y, r, term = O.maze_step(x, y, 0, walls, goal)
    score += r
    assert not term
  assert score == -(cap - 2)
  assert (out["score"] == float(score)).all() and (out["length"] == cap).all() and not out["finished"].any()
  s = out["summary"]
  assert s["success_rate"] == 0.0 and s["mean_score"] == float(score) and s["mean_length_finished"] is None
  assert int(ev.streams.pos[0]) == (624 if mode == "greedy" else 2 * 2 * cap)    # two words per sampled step


# ---- 6. a framed env against a hand-written loop ------------------------------------------------------------------
@pytest.mark.parametrize("graphs", [False, True], ids=["eager", "graphs"])
def test_framed_env_matches_hand_written_loop(graphs):
  from unreal_b200 import kernels as K
  from unreal_b200.environment.environment import Environment
  m, episodes, cap = 16, 2, 40
  args = {'producer': 'table', 'seed': 3}
  net = _net(seed=5, actions=3)
  ev = _evaluator(net, env_type='synthetic', num_envs=m, max_episode_steps=cap, use_graphs=graphs, env_args=args)
  assert ev.path == 'generic'
  out = ev.run(episodes)

  env = Environment.create_environment('synthetic', '', env_args=dict(args, num_envs=m, device=DEV))
  env.reset()                                        # Evaluator.run starts with a reset of every env
  streams = K.MtStreams(np.arange(m), DEV)
  c = torch.zeros(m, 256, device=DEV); h = torch.zeros(m, 256, device=DEV)
  active = torch.ones(m, dtype=torch.uint8, device=DEV)
  score = np.zeros(m, np.float32); length = np.zeros(m, np.int64); ep = np.zeros(m, np.int64)
  want = {k: np.zeros((m, episodes), dt) for k, dt in (("score", np.float32), ("length", np.int32), ("finished", np.uint8))}
  with torch.no_grad():
    while active.any():
      lar = K.rollout_lar(env.last_action, env.last_reward, 3)
      pi, _ = net.act_step(env.last_state, lar, c, h, active)
      action = streams.choose_action(pi, active)
      _, r, t, _ = env.process(action, active=active)
      r, t, act = r.cpu().numpy(), t.cpu().numpy(), active.cpu().numpy()
      capped = np.zeros(m, np.uint8); done = np.zeros(m, bool)
      for e in range(m):
        if not act[e]:
          continue
        score[e] += r[e]; length[e] += 1
        if t[e] or length[e] >= cap:
          want["score"][e, ep[e]] = score[e]; want["length"][e, ep[e]] = length[e]; want["finished"][e, ep[e]] = t[e]
          ep[e] += 1; score[e] = 0; length[e] = 0; done[e] = True
          capped[e] = 0 if t[e] else 1
      env.reset(torch.from_numpy(capped).to(DEV))
      d = torch.from_numpy(done).to(DEV)
      c[d] = 0.0; h[d] = 0.0
      active = torch.from_numpy((act.astype(bool) & ~(done & (ep >= episodes))).astype(np.uint8)).to(DEV)
  for k in want:
    assert np.array_equal(out[k].cpu().numpy(), want[k]), k
  assert torch.equal(ev.streams.mt, streams.mt) and torch.equal(ev.streams.pos, streams.pos)
  assert want["finished"].sum() > 0 or (want["length"] == cap).all()


# ---- 7. the CLI ---------------------------------------------------------------------------------------------------
def _cli(*args):
  r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "evaluate.py")] + list(args), cwd=ROOT,
                     capture_output=True, text=True, timeout=900)
  assert r.returncode == 0, r.stderr[-3000:]
  return json.loads(r.stdout.strip().splitlines()[-1])


def test_cli_round_trip(tmp_path):
  from unreal_b200.train import checkpoint
  from unreal_b200.train.rmsprop_applier import RMSPropApplier
  from unreal_b200.train.tf_checkpoint import save_tf_checkpoint
  from unreal_b200.train.trainer import Trainer
  net = _net(seed=12, n=4)
  ap = RMSPropApplier(7e-4, decay=0.99, momentum=0.0, epsilon=0.1, clip_norm=40.0)
  tr = Trainer(0, net, 7e-4, None, ap, 'maze', '', True, True, True, True, 0.05, 0.001, 20, 20, 0.99, 0.9, 40, 10 ** 7,
               "cuda:0", {'segnet_mode': 0}, (84, 84), True, 0, np.random.RandomState(1), 50.0, 0.0, 0.0, num_envs=4,
               seeds=np.arange(4), obs_cells=True)
  tr.prepare()
  while not tr.experience.is_full():
    tr.process(None, 0)
  tr.process(None, 0)
  path = str(tmp_path / "agent.pt")
  checkpoint.save(path, tr)
  prefix = str(tmp_path / "checkpoint-100")
  save_tf_checkpoint(net, prefix)
  ev = _evaluator(net, num_envs=8, seeds=5 + np.arange(8), mode='sample', max_episode_steps=60)
  want = ev.run(2)["summary"]
  for flag, src in (("--checkpoint", path), ("--tf-checkpoint", prefix)):
    got = _cli(flag, src, "--envs", "8", "--episodes", "2", "--mode", "sample", "--max-steps", "60", "--seed", "5")
    for k, v in want.items():
      if k != "wall_s":
        assert got[k] == v, (flag, k)
  bad = dict(torch.load(path, weights_only=True))
  bad["variables"] = dict(bad["variables"]); bad["variables"]["W_base_fc_p"] = torch.zeros(256, 3)
  torch.save(bad, str(tmp_path / "bad.pt"))
  r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "evaluate.py"), "--checkpoint", str(tmp_path / "bad.pt")],
                     cwd=ROOT, capture_output=True, text=True, timeout=900)
  assert r.returncode != 0 and "checkpoint rejected" in r.stderr
  tr.stop()
