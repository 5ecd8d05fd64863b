"""Evaluator: whole episodes of a frozen policy, batched over M envs -- what the reference's evaluate.py does for MINOS,
for the env types of this package.

    ev = Evaluator(network, env_type='maze', num_envs=M, mode='sample')       # or mode='greedy'
    res = ev.run(episodes_per_env=E)
    res['score'] f32 [M,E], res['length'] i32 [M,E], res['finished'] u8 [M,E]  (device tensors), res['summary'] (host dict)

Each env plays E episodes in order under the weights the network holds when `run` starts (nothing updates them during
the run).  The rules, per env:

  * Episode start -- as the reference after a terminal (trainer.py:201-202, :293): env reset, LSTM state (c, h) zeroed,
    last action 0, last reward 0, so the first LSTM input row ends in one-hot(0) ++ [0]
    (ExperienceFrame.concat_action_and_reward).  `run` starts every env this way.
  * Action -- 'sample': RandomState.choice(A, p=pi) (trainer.py:147-148) on the evaluator's OWN per-env MT19937 stream,
    seeded with `seeds` (default arange(M)) when the evaluator is built and continued by later runs; bit-exact with
    numpy like the Trainer's draws.  'greedy': argmax of pi, the lowest index on ties (numpy / torch argmax), no draw.
    A greedy maze episode is deterministic, so all M envs play the same episode: one env is enough.
  * Step cap -- an episode that reaches `max_episode_steps` steps without a terminal ends there with finished = 0, its
    score so far and length = cap, and the env is reset as after a terminal (the maze has no time limit of its own).
    An episode whose terminal falls on the cap step is finished (finished = 1).
  * finished -- the episode ended by itself: for the maze, the goal was reached.
  * End of run -- an env that has played E episodes is inactive: no step, no draw, its LSTM rows are not touched.
    `run` ends when every env is inactive.
  * Isolation -- the evaluator owns its env, LSTM state, GEMM operand, RNG streams and result buffers.  It reads the
    network's parameters and shadows and writes nothing a Trainer sharing the network reads (the model's own LSTM
    state and acting operand, its parameter buffers, the Trainer's streams, env and ring are untouched).  A maze
    evaluator sets the maze map like any maze env (env_args={'map_data': ...}); keep it the map the Trainer uses.

Two paths, chosen from what the code can observe (`path`):

  * 'fused' -- env_type 'maze' and a model whose maze cell tables are on (`UnrealModel._use_tables` for cell
    observations: the defaults).  A step is the acting GEMM on the evaluator's bf16 [x, h] operand, the model's
    cell + heads kernel(s) (whatever `run_base_policy_and_value` uses, so pi is bit-identical to the public acting step)
    and unreal_maze_eval_act, which does everything after pi and writes the next step's operand rows itself.
  * 'generic' -- every other case (framed env types such as 'synthetic' and registered producers, or a maze model
    without cell tables): the public pieces -- `UnrealModel.act_step` on the evaluator's state, `choose_action` on its
    streams or argmax, `env.process(action, active=...)`, torch ops for the accounting and resets.  Both paths give
    identical scores, lengths, finished flags and RNG streams (tests/test_gpu_evaluate.py).

Steps run in chunks of CHUNK; with `use_graphs` the first chunk runs eagerly and is then captured into one CUDA graph
that later chunks (and later runs with the same E) replay.  The host reads back one count of running envs per chunk.
"""
import time

import numpy as np
import torch

from .. import _lib
from .. import kernels as K
from ..environment.environment import Environment


class Evaluator(object):
  CHUNK = 32      # steps per captured chunk (even: the framed env's two frame buffers are back in place after a chunk)

  def __init__(self, network, env_type='maze', env_name='', num_envs=1, seeds=None, mode='sample', max_episode_steps=2000,
               device='cuda:0', use_graphs=True, env_args=None, fused=None):
    """fused: None picks the path as described above; False forces the generic loop; True requires the fused path."""
    _lib.require_device()
    if mode not in ('sample', 'greedy'):
      raise _lib.UnrealError("mode must be 'sample' or 'greedy', got %r" % (mode,))
    if int(max_episode_steps) < 1 or int(num_envs) < 1:
      raise _lib.UnrealError("num_envs and max_episode_steps must be >= 1")
    self.net = network
    self.env_type = env_type
    self.mode = mode
    self.greedy = mode == 'greedy'
    self.num_envs = m = int(num_envs)
    self.max_episode_steps = int(max_episode_steps)
    self.device = d = torch.device(device if str(device).startswith("cuda") else "cuda:0")
    self.use_graphs = bool(use_graphs)
    self.action_size = a = int(network._action_size)
    self.objective_size = int(network._objective_size)
    maze = env_type == 'maze'
    cells = maze and network.fused_conv and network.fused_encoder
    args = {'num_envs': m, 'device': d, 'auto_reset': True}
    if maze:
      args['obs_dtype'] = torch.int32 if cells else torch.float32
    args.update(env_args or {})
    with torch.cuda.device(d):
      self.env = Environment.create_environment(env_type, env_name, env_args=args)
      env_a = self.env.get_action_size() if maze else int(self.env.action_size)
      if env_a != a:
        raise _lib.UnrealError("the network has %d actions, env_type %r has %d" % (a, env_type, env_a))
      if int(getattr(self.env, 'objective_size', 0)) != self.objective_size:
        raise _lib.UnrealError("the network's objective size %d differs from the env's" % self.objective_size)
      can_fuse = maze and cells and network._use_tables(self.env.last_state['image']) and self.objective_size == 0
      if fused and not can_fuse:
        raise _lib.UnrealError("the fused evaluation step needs env_type 'maze' and a model with maze cell tables")
      self.path = 'fused' if (can_fuse and fused is not False) else 'generic'
      self.streams = K.MtStreams(np.arange(m) if seeds is None else np.asarray(seeds), d)
      if self.streams.n != m:
        raise _lib.UnrealError("seeds must hold one seed per env (%d)" % m)
      self.lstm_c = torch.zeros(m, 256, dtype=torch.float32, device=d)
      self.lstm_h = torch.zeros(m, 256, dtype=torch.float32, device=d)
      self.xh = torch.zeros(m, network.kx + 256, dtype=torch.bfloat16, device=d)
      self._gates = torch.empty(m, 1024, dtype=network._gates_dtype(), device=d)
      self.ep = dict(score=torch.zeros(m, dtype=torch.float32, device=d), length=torch.zeros(m, dtype=torch.int32, device=d),
                     index=torch.zeros(m, dtype=torch.int32, device=d), active=torch.zeros(m, dtype=torch.uint8, device=d))
      self._action = torch.zeros(m, dtype=torch.int32, device=d)
      self._lar = torch.zeros(m, a + 1 + self.objective_size, dtype=torch.float32, device=d)
      self._running = torch.zeros(1, dtype=torch.int64, device=d)
    self.res = None
    self._episodes = None
    self._graph = None
    self.steps = 0            # steps (chunks * CHUNK) of the last run, counting the idle tail of the last chunk

  # -- one step ---------------------------------------------------------------------------------------------------
  def _fused_step(self):
    net = self.net
    p32 = net._views(net.flat)
    gates = net._xh_gates(p32, self.xh, out=self._gates)
    pi, _ = net._act_cell_heads(p32, gates, self.lstm_c, self.lstm_h, self.ep["active"])
    K.maze_eval_act(pi, self.greedy, None if self.greedy else self.streams, self.env.state, self.ep, self.res,
                    self.lstm_c, self.lstm_h, net._fc_tab_act, self.xh, net.kx, self.max_episode_steps)

  def _generic_step(self):
    env, net, ep, res = self.env, self.net, self.ep, self.res
    active = ep["active"]
    lar = K.rollout_lar(env.last_action, env.last_reward, self.action_size, getattr(env, 'objective', None), out=self._lar)
    pi, _ = net.act_step(env.last_state, lar, self.lstm_c, self.lstm_h, active, xh=self.xh)
    if self.greedy:
      self._action.copy_(torch.argmax(pi, dim=1))
    else:
      self.streams.choose_action(pi, active, out=self._action)
    kw = {'out_pc': False} if self.env_type == 'maze' else {}
    _, reward, terminal, _ = env.process(self._action, active=active, **kw)
    act = active.to(torch.bool)
    ep["score"].add_(reward)                       # inactive envs get reward 0
    ep["length"].add_(active.to(torch.int32))
    term = terminal.to(torch.bool) & act
    capped = act & ~term & (ep["length"] >= self.max_episode_steps)
    done = term | capped
    idx = self._row_base + ep["index"].clamp(max=self._episodes - 1).to(torch.int64)
    for key, val in (("score", ep["score"]), ("length", ep["length"]), ("finished", term.to(torch.uint8))):
      flat = res[key].view(-1)
      flat.scatter_(0, idx, torch.where(done, val, flat.gather(0, idx)))
    ep["index"].add_(done.to(torch.int32))
    env.reset(capped.to(torch.uint8))              # terminals were reset by the env itself (auto_reset)
    self.lstm_c.masked_fill_(done.unsqueeze(1), 0.0)
    self.lstm_h.masked_fill_(done.unsqueeze(1), 0.0)
    ep["score"].masked_fill_(done, 0.0)
    ep["length"].masked_fill_(done, 0)
    active.copy_((act & ~(done & (ep["index"] >= self._episodes))).to(torch.uint8))

  def _chunk(self):
    step = self._fused_step if self.path == 'fused' else self._generic_step
    for _ in range(self.CHUNK):
      step()
    self._running.copy_(self.ep["active"].sum())

  # -- a run --------------------------------------------------------------------------------------------------------
  def _start(self, episodes):
    m, d, net = self.num_envs, self.device, self.net
    if self._episodes != episodes:
      self.res = dict(score=torch.zeros(m, episodes, dtype=torch.float32, device=d),
                      length=torch.zeros(m, episodes, dtype=torch.int32, device=d),
                      finished=torch.zeros(m, episodes, dtype=torch.uint8, device=d))
      self._row_base = torch.arange(m, dtype=torch.int64, device=d) * episodes
      self._episodes = episodes
      self._graph = None                          # the captured chunk holds the result buffers of this E
    for t in self.res.values():
      t.zero_()
    self.env.reset()
    self.lstm_c.zero_(); self.lstm_h.zero_()
    self.ep["score"].zero_(); self.ep["length"].zero_(); self.ep["index"].zero_(); self.ep["active"].fill_(1)
    self.xh.zero_()
    if self.path == 'fused':
      # the first step's operand rows, as unreal_maze_eval_act writes them after a reset: the start cell's fc1 row,
      # one-hot(0) ++ [0], h = 0
      K.cell_gather(net._fc_tab_act, self.env.state.pos, out=self.xh[:, :256])
      self.xh[:, 256].fill_(1.0)

  def run(self, episodes_per_env=1):
    """Play `episodes_per_env` episodes in every env -> dict(score f32 [M,E], length i32 [M,E], finished u8 [M,E] (device
    tensors), summary (host dict: episodes, success_rate, mean_score, mean / median length of finished episodes,
    env_steps, wall_s, ...))."""
    e = int(episodes_per_env)
    if e < 1:
      raise _lib.UnrealError("episodes_per_env must be >= 1")
    with torch.cuda.device(self.device), torch.no_grad():
      self._start(e)
      torch.cuda.synchronize(self.device)
      t0 = time.perf_counter()
      chunks = 0
      while True:
        if self._graph is not None:
          self._graph.replay()
        else:
          self._chunk()
          if self.use_graphs:
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            with _lib.graph_capture(g):           # recorded, not executed
              self._chunk()
            self._graph = g
        chunks += 1
        if int(self._running.item()) == 0:       # the chunk's only host read-back
          break
      torch.cuda.synchronize(self.device)
      wall = time.perf_counter() - t0
      self.steps = chunks * self.CHUNK
      out = {k: v.clone() for k, v in self.res.items()}
    out["summary"] = self._summary(out, wall)
    return out

  def _summary(self, out, wall):
    score = out["score"].cpu().numpy().astype(np.float64)
    length = out["length"].cpu().numpy()
    fin = out["finished"].cpu().numpy().astype(bool)
    done_len = length[fin]
    return dict(env_type=self.env_type, mode=self.mode, path=self.path, envs=self.num_envs,
                episodes_per_env=int(score.shape[1]), episodes=int(score.size), success_rate=float(fin.mean()),
                mean_score=float(score.mean()),
                mean_length_finished=float(done_len.mean()) if done_len.size else None,
                median_length_finished=float(np.median(done_len)) if done_len.size else None,
                max_episode_steps=self.max_episode_steps, env_steps=int(length.astype(np.int64).sum()), wall_s=wall)
