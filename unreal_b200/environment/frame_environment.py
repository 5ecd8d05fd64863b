"""Generic-frame environment adapter (SURVEY.md 8f-4): the `process(action) -> (state, reward, terminal,
pixel_change)` contract of environment/{lab,gym,indoor}_environment.py, batched over N envs, for
frames that have no closed form.  A *producer* supplies the frames (a device generator, or host
simulators behind `HostEnvProducer`); the adapter owns everything the reference env classes do
around the simulator call:

  * the pixel change between the previous and the new frame (environment.py:93-99) -> K2,
  * `last_state / last_action / last_reward` (indoor_environment.py:117-139, lab_environment.py:120-131),
  * the packed `ExperienceFrame` record of the step for the replay ring (`frame_rec`),
  * reset of the envs whose episode ended (trainer.py:201-202, :292: `if terminal: reset()`), so that a
    rollout window never returns to Python for terminal handling.

Frames are uint8 [N,H,W,3] on the device (1 = 255, the reference's `image / 255.0` preprocessing is
applied on load by K2 and by the network's frame kernel); 21 168 B per 84x84 frame instead of the
reference's 84 672 B float32 state.  Host simulators that return float32 frames are staged as float32
and converted to uint8 on the device by the ingest kernel (HostEnvProducer).
"""
import queue
import threading
import weakref

import numpy as np
import torch

from .. import _lib
from .. import kernels as K
from . import environment


class FrameProducer(object):
  """What the adapter needs from a frame source.  All tensors live on `device`.

  reset(mask, out, objective)             write the first frame of a new episode into out[e] for every e with
                               mask[e] != 0 (mask None: all envs)
  step(action, active, out, reward, terminal, objective)
                               advance the envs with active[e] != 0 (None: all) by action[e]: new frame
                               into out[e], reward[e] f32, terminal[e] u8; rows of inactive envs must be
                               left alone in `out` and get reward 0 / terminal 0
  `objective` ([N,G] f32 or None) receives state['objective'] of the new state when objective_size > 0.
  """
  action_size = 3
  objective_size = 0
  frame_shape = (84, 84, 3)

  def reset(self, mask, out, objective=None):
    raise NotImplementedError

  def step(self, action, active, out, reward, terminal, objective=None):
    raise NotImplementedError


class TableFrameProducer(FrameProducer):
  """Deterministic frames for parity tests: every (env, step counter, action) hashes into a table of K
  seeded random uint8 frames, a reward in {-1, -.5, 0, .5, 1} and a terminal flag.  The numpy twin is
  oracle/unreal_oracle.py:TableFrameEnvOracle."""
  K_FRAMES = 32
  MOD = 1000003

  def __init__(self, num_envs, device, action_size=3, seed=0, first_env=0, frame_shape=(84, 84, 3)):
    self.num_envs = int(num_envs)
    self.device = torch.device(device)
    self.action_size = int(action_size)
    self.frame_shape = tuple(frame_shape)
    self.table = torch.from_numpy(self.make_table(seed, self.frame_shape)).to(self.device)
    self.env_id = torch.arange(first_env, first_env + self.num_envs, dtype=torch.int64, device=self.device)
    self.counter = torch.zeros(self.num_envs, dtype=torch.int64, device=self.device)

  @staticmethod
  def make_table(seed, frame_shape=(84, 84, 3)):
    return np.random.RandomState(seed).randint(0, 256, size=(TableFrameProducer.K_FRAMES,) + tuple(frame_shape)).astype(np.uint8)

  def _hash(self, a_plus_1):
    return (self.env_id * 7919 + self.counter * 104729 + a_plus_1 * 613) % self.MOD

  def export_state(self):
    return {"counter": self.counter}

  def import_state(self, st):
    self.counter.copy_(st["counter"].to(self.device))

  def reset(self, mask, out, objective=None):
    m = torch.ones(self.num_envs, dtype=torch.bool, device=self.device) if mask is None else mask.to(torch.bool)
    self.counter.add_(m.to(torch.int64))
    h = self._hash(torch.zeros_like(self.counter))
    K.rows_select(out, self.table, (h % self.K_FRAMES).contiguous(), m)

  def step(self, action, active, out, reward, terminal, objective=None):
    m = torch.ones(self.num_envs, dtype=torch.bool, device=self.device) if active is None else active.to(torch.bool)
    self.counter.add_(m.to(torch.int64))
    h = self._hash(action.to(torch.int64) + 1)
    K.rows_select(out, self.table, (h % self.K_FRAMES).contiguous(), m)
    q = h // self.K_FRAMES
    r = torch.where(h % 3 == 0, ((q % 5) - 2).to(torch.float32) * 0.5, torch.zeros((), device=self.device))
    reward.copy_(torch.where(m, r, torch.zeros_like(r)))
    terminal.copy_(((h % 29 == 0) & m).to(torch.uint8))


class RandomFrameProducer(FrameProducer):
  """Frames of the MINOS observation shape from a seeded device generator (BASELINE configs[4]; MINOS
  scenes are unavailable offline): fresh U{0..255} pixels every step, zero reward, fixed-length episodes."""

  def __init__(self, num_envs, device, action_size=3, seed=0, episode_len=200, frame_shape=(84, 84, 3),
               objective_size=0):
    self.num_envs = int(num_envs)
    self.device = torch.device(device)
    self.action_size = int(action_size)
    self.objective_size = int(objective_size)
    self.frame_shape = tuple(frame_shape)
    self.episode_len = int(episode_len)
    self.gen = torch.Generator(device=self.device).manual_seed(int(seed))
    self.t = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device)

  def export_state(self):
    return {"t": self.t, "generator": self.gen.get_state()}

  def import_state(self, st):
    self.t.copy_(st["t"].to(self.device))
    self.gen.set_state(st["generator"].cpu())

  def _draw(self, mask, out):
    fresh = torch.randint(0, 256, out.shape, dtype=torch.uint8, device=self.device, generator=self.gen)
    K.rows_select(out, fresh, None, mask)

  def reset(self, mask, out, objective=None):
    self._draw(mask, out)
    if mask is None:
      self.t.zero_()
    else:
      self.t.mul_(1 - mask.to(torch.int32))
    if objective is not None:
      objective.zero_()

  def step(self, action, active, out, reward, terminal, objective=None):
    self._draw(active, out)
    self.t.add_(1 if active is None else active.to(torch.int32))
    reward.zero_()
    done = self.t >= self.episode_len
    if active is not None:
      done = done & active.to(torch.bool)
    terminal.copy_(done.to(torch.uint8))


class _EnvThreads(object):
  """k long-lived daemon threads; thread i owns the envs [lo_i, hi_i) for its whole life, so a simulator object is only
  ever called from one thread.  `run(job)` hands every thread job(lo, hi) and returns what each returned, in order."""

  def __init__(self, n, k):
    self.slices = [(i * n // k, (i + 1) * n // k) for i in range(k)]
    self._jobs = [queue.SimpleQueue() for _ in range(k)]
    self._done = [queue.SimpleQueue() for _ in range(k)]
    self._threads = [threading.Thread(target=_env_thread, args=(self._jobs[i], self._done[i], lo, hi), daemon=True,
                                      name="unreal-env-%d" % i) for i, (lo, hi) in enumerate(self.slices)]
    for t in self._threads:
      t.start()
    self._finalizer = weakref.finalize(self, _EnvThreads._stop, self._jobs)
    self._finalizer.atexit = False      # daemon threads end with the interpreter; never join one stuck in an env

  @staticmethod
  def _stop(jobs):
    for q in jobs:
      q.put(None)

  def run(self, job):
    for q in self._jobs:
      q.put(job)
    return [d.get() for d in self._done]

  def close(self):
    self._finalizer()
    for t in self._threads:
      t.join()


def _env_thread(jobs, done, lo, hi):
  while True:
    job = jobs.get()
    if job is None:
      return
    done.put(job(lo, hi))
    job = None          # a finished job keeps no reference to its producer


class HostEnvProducer(FrameProducer):
  """N reference-style env objects on the host (anything with the Environment instance contract of
  environment.py:76-86: `process(action) -> (state, reward, terminal, pixel_change)`, `reset()`,
  `last_state['image']` as float [0,1] or uint8 [H,W,3]) feeding the device path.

  `workers=1` calls every env from the calling thread (simulators bound to a thread, such as GL contexts, keep
  working); `workers=k` starts k daemon threads, each owning a fixed contiguous slice of the envs, which step their
  envs concurrently (the reference's lab / gym envs block in a Pipe `recv()`, which releases the GIL).  An env whose
  step is terminal is reset by its thread right away (trainer.py:201-202).  The threads write frames, rewards,
  terminals and objectives into pinned staging, and one kernel (unreal_host_frames_ingest) reads it in place and does
  everything the adapter does around the simulator call.  Per step the action (and the active mask) come back to the
  host once; nothing is uploaded.  Staging holds frames as the envs produce them: uint8, or float32 for float frames
  (float64 frames are rounded to float32 on the way in), fixed by the first env's first frame (its `last_state`
  after construction).  The envs' own pixel_change is
  ignored -- the kernel recomputes it from the same two frames (K2).

  A failing env call raises UnrealError naming the env, after every thread has stopped writing; the producer then
  refuses further calls.  `close()` (BatchedFrameEnvironment.stop()) ends the threads."""

  def __init__(self, envs, device, action_size, objective_size=0, frame_shape=(84, 84, 3), workers=1):
    self.envs = list(envs)
    self.num_envs = n = len(self.envs)
    self.device = torch.device(device)
    self.action_size = int(action_size)
    self.objective_size = g = int(objective_size)
    self.frame_shape = tuple(frame_shape)
    first = getattr(self.envs[0], 'last_state', None) if n else None
    if first is None or 'image' not in first:
      raise _lib.UnrealError("HostEnvProducer: env 0 has no last_state['image'] after construction; its first frame "
                             "fixes the staging dtype")
    self.stage_dtype = torch.uint8 if np.asarray(first['image']).dtype == np.uint8 else torch.float32
    pin = lambda *shape, dtype=torch.float32: torch.zeros(*shape, dtype=dtype).pin_memory()  # noqa: E731
    self._step_frames = pin(n, *self.frame_shape, dtype=self.stage_dtype)
    self._reset_frames = pin(n, *self.frame_shape, dtype=self.stage_dtype)
    self._reward = pin(n)
    self._terminal = pin(n, dtype=torch.uint8)
    self._step_obj = pin(n, max(1, g))
    self._reset_obj = pin(n, max(1, g))
    self._action = pin(n, dtype=torch.int32)
    self._mask = pin(n, dtype=torch.uint8)
    self._np = {k: getattr(self, '_' + k).numpy() for k in ('step_frames', 'reset_frames', 'reward', 'terminal',
                                                            'step_obj', 'reset_obj', 'action', 'mask')}
    self._copied = torch.cuda.Event()       # the action / mask read-back has landed
    self._ingested = torch.cuda.Event()     # the last ingest has read the staging
    self._failed = None
    k = max(1, min(int(workers), n))
    self._threads = _EnvThreads(n, k) if k > 1 else None
    self.workers = k

  @staticmethod
  def _u8(image):
    """The host twin of the kernel's float conversion (the inverse of `image / 255.0`)."""
    a = np.asarray(image)
    if a.dtype == np.uint8:
      return a
    return np.rint(a.astype(np.float64) * 255.0).clip(0, 255).astype(np.uint8)

  def close(self):
    if self._threads is not None:
      self._threads.close()
      self._threads = None

  # ---- host side: runs on the env's own thread -------------------------------------------------------------------
  def _put(self, frames, obj, e, state):
    img = np.asarray(state['image'])
    if (img.dtype == np.uint8) != (self.stage_dtype == torch.uint8):
      raise _lib.UnrealError("env %d produced a %s frame; the staging holds %s frames (fixed by env 0's first frame)"
                             % (e, img.dtype, self.stage_dtype))
    if img.shape != self.frame_shape:
      raise _lib.UnrealError("env %d produced a frame of shape %s, not %s" % (e, img.shape, self.frame_shape))
    frames[e] = img
    if self.objective_size:
      obj[e, :self.objective_size] = np.asarray(state['objective'], dtype=np.float32)

  def _step_rows(self, lo, hi):
    s = self._np
    for e in range(lo, hi):
      if not s['mask'][e]:
        continue
      try:
        state, r, t, _ = self.envs[e].process(int(s['action'][e]))
        self._put(s['step_frames'], s['step_obj'], e, state if isinstance(state, dict) else {'image': state})
        s['reward'][e] = r
        s['terminal'][e] = 1 if t else 0
        if t:
          self.envs[e].reset()
          self._put(s['reset_frames'], s['reset_obj'], e, self.envs[e].last_state)
      except BaseException as ex:   # noqa: B902 -- handed to the calling thread
        return e, ex
    return None

  def _reset_rows(self, lo, hi):
    s = self._np
    for e in range(lo, hi):
      if not s['mask'][e]:
        continue
      try:
        self.envs[e].reset()
        self._put(s['reset_frames'], s['reset_obj'], e, self.envs[e].last_state)
      except BaseException as ex:   # noqa: B902
        return e, ex
    return None

  # ---- calling thread ---------------------------------------------------------------------------------------------
  def _run(self, job, action, mask):
    if self._failed is not None:
      raise _lib.UnrealError("HostEnvProducer: env %d failed earlier; the producer takes no further calls" % self._failed)
    self._ingested.synchronize()           # the previous ingest has finished reading the staging
    if action is not None:
      self._action.copy_(action, non_blocking=True)
    if mask is not None:
      self._mask.copy_(mask, non_blocking=True)
    else:
      self._np['mask'].fill(1)
    if action is not None or mask is not None:
      self._copied.record()
      self._copied.synchronize()
    out = [job(0, self.num_envs)] if self._threads is None else self._threads.run(job)
    errors = [x for x in out if x is not None]
    if errors:
      e, ex = min(errors, key=lambda x: x[0])
      self._failed = e
      raise _lib.UnrealError("HostEnvProducer: env %d raised %s: %s" % (e, type(ex).__name__, ex)) from ex

  @staticmethod
  def _u8_mask(mask):
    return mask if mask is None or mask.dtype == torch.uint8 else mask.to(torch.uint8)

  def fused_reset(self, mask, out, objective=None, last_action=None, last_reward=None):
    """reset() of the envs with mask[e] != 0 (None: all): first frame into out[e], objective, last_action /
    last_reward zeroed (both nullable)."""
    mask = self._u8_mask(mask)
    self._run(self._reset_rows, None, mask)
    K.host_frames_ingest(self._reset_frames, out, reset_objective=self._reset_obj, active=mask,
                         last_action=last_action, last_reward=last_reward,
                         objective=objective if self.objective_size else None)
    self._ingested.record()

  def reset(self, mask, out, objective=None):
    self.fused_reset(mask, out, objective)

  def fused_step(self, action, active, prev, out, copy_inactive, pc, reward, terminal, rec, last_action, last_reward,
                 objective=None):
    """One step of the envs with active[e] != 0 (None: all) and everything BatchedFrameEnvironment.process does
    around it, in one launch (unreal_host_frames_ingest)."""
    active = self._u8_mask(active)
    self._run(self._step_rows, action, active)
    K.host_frames_ingest(self._reset_frames, out, step_frames=self._step_frames, step_reward=self._reward,
                         step_terminal=self._terminal, step_objective=self._step_obj, reset_objective=self._reset_obj,
                         action=action, active=active, prev=prev, copy_inactive=copy_inactive, pc=pc, rec=rec,
                         reward=reward, terminal=terminal, last_action=last_action, last_reward=last_reward,
                         objective=objective if self.objective_size else None)
    self._ingested.record()


class BatchedFrameEnvironment(environment.Environment):
  """N generic-frame envs in lock step behind the Environment instance contract, device resident."""

  def __init__(self, producer, device='cuda:0'):
    environment.Environment.__init__(self)
    _lib.require_device()
    self.producer = producer
    self.num_envs = n = int(producer.num_envs)
    self.device = d = torch.device(device)
    self.action_size = int(producer.action_size)
    self.objective_size = g = int(producer.objective_size)
    self.frame_shape = tuple(producer.frame_shape)
    h, w = self.frame_shape[:2]
    with torch.cuda.device(d):
      self._obs = torch.zeros(n, *self.frame_shape, dtype=torch.uint8, device=d)     # the current frame
      self._next = torch.zeros_like(self._obs)
      self._pc = torch.zeros(n, (h - 4) // 4, (w - 4) // 4, dtype=torch.float32, device=d)
      self._reward = torch.zeros(n, dtype=torch.float32, device=d)
      self._terminal = torch.zeros(n, dtype=torch.uint8, device=d)
      self.last_action = torch.zeros(n, dtype=torch.int32, device=d)
      self.last_reward = torch.zeros(n, dtype=torch.float32, device=d)
      self.frame_rec = torch.zeros(n, dtype=torch.int64, device=d)
      self.objective = torch.zeros(n, g, dtype=torch.float32, device=d) if g else None
      self._cur = self._obs
      self.reset()

  def stop(self):
    """Ends the producer's worker threads, if it has any."""
    if hasattr(self.producer, 'close'):
      self.producer.close()

  def _state(self, frame):
    s = {'image': frame}
    if self.objective is not None:
      s['objective'] = self.objective
    return s

  def reset(self, mask=None):
    """reset() of the reference env classes for every env (or those with mask != 0)."""
    with torch.cuda.device(self.device):
      if hasattr(self.producer, 'fused_reset'):
        self.producer.fused_reset(mask, self._cur, self.objective, self.last_action, self.last_reward)
        self.last_state = self._state(self._cur)
        return
      self.producer.reset(mask, self._cur, self.objective)
      if mask is None:
        self.last_action.zero_(); self.last_reward.zero_()
      else:
        keep = mask == 0
        self.last_action.mul_(keep.to(torch.int32)); self.last_reward.mul_(keep.to(torch.float32))
    self.last_state = self._state(self._cur)

  def export_state(self):
    """Everything the next step depends on (checkpoints): the current frames are state, not a function of it."""
    if not hasattr(self.producer, "export_state"):
      raise _lib.UnrealError("%s cannot be checkpointed (host simulators keep their own state)" % type(self.producer).__name__)
    d = {"frame": self._cur, "last_action": self.last_action, "last_reward": self.last_reward}
    if self.objective is not None:
      d["objective"] = self.objective
    d.update({"producer." + k: v for k, v in self.producer.export_state().items()})
    return d

  def import_state(self, st):
    self.set_current(st["frame"].to(self.device))
    self.last_action.copy_(st["last_action"].to(self.device)); self.last_reward.copy_(st["last_reward"].to(self.device))
    if self.objective is not None:
      self.objective.copy_(st["objective"].to(self.device))
    self.producer.import_state({k[len("producer."):]: v for k, v in st.items() if k.startswith("producer.")})

  def set_current(self, frame):
    """Adopt `frame` [N,H,W,3] as every env's current frame (copied into the env's own buffer)."""
    self._obs.copy_(frame)
    self._cur = self._obs
    self.last_state = self._state(self._cur)

  def process(self, action, active=None, out_obs=None, out_pc=None, out_reward=None, out_terminal=None, flag=1):
    """One env step for all (active) envs.  Returned tensors are owned by the env and overwritten by
    the next call unless out_* buffers are supplied.  After the call `last_state` is the new frame --
    for envs whose episode just ended, the first frame of their next episode."""
    prev = self._cur
    if out_obs is prev:
      raise _lib.UnrealError("out_obs must not be the buffer holding the current frame")
    if out_obs is None:
      out_obs = self._next if prev is self._obs else self._obs
    pc = self._pc if out_pc is None else out_pc
    reward = self._reward if out_reward is None else out_reward
    terminal = self._terminal if out_terminal is None else out_terminal
    own = out_obs is self._obs or out_obs is self._next
    with torch.cuda.device(self.device):
      if hasattr(self.producer, 'fused_step'):
        self.producer.fused_step(action, active, prev, out_obs, own, pc, reward, terminal, self.frame_rec,
                                 self.last_action, self.last_reward, self.objective)
        self._cur = out_obs
        self.last_state = self._state(out_obs)
        return self.last_state, reward, terminal, pc
      if own:
        out_obs.copy_(prev)                    # inactive envs keep their frame (caller-supplied buffers: untouched rows)
      self.producer.step(action, active, out_obs, reward, terminal, self.objective)
      K.pixel_change(out_obs, prev, out=pc)    # environment.py:93-99
      K.frame_pack(action, reward, terminal, self.last_action, self.last_reward, active, out=self.frame_rec)
      term = terminal if active is None else (terminal & active)
      self.producer.reset(term, out_obs, self.objective)
      act_m = torch.ones_like(term, dtype=torch.bool) if active is None else active.to(torch.bool)
      ended = term.to(torch.bool)
      zero_a = torch.zeros_like(self.last_action)
      zero_r = torch.zeros_like(self.last_reward)
      self.last_action.copy_(torch.where(act_m, torch.where(ended, zero_a, action), self.last_action))
      self.last_reward.copy_(torch.where(act_m, torch.where(ended, zero_r, reward), self.last_reward))
    self._cur = out_obs
    state = self._state(out_obs)
    self.last_state = state
    return state, reward, terminal, pc
