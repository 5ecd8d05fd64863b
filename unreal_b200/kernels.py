"""Thin tensor-level wrappers over the C ABI (one function per entry point family).

All tensors are CUDA tensors owned by the caller; the wrappers allocate outputs when they
are not passed in, enqueue on torch's current stream and never synchronise.
"""
import ctypes

import torch

from . import _lib
from ._lib import call, ptr, stream_ptr

FRAME = 84
PC = 20
MT_WORDS = 624


# ---------------------------------------------------------------------------- maze
def maze_set_map(map49=None):
  call("unreal_maze_set_map", None if map49 is None else map49.encode())


def maze_layout():
  v = [ctypes.c_int() for _ in range(4)]
  walls = (ctypes.c_uint8 * 49)()
  call("unreal_maze_get_layout", *[ctypes.byref(x) for x in v], walls)
  return (v[0].value, v[1].value), (v[2].value, v[3].value), bytes(walls)


class MazeState(object):
  """SoA device state of N mazes: what MazeEnvironment keeps in self.x/self.y/last_action/
  last_reward (maze_environment.py:50-55, :125-127)."""

  def __init__(self, n, device):
    self.n = n
    self.device = torch.device(device)
    self.pos = torch.zeros(n, 2, dtype=torch.int32, device=device)
    self.last_action = torch.zeros(n, dtype=torch.int32, device=device)
    self.last_reward = torch.zeros(n, dtype=torch.float32, device=device)
    maze_reset(self)


def maze_reset(state, mask=None):
  call("unreal_maze_reset", ptr(state.pos, torch.int32), ptr(state.last_action, torch.int32),
       ptr(state.last_reward, torch.float32), ptr(mask, torch.uint8), state.n, stream_ptr())


def maze_step(state, action, obs=None, pc=None, reward=None, terminal=None, frame_rec=None, active=None,
              auto_reset=False):
  """One process() for every env.  Returns (reward, terminal); obs/pc/frame_rec are filled
  when given (pass None to skip that output)."""
  n = state.n
  dev = state.device
  if reward is None:
    reward = torch.empty(n, dtype=torch.float32, device=dev)
  if terminal is None:
    terminal = torch.empty(n, dtype=torch.uint8, device=dev)
  cell_obs = obs if (obs is not None and obs.dtype == torch.int32) else None
  if cell_obs is not None:      # "cell observation": the frame stays implicit (render-fused conv1), obs receives the cells
    if cell_obs.numel() != n * 2:
      raise _lib.UnrealError("an int32 (cell) observation buffer must hold [N,2]")
    obs = None
  if obs is not None and obs.numel() != n * FRAME * FRAME * 3:
    raise _lib.UnrealError("obs must hold [N,84,84,3]")
  if pc is not None and (pc.numel() != n * PC * PC or pc.dtype != torch.float32):
    raise _lib.UnrealError("pc must be float32 [N,20,20]")
  call("unreal_maze_step", ptr(state.pos, torch.int32), ptr(action, torch.int32, "action"),
       ptr(active, torch.uint8, "active"), ptr(reward, torch.float32), ptr(terminal, torch.uint8),
       ptr(state.last_action, torch.int32), ptr(state.last_reward, torch.float32),
       ptr(obs), _lib.dtype_tag(obs) if obs is not None else _lib.F32, ptr(pc),
       ptr(frame_rec, torch.int64, "frame_rec"), n, 1 if auto_reset else 0, stream_ptr())
  if cell_obs is not None:
    if active is None:
      cell_obs.copy_(state.pos.view_as(cell_obs))
    else:                        # like the render kernels: rows of inactive envs are left alone
      co = cell_obs.view(n, 2)
      torch.where(active.view(n, 1).bool(), state.pos.view(n, 2), co, out=co)
  return reward, terminal


def maze_window(state, actions, obs=None, pc=None, reward=None, terminal=None, frame_rec=None, auto_reset=False):
  """T process() calls of every env in ONE launch (the T actions are known up front): actions [T,N] i32; obs
  [T,N,84,84,3] f32 / u8, pc [T,N,20,20], reward / terminal / frame_rec [T,N] are filled when given.  Equal to T
  maze_step() calls; `state` ends T steps later."""
  t, n = actions.shape
  dev = state.device
  if n != state.n:
    raise _lib.UnrealError("actions must be [T, %d]" % state.n)
  if reward is None:
    reward = torch.empty(t, n, dtype=torch.float32, device=dev)
  if terminal is None:
    terminal = torch.empty(t, n, dtype=torch.uint8, device=dev)
  if obs is not None and (obs.numel() != t * n * FRAME * FRAME * 3 or obs.dtype not in (torch.float32, torch.uint8)):
    raise _lib.UnrealError("obs must hold [T,N,84,84,3] float32 or uint8")
  if pc is not None and (pc.numel() != t * n * PC * PC or pc.dtype != torch.float32):
    raise _lib.UnrealError("pc must be float32 [T,N,20,20]")
  call("unreal_maze_window", ptr(state.pos, torch.int32), ptr(actions, torch.int32, "actions"), ptr(reward, torch.float32),
       ptr(terminal, torch.uint8), ptr(state.last_action, torch.int32), ptr(state.last_reward, torch.float32), ptr(obs),
       _lib.dtype_tag(obs) if obs is not None else _lib.F32, ptr(pc), ptr(frame_rec, torch.int64, "frame_rec"), n, t,
       1 if auto_reset else 0, stream_ptr())
  return reward, terminal


def obs_shape(dtype):
  """Per-frame shape of a maze observation buffer: [84,84,3] for f32 / u8, the space-to-depth planes
  [6,441,8] for bf16 (the layout conv1 consumes directly), and [2] for int32 -- the agent CELL itself: a maze
  frame is a pure function of it, and the render-fused conv1 kernels (unreal_conv1_fwd_maze /
  unreal_conv1_wgrad_maze) build their input tiles from the cell, so no frame exists in HBM at all."""
  if dtype == torch.int32:
    return (2,)
  return (6, 441, 8) if dtype == torch.bfloat16 else (FRAME, FRAME, 3)


def maze_render(pos, out=None, dtype=torch.float32):
  m = pos.shape[0]
  if (out is not None and out.dtype == torch.int32) or (out is None and dtype == torch.int32):
    if out is None:              # cell observation: the "render" of a cell is the cell
      return pos.reshape(m, 2).clone()
    out.copy_(pos.view_as(out))
    return out
  if out is None:
    out = torch.empty(m, *obs_shape(dtype), dtype=dtype, device=pos.device)
  call("unreal_maze_render", ptr(pos, torch.int32, "pos"), ptr(out), _lib.dtype_tag(out), m, stream_ptr())
  return out


def maze_pixel_change(pos0, pos1, out=None):
  m = pos0.shape[0]
  if out is None:
    out = torch.empty(m, PC, PC, dtype=torch.float32, device=pos0.device)
  call("unreal_maze_pixel_change", ptr(pos0, torch.int32), ptr(pos1, torch.int32), ptr(out, torch.float32), m,
       stream_ptr())
  return out


def maze_pc_targets(pos0, pos1, length, boot, gamma_pc, out=None):
  """pos0, pos1 int32 [T,N,2] (time-major cells of the replayed frames and their successors), length int32 [N] or None,
  boot f32 [N,20,20] -> pixel-control targets f32 [T,N,20,20] = maze_pixel_change + pc_targets in one pass."""
  t, n = pos0.shape[0], pos0.shape[1]
  if out is None:
    out = torch.empty(t, n, PC, PC, dtype=torch.float32, device=pos0.device)
  call("unreal_maze_pc_targets", ptr(pos0, torch.int32), ptr(pos1, torch.int32), ptr(length, torch.int32),
       ptr(boot, torch.float32), float(gamma_pc), ptr(out, torch.float32), t, n, stream_ptr())
  return out


def maze_rollout_targets(rec, values, boot_value, boot_q, gamma, gamma_pc, R=None, adv=None, pc_tgt=None):
  """rec int64 [T,N] (the frame records of a maze pass), values f32 [T,N], boot_value f32 [N], boot_q f32 [N,20,20]
  -> (R, adv [T,N], pc_tgt [T,N,20,20]) = nstep_returns + pc_targets of the pass, without its pixel-change maps."""
  t, n = rec.shape
  if R is None:
    R = torch.empty(t, n, dtype=torch.float32, device=rec.device)
  if adv is None:
    adv = torch.empty(t, n, dtype=torch.float32, device=rec.device)
  if pc_tgt is None:
    pc_tgt = torch.empty(t, n, PC, PC, dtype=torch.float32, device=rec.device)
  call("unreal_maze_rollout_targets", ptr(rec, torch.int64, "rec"), ptr(values, torch.float32, "values"),
       ptr(boot_value, torch.float32, "boot_value"), ptr(boot_q, torch.float32, "boot_q"), float(gamma), float(gamma_pc),
       ptr(R, torch.float32, "R"), ptr(adv, torch.float32, "adv"), ptr(pc_tgt, torch.float32, "pc_tgt"), t, n,
       stream_ptr())
  return R, adv, pc_tgt


# ---------------------------------------------------------------------------- pixel change (generic)
def pixel_change(cur, prev, out=None):
  """cur, prev [M,H,W,C] float32 or uint8 -> [M,(H-4)//4,(W-4)//4] float32."""
  m, h, w, c = cur.shape
  if out is None:
    out = torch.empty(m, (h - 4) // 4, (w - 4) // 4, dtype=torch.float32, device=cur.device)
  if prev.shape != cur.shape or prev.dtype != cur.dtype:
    raise _lib.UnrealError("cur and prev must have the same shape and dtype")
  call("unreal_pixel_change", ptr(cur), ptr(prev), _lib.dtype_tag(cur), ptr(out, torch.float32), m, h, w, c,
       stream_ptr())
  return out


def pixel_change_stream(frames, out=None):
  """frames [S,L+1,H,W,C] -> [S,L,ph,pw]; each frame is read once."""
  s, l1, h, w, c = frames.shape
  if out is None:
    out = torch.empty(s, l1 - 1, (h - 4) // 4, (w - 4) // 4, dtype=torch.float32, device=frames.device)
  call("unreal_pixel_change_stream", ptr(frames), _lib.dtype_tag(frames), ptr(out, torch.float32), s, l1 - 1, h, w,
       c, stream_ptr())
  return out


def selfcheck_arith():
  """-> (mismatches of the two-instruction s/3 over every float in [2^-100, 2^100], mismatches of v/255 over all bytes)."""
  out = torch.zeros(2, dtype=torch.int64, device="cuda")
  call("unreal_selfcheck_arith", ptr(out), stream_ptr())
  return tuple(int(x) for x in out.tolist())


def subsample(a, width, out=None):
  """a [M,H,W] f32 -> [M,H/width,W/width]: Environment._subsample (environment.py:88-91)."""
  m, h, w = a.shape
  if out is None:
    out = torch.empty(m, h // width, w // width, dtype=torch.float32, device=a.device)
  call("unreal_subsample", ptr(a, torch.float32, "a"), ptr(out, torch.float32, "out"), m, h, w, int(width), stream_ptr())
  return out


# ---------------------------------------------------------------------------- targets
def nstep_returns(r, v, term, boot, gamma, out_R=None, out_adv=None):
  t, n = r.shape
  if out_R is None:
    out_R = torch.empty_like(r)
  if v is not None and out_adv is None:
    out_adv = torch.empty_like(r)
  call("unreal_nstep_returns", ptr(r, torch.float32), ptr(v, torch.float32), ptr(term, torch.uint8),
       ptr(boot, torch.float32), float(gamma), ptr(out_R, torch.float32), ptr(out_adv, torch.float32), t, n,
       stream_ptr())
  return out_R, out_adv


def sequence_returns(r, length, boot, gamma, out=None):
  n, l = r.shape
  if out is None:
    out = torch.empty_like(r)
  call("unreal_sequence_returns", ptr(r, torch.float32), ptr(length, torch.int32), ptr(boot, torch.float32),
       float(gamma), ptr(out, torch.float32), n, l, stream_ptr())
  return out


def pc_targets(pc, term, length, boot, gamma_pc, out=None):
  t, n = pc.shape[0], pc.shape[1]
  if out is None:
    out = torch.empty_like(pc)
  call("unreal_pc_targets", ptr(pc, torch.float32), ptr(term, torch.uint8), ptr(length, torch.int32),
       ptr(boot, torch.float32), float(gamma_pc), ptr(out, torch.float32), t, n, stream_ptr())
  return out


# ---------------------------------------------------------------------------- RNG
class MtStreams(object):
  """One numpy-legacy RandomState stream per env, resident on the device."""

  def __init__(self, seeds, device):
    seeds = torch.as_tensor(seeds, dtype=torch.int64).to(device)
    self.n = seeds.numel()
    self.device = torch.device(device)
    self.mt = torch.empty(MT_WORDS, self.n, dtype=torch.int32, device=device)
    self.pos = torch.empty(self.n, dtype=torch.int32, device=device)
    s32 = (seeds & 0xFFFFFFFF).to(torch.int64)
    s32 = torch.where(s32 >= 2 ** 31, s32 - 2 ** 32, s32).to(torch.int32)  # same 32 bits
    call("unreal_mt_seed", ptr(self.mt), ptr(self.pos), ptr(s32), self.n, stream_ptr())

  # The device keeps numpy's own (key[624], pos) representation, so a stream can be exchanged
  # with an np.random.RandomState at any time.
  def load_numpy_state(self, random_state, env=0):
    """Copy `random_state`'s MT19937 state into env `env`'s stream."""
    name, key, pos, _, _ = random_state.get_state()
    if name != 'MT19937':
      raise _lib.UnrealError("RandomState must be MT19937")
    import numpy as np
    self.mt[:, env].copy_(torch.from_numpy(np.ascontiguousarray(key, dtype=np.uint32).view(np.int32).copy()))
    self.pos[env] = int(pos)

  def store_numpy_state(self, random_state, env=0):
    """Write env `env`'s stream back into `random_state` (draws made on the device become
    visible to every other user of that RandomState)."""
    import numpy as np
    key = self.mt[:, env].cpu().numpy().view(np.uint32).copy()
    st = random_state.get_state()
    random_state.set_state((st[0], key, int(self.pos[env]), st[3], st[4]))

  def randint(self, high, k=1):
    out = torch.empty(self.n, k, dtype=torch.int32, device=self.device)
    call("unreal_mt_randint", ptr(self.mt), ptr(self.pos), int(high), ptr(out), self.n, k, stream_ptr())
    return out

  def choose_action(self, pi, active=None, out=None):
    n, a = pi.shape
    if out is None:
      out = torch.zeros(n, dtype=torch.int32, device=self.device)
    call("unreal_choose_action", ptr(self.mt), ptr(self.pos), ptr(pi, torch.float32, "pi"),
         ptr(active, torch.uint8), ptr(out, torch.int32), n, a, stream_ptr())
    return out


# ---------------------------------------------------------------------------- replay ring
class ReplayRing(object):
  """Device ring of packed frame records, H slots for each of N envs (library-owned)."""

  def __init__(self, n_envs, history_size, device):
    self.n = int(n_envs)
    self.h = int(history_size)
    self.device = torch.device(device)
    h = ctypes.c_void_p()
    with torch.cuda.device(self.device):
      _lib.check(_lib.lib.unreal_replay_create(ctypes.byref(h), self.n, self.h), "unreal_replay_create")
    self._h = h

  def close(self):
    if self._h is not None:
      _lib.lib.unreal_replay_destroy(self._h)
      self._h = None

  def __del__(self):
    try:
      self.close()
    except Exception:
      pass

  def reset(self):
    call("unreal_replay_reset", self._h, stream_ptr())

  def add(self, frame_rec):
    if frame_rec.numel() != self.n:
      raise _lib.UnrealError("frame_rec must hold one record per env")
    call("unreal_replay_add", self._h, ptr(frame_rec, torch.int64, "frame_rec"), stream_ptr())

  def add_slots(self, frame_rec, out=None):
    """add() that reports the ring slot each frame went to: [N] i32, -1 where it was discarded."""
    if frame_rec.numel() != self.n:
      raise _lib.UnrealError("frame_rec must hold one record per env")
    slot = out if out is not None else torch.empty(self.n, dtype=torch.int32, device=self.device)
    call("unreal_replay_add_slots", self._h, ptr(frame_rec, torch.int64, "frame_rec"), ptr(slot, torch.int32, "slot"),
         stream_ptr())
    return slot

  def store(self, payload, src, slot):
    """payload [N,H,...] <- src [N,...] at slot [N] (framed mode; skipped where slot < 0)."""
    if payload.shape[0] != self.n or payload.shape[1] != self.h or tuple(payload.shape[2:]) != tuple(src.shape[1:]) \
        or src.shape[0] != self.n or payload.dtype != src.dtype:
      raise _lib.UnrealError("ring payload %s / source %s do not match a %d x %d ring" %
                             (tuple(payload.shape), tuple(src.shape), self.n, self.h))
    item = payload[0, 0].numel() * payload.element_size()
    call("unreal_ring_store", ptr(payload, name="payload"), ptr(src, name="src"), ptr(slot, torch.int32, "slot"),
         self.n, self.h, item, stream_ptr())

  def gather(self, payload, start, length, seq_len, time_major=True, out=None):
    """Payloads of the sampled sequences: [L,N,...] (time_major) or [N,L,...]; zero past `length`
    (None: all seq_len items, the reward-prediction case)."""
    if payload.shape[0] != self.n or payload.shape[1] != self.h:
      raise _lib.UnrealError("ring payload %s does not match a %d x %d ring" % (tuple(payload.shape), self.n, self.h))
    item_shape = tuple(payload.shape[2:])
    shape = ((seq_len, self.n) if time_major else (self.n, seq_len)) + item_shape
    if out is None:
      out = torch.empty(shape, dtype=payload.dtype, device=self.device)
    elif tuple(out.shape) != shape or out.dtype != payload.dtype:
      raise _lib.UnrealError("gather output must be %s %s" % (shape, payload.dtype))
    item = payload[0, 0].numel() * payload.element_size()
    call("unreal_replay_gather", self._h, ptr(payload, name="payload"), item, ptr(start, torch.int32, "start"),
         ptr(length, torch.int32, "length"), int(seq_len), 1 if time_major else 0, ptr(out, name="out"), stream_ptr())
    return out

  def state(self):
    """-> dict(full u8, count i32, top i64, n_pos i32, n_neg i32), each [N]."""
    d = self.device
    out = dict(full=torch.empty(self.n, dtype=torch.uint8, device=d),
               count=torch.empty(self.n, dtype=torch.int32, device=d),
               top=torch.empty(self.n, dtype=torch.int64, device=d),
               n_pos=torch.empty(self.n, dtype=torch.int32, device=d),
               n_neg=torch.empty(self.n, dtype=torch.int32, device=d))
    call("unreal_replay_state", self._h, ptr(out["full"]), ptr(out["count"]), ptr(out["top"]), ptr(out["n_pos"]),
         ptr(out["n_neg"]), stream_ptr())
    return out

  def export_state(self):
    """Verbatim copy of the ring: dict(rec [N,H] i64, top i64, count / n_pos / n_neg i32)."""
    d = self.device
    out = dict(rec=torch.empty(self.n, self.h, dtype=torch.int64, device=d),
               top=torch.empty(self.n, dtype=torch.int64, device=d),
               count=torch.empty(self.n, dtype=torch.int32, device=d),
               n_pos=torch.empty(self.n, dtype=torch.int32, device=d),
               n_neg=torch.empty(self.n, dtype=torch.int32, device=d))
    call("unreal_replay_copy", self._h, 0, ptr(out["rec"]), ptr(out["top"]), ptr(out["count"]), ptr(out["n_pos"]),
         ptr(out["n_neg"]), stream_ptr())
    return out

  def import_state(self, st):
    if tuple(st["rec"].shape) != (self.n, self.h):
      raise _lib.UnrealError("replay checkpoint is for %s envs x frames, ring is %d x %d" % (tuple(st["rec"].shape), self.n, self.h))
    t = {k: st[k].to(self.device).contiguous() for k in ("rec", "top", "count", "n_pos", "n_neg")}
    call("unreal_replay_copy", self._h, 1, ptr(t["rec"], torch.int64), ptr(t["top"], torch.int64),
         ptr(t["count"], torch.int32), ptr(t["n_pos"], torch.int32), ptr(t["n_neg"], torch.int32), stream_ptr())
    torch.cuda.current_stream().synchronize()      # `t` must outlive the copies

  def sample_sequence(self, streams, seq_len):
    """-> start [N] i32, len [N] i32, rec [N, seq_len] i64 (zero past len)."""
    d = self.device
    start = torch.empty(self.n, dtype=torch.int32, device=d)
    length = torch.empty(self.n, dtype=torch.int32, device=d)
    rec = torch.empty(self.n, seq_len, dtype=torch.int64, device=d)
    call("unreal_replay_sample_sequence", self._h, ptr(streams.mt), ptr(streams.pos), int(seq_len), ptr(start),
         ptr(length), ptr(rec), stream_ptr())
    return start, length, rec

  def sample_rp(self, streams):
    """-> start [N] i32 (raw position of the first of four frames), rec [N, 4] i64."""
    d = self.device
    start = torch.empty(self.n, dtype=torch.int32, device=d)
    rec = torch.empty(self.n, 4, dtype=torch.int64, device=d)
    call("unreal_replay_sample_rp", self._h, ptr(streams.mt), ptr(streams.pos), ptr(start), ptr(rec), stream_ptr())
    return start, rec


def rows_select(out, src, idx=None, mask=None):
  """out[e] <- src[idx[e]] (idx None: src[e]) for the envs with mask[e] != 0 (None: all); rows = everything after dim 0."""
  n = out.shape[0]
  if out.dtype != src.dtype or tuple(out.shape[1:]) != tuple(src.shape[1:]):
    raise _lib.UnrealError("rows_select: out %s %s and src %s %s rows differ" % (tuple(out.shape), out.dtype, tuple(src.shape), src.dtype))
  if idx is None and src.shape[0] != n:
    raise _lib.UnrealError("rows_select: without idx, src must hold one row per env")
  item = out[0].numel() * out.element_size()
  if mask is not None and mask.dtype == torch.bool:
    mask = mask.to(torch.uint8)
  call("unreal_rows_select", ptr(out, name="out"), ptr(src, name="src"), ptr(idx, torch.int64, "idx"),
       ptr(mask, torch.uint8, "mask"), n, item, stream_ptr())
  return out


def frame_unpack(rec, fields=("pos0", "pos1", "action", "reward", "terminal", "last_action", "last_reward", "valid")):
  """Packed records (any shape) -> dict of SoA tensors with that shape (+[2] for positions)."""
  m = rec.numel()
  d = rec.device
  shape = tuple(rec.shape)
  spec = dict(pos0=(torch.int32, shape + (2,)), pos1=(torch.int32, shape + (2,)), action=(torch.int32, shape),
              reward=(torch.float32, shape), terminal=(torch.uint8, shape), last_action=(torch.int32, shape),
              last_reward=(torch.float32, shape), valid=(torch.uint8, shape))
  out = {k: torch.empty(spec[k][1], dtype=spec[k][0], device=d) for k in fields}
  g = lambda k: ptr(out[k]) if k in out else None  # noqa: E731
  call("unreal_frame_unpack", ptr(rec, torch.int64, "rec"), m, g("pos0"), g("pos1"), g("action"), g("reward"),
       g("terminal"), g("last_action"), g("last_reward"), g("valid"), stream_ptr())
  return out


def frame_pack(action, reward, terminal, last_action=None, last_reward=None, active=None, out=None):
  """SoA step outputs of a generic-frame env -> packed records [N] i64 (rewards as their sign)."""
  n = action.numel()
  rec = out if out is not None else torch.empty(n, dtype=torch.int64, device=action.device)
  call("unreal_frame_pack", ptr(action, torch.int32, "action"), ptr(reward, torch.float32, "reward"),
       ptr(terminal, torch.uint8, "terminal"), ptr(last_action, torch.int32, "last_action"),
       ptr(last_reward, torch.float32, "last_reward"), ptr(active, torch.uint8, "active"),
       ptr(rec, torch.int64, "rec"), n, stream_ptr())
  return rec


# ---------------------------------------------------------------------------- optimiser
def grad_sumsq(grad, out=None):
  """sum(grad^2) as a device double; `out` (1-element float64) is accumulated into."""
  if out is None:
    out = torch.zeros(1, dtype=torch.float64, device=grad.device)
  call("unreal_grad_sumsq", ptr(grad, torch.float32, "grad"), grad.numel(), ptr(out, torch.float64), stream_ptr())
  return out


def rmsprop_update(var, rms, mom, grad, sumsq, lr, decay, momentum, eps, clip_norm, grad_scale=1.0, grad_norm=None):
  if isinstance(lr, torch.Tensor):       # learning rate in device memory (read when the kernel runs)
    call("unreal_rmsprop_update_dlr", ptr(var, torch.float32, "var"), ptr(rms, torch.float32, "rms"),
         ptr(mom, torch.float32, "mom"), ptr(grad, torch.float32, "grad"), var.numel(),
         ptr(sumsq, torch.float64, "sumsq"), float(grad_scale), ptr(lr, torch.float32, "lr"), float(decay), float(momentum),
         float(eps), float(clip_norm), ptr(grad_norm, torch.float32, "grad_norm"), stream_ptr())
    return grad_norm
  call("unreal_rmsprop_update", ptr(var, torch.float32, "var"), ptr(rms, torch.float32, "rms"),
       ptr(mom, torch.float32, "mom"), ptr(grad, torch.float32, "grad"), var.numel(),
       ptr(sumsq, torch.float64, "sumsq"), float(grad_scale), float(lr), float(decay), float(momentum), float(eps),
       float(clip_norm), ptr(grad_norm, torch.float32, "grad_norm"), stream_ptr())
  return grad_norm


# ---------------------------------------------------------------------------- K7: tcgen05 GEMM
def _mat(t, name):
  """(data_ptr, leading dimension) of a 2-D bf16 CUDA tensor whose rows are contiguous."""
  if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dim() != 2 or t.dtype != torch.bfloat16:
    raise _lib.UnrealError("%s must be a 2-D bfloat16 CUDA tensor" % name)
  if t.stride(1) != 1 and t.shape[1] != 1:
    raise _lib.UnrealError("%s must have contiguous rows" % name)
  return t.data_ptr(), t.stride(0)


def gemm_bf16(a, b, out=None, a_mn_major=False, b_mn_major=False, bias=None, add=None, relu=False,
              accumulate=False, split_k=1, out_dtype=torch.float32):
  """C[M,N] = act(A @ B + bias + add) on the tcgen05 tensor path, fp32 accumulation.

  a: [M,K] bf16 (or [K,M] when a_mn_major), b: [N,K] bf16 (or [K,N] when b_mn_major -- TF's
  [in,out] weight layout).  out: f32 or bf16 [M,N] with contiguous rows (allocated if None)."""
  if a_mn_major:
    k, m = a.shape
  else:
    m, k = a.shape
  if b_mn_major:
    kb, n = b.shape
  else:
    n, kb = b.shape
  if kb != k:
    raise _lib.UnrealError("gemm_bf16: inner dimensions differ (%d vs %d)" % (k, kb))
  if out is None:
    out = (torch.zeros if (accumulate or split_k > 1) else torch.empty)(m, n, dtype=out_dtype, device=a.device)
  if out.dim() != 2 or tuple(out.shape) != (m, n) or (out.stride(1) != 1 and n != 1):
    raise _lib.UnrealError("gemm_bf16: out must be [%d,%d] with contiguous rows" % (m, n))
  if out.dtype not in (torch.float32, torch.bfloat16):
    raise _lib.UnrealError("gemm_bf16: out must be float32 or bfloat16")
  if add is not None and (add.dtype != torch.float32 or tuple(add.shape) != (m, n) or add.stride(0) != out.stride(0)):
    raise _lib.UnrealError("gemm_bf16: add must be f32 [M,N] with the same row stride as out")
  pa, lda = _mat(a, "a")
  pb, ldb = _mat(b, "b")
  call("unreal_gemm_bf16", pa, lda, 1 if a_mn_major else 0, pb, ldb, 1 if b_mn_major else 0, out.data_ptr(),
       out.stride(0), 1 if out.dtype == torch.bfloat16 else 0, ptr(bias, torch.float32, "bias"),
       None if add is None else add.data_ptr(), 1 if relu else 0, 1 if accumulate else 0, int(split_k), m, n, k,
       stream_ptr())
  return out


# ---------------------------------------------------------------------------- K7: conv / LSTM support
def im2col(x, kh, kw, stride, out=None):
  """x [S,H,W,C] f32 / u8 / bf16 -> bf16 [S*OH*OW, KH*KW*C] patches (HWIO column order)."""
  s, h, w, c = x.shape
  oh, ow = (h - kh) // stride + 1, (w - kw) // stride + 1
  if out is None:
    out = torch.empty(s * oh * ow, kh * kw * c, dtype=torch.bfloat16, device=x.device)
  call("unreal_im2col", ptr(x, None, "x"), _lib.dtype_tag(x), ptr(out, torch.bfloat16, "out"), s, h, w, c, kh, kw,
       stride, stream_ptr())
  return out


def col2im(cols, s, h, w, c, kh, kw, stride, bias=None, relu=False, out_dtype=torch.float32, out=None):
  """cols [S*OH*OW, KH*KW*C] f32/bf16 -> [S,H,W,C]: sum of overlapping taps (+ bias, ReLU)."""
  if out is None:
    out = torch.empty(s, h, w, c, dtype=out_dtype, device=cols.device)
  call("unreal_col2im", ptr(cols, None, "cols"), _lib.dtype_tag(cols), ptr(out, None, "out"), _lib.dtype_tag(out),
       ptr(bias, torch.float32, "bias"), 1 if relu else 0, s, h, w, c, kh, kw, stride, stream_ptr())
  return out


def lstm_cell_fwd(gates, c_prev, c_out, h_out, h16_out):
  """h16_out [n,256] bf16; a column slice of a wider row-major buffer is accepted (rows stride(0) apart)."""
  n = gates.shape[0]
  if gates.dtype == torch.bfloat16:       # bf16 gate storage
    if h16_out.dim() != 2 or h16_out.shape[1] != 256 or h16_out.stride(1) != 1 or h16_out.dtype != torch.bfloat16:
      raise _lib.UnrealError("h16_out must be bf16 [n,256] with contiguous rows")
    call("unreal_lstm_cell_fwd_g16", ptr(gates, torch.bfloat16, "gates"), ptr(c_prev, torch.float32, "c_prev"),
         ptr(c_out, torch.float32, "c_out"), ptr(h_out, torch.float32, "h_out"), h16_out.data_ptr(), int(h16_out.stride(0)),
         n, stream_ptr())
    return
  if h16_out.is_contiguous():
    call("unreal_lstm_cell_fwd", ptr(gates, torch.float32, "gates"), ptr(c_prev, torch.float32, "c_prev"),
         ptr(c_out, torch.float32, "c_out"), ptr(h_out, torch.float32, "h_out"), ptr(h16_out, torch.bfloat16, "h16_out"),
         n, stream_ptr())
    return
  if h16_out.dim() != 2 or h16_out.shape[1] != 256 or h16_out.stride(1) != 1 or h16_out.dtype != torch.bfloat16:
    raise _lib.UnrealError("h16_out must be bf16 [n,256] with contiguous rows")
  call("unreal_lstm_cell_fwd_ld", ptr(gates, torch.float32, "gates"), ptr(c_prev, torch.float32, "c_prev"),
       ptr(c_out, torch.float32, "c_out"), ptr(h_out, torch.float32, "h_out"), h16_out.data_ptr(), int(h16_out.stride(0)),
       n, stream_ptr())


def _rows2d(t, cols, dtype, name):
  """[n, cols] view with contiguous rows (a column slice of a wider row-major buffer is accepted) -> (pointer, row pitch)."""
  if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype != dtype or t.dim() != 2 or t.shape[1] != cols or t.stride(1) != 1:
    raise _lib.UnrealError("%s must be a CUDA %s [n,%d] tensor with contiguous rows" % (name, dtype, cols))
  return t.data_ptr(), int(t.stride(0))


def tile32(x, rows=None):
  """[n, C] row-major -> the 32-row tiled layout of unreal_lstm_step_fwd / _bwd, [rows, C] with rows = n rounded up to 32
  (16-byte chunk ch of row r at chunk index (r // 32 * chunks_per_row + ch) * 32 + r % 32)."""
  n, c = x.shape
  e = 16 // x.element_size()
  rows = (n + 31) // 32 * 32 if rows is None else rows
  buf = x.new_zeros(rows, c)
  buf[:n] = x
  return buf.view(rows // 32, 32, c // e, e).permute(0, 2, 1, 3).contiguous().view(rows, c)


def untile32(xt, n):
  """inverse of tile32: the first n rows, row-major"""
  rows, c = xt.shape
  e = 16 // xt.element_size()
  return xt.view(rows // 32, c // e, 32, e).permute(0, 2, 1, 3).reshape(rows, c)[:n]


def lstm_step_fwd(xh, w, bias, c_prev, c_out, h_out=None, h16_out=None, acts=None, active=None, h_copy=None, tiled=False):
  """One LSTM step in one launch (unreal_lstm_step_fwd): step GEMM over xh [n,k] bf16 (rows may be a slice) x w [k,1024]
  with the cell in the epilogue.  c_out may be c_prev (acting: in place, only rows with active != 0).
  tiled: c_prev, c_out, acts are `tile32` buffers [n rounded up to 32, .]."""
  n, k = xh.shape
  xp, ldx = _rows2d(xh, k, torch.bfloat16, "xh")
  if w.shape != (k, 1024):
    raise _lib.UnrealError("w must be [%d,1024], got %s" % (k, tuple(w.shape)))
  hp, hld = (None, 0) if h16_out is None else _rows2d(h16_out, 256, torch.bfloat16, "h16_out")
  nt = (n + 31) // 32 * 32 if tiled else n
  for name, t, rows in (("c_prev", c_prev, nt), ("c_out", c_out, nt), ("h_out", h_out, n), ("h_copy", h_copy, n)):
    if t is not None and tuple(t.shape) != (rows, 256):
      raise _lib.UnrealError("%s must be [%d,256]" % (name, rows))
  if acts is not None and tuple(acts.shape) != (nt, 1024):
    raise _lib.UnrealError("acts must be [%d,1024]" % nt)
  call("unreal_lstm_step_fwd", xp, ldx, ptr(w, torch.bfloat16, "w"), ptr(bias, torch.float32, "bias"),
       ptr(c_prev, torch.float32, "c_prev"), ptr(c_out, torch.float32, "c_out"), ptr(h_out, torch.float32, "h_out"),
       ptr(h_copy, torch.float32, "h_copy"), hp, hld, ptr(acts, torch.bfloat16, "acts"), ptr(active, torch.uint8, "active"),
       1 if tiled else 0, n, k, stream_ptr())


def lstm_step_bwd(dgates_next, wh, acts, c_prev, c, dh, dc, dgates, dh2=None, tiled=False):
  """One backward LSTM step in one launch (unreal_lstm_step_bwd): dh_rec = dgates_next [n,1024] x wh [256,1024]^T, then the
  cell's backward pass of this step on dh + dh_rec -> dgates [n,1024] bf16, dc [n,256] in place.  dgates_next None: the
  unroll's last step (dh + dh2).  tiled: acts, c_prev, c, dc are `tile32` buffers."""
  n = dgates.shape[0]
  wp, ldw = _rows2d(wh, 1024, torch.bfloat16, "wh")
  if wh.shape[0] != 256:
    raise _lib.UnrealError("wh must be [256,1024]")
  nt = (n + 31) // 32 * 32 if tiled else n
  for name, t, rows, cols in (("dgates_next", dgates_next, n, 1024), ("acts", acts, nt, 1024), ("dgates", dgates, n, 1024),
                              ("c_prev", c_prev, nt, 256), ("c", c, nt, 256), ("dh", dh, n, 256), ("dh2", dh2, n, 256),
                              ("dc", dc, nt, 256)):
    if t is not None and tuple(t.shape) != (rows, cols):
      raise _lib.UnrealError("%s must be [%d,%d]" % (name, rows, cols))
  call("unreal_lstm_step_bwd", ptr(dgates_next, torch.bfloat16, "dgates_next"), wp, ldw, ptr(acts, torch.bfloat16, "acts"),
       ptr(c_prev, torch.float32, "c_prev"), ptr(c, torch.float32, "c"), ptr(dh, torch.float32, "dh"), ptr(dh2, torch.float32, "dh2"),
       ptr(dc, torch.float32, "dc"), ptr(dgates, torch.bfloat16, "dgates"), 1 if tiled else 0, n, stream_ptr())


def lstm_cell_bwd(gates_act, c_prev, c, dh, dc, dgates16, dh_rec=None):
  """dh (+ dh_rec): gradient w.r.t. h_t; dc in / out; dgates16 [n,1024] bf16 out."""
  n = gates_act.shape[0]
  if gates_act.dtype == torch.bfloat16:
    call("unreal_lstm_cell_bwd_g16", ptr(gates_act, torch.bfloat16, "gates_act"), ptr(c_prev, torch.float32, "c_prev"),
         ptr(c, torch.float32, "c"), ptr(dh, torch.float32, "dh"), ptr(dh_rec, torch.float32, "dh_rec"),
         ptr(dc, torch.float32, "dc"), ptr(dgates16, torch.bfloat16, "dgates16"), n, stream_ptr())
    return
  call("unreal_lstm_cell_bwd2", ptr(gates_act, torch.float32, "gates_act"), ptr(c_prev, torch.float32, "c_prev"),
       ptr(c, torch.float32, "c"), ptr(dh, torch.float32, "dh"), ptr(dh_rec, torch.float32, "dh_rec"),
       ptr(dc, torch.float32, "dc"), ptr(dgates16, torch.bfloat16, "dgates16"), n, stream_ptr())


def s2d_frames(frames, out=None):
  """frames [S,84,84,3] f32 / u8 -> space-to-depth bf16, plane-major [S,6,441,8]:
  x''[s, q, Y*21+X, e] = frame[s, 4Y+dy, 4X+dx, c] with dy*12 + dx*3 + c = q*8 + e."""
  s = frames.shape[0]
  if tuple(frames.shape[1:]) != (84, 84, 3):
    raise _lib.UnrealError("s2d_frames expects [S,84,84,3] frames")
  if out is None:
    out = torch.empty(s, 6, 441, 8, dtype=torch.bfloat16, device=frames.device)
  call("unreal_s2d_frames", ptr(frames, None, "frames"), _lib.dtype_tag(frames), ptr(out, torch.bfloat16, "out"), s,
       stream_ptr())
  return out


def conv1_w_planes(w16):
  """conv1 filter [8,8,3,16] (bf16) -> [4 taps, 6 channel chunks, 16 outputs, 8] : the un-swizzled
  K-major UMMA B operand of each tap, resident in shared memory for the whole conv1 kernel."""
  taps = _tap_major(w16, 4).view(16, 4, 64)[:, :, :48]
  return taps.reshape(16, 4, 6, 8).permute(1, 2, 0, 3).contiguous()


def _tap_major(w16, stride):
  """HWIO filter [2s,2s,C,O] (bf16) -> tap-major K-major matrix [O, 4*64]: tap t = by*2+bx holds
  W[s*by+dy, s*bx+dx, c, o] in (dy,dx,c) order, zero padded to 64 columns."""
  k, _, c, o = w16.shape
  s = stride
  t = w16.reshape(2, s, 2, s, c, o).permute(5, 0, 2, 1, 3, 4).reshape(o, 4, s * s * c)   # [o, (by,bx), (dy,dx,c)]
  out = torch.zeros(o, 4, 64, dtype=w16.dtype, device=w16.device)
  out[:, :, :s * s * c] = t
  return out.reshape(o, 256).contiguous()


def conv_taps(w16, stride):
  """conv2's HWIO filter [4,4,16,32] (bf16) -> the K-major matrix [O, 256] the fused kernel keeps resident:
  K = (ky, kx, c), i.e. one 64-column (128-byte) slice per filter row ky."""
  k, _, c, o = w16.shape
  if (k, stride) != (4, 2) or c not in (16, 8):
    raise _lib.UnrealError("conv_taps: the fused forward kernel is conv2's geometry (4x4x16 or 4x4x8, stride 2)")
  return w16.reshape(k * k * c, o).t().contiguous()


def conv_fwd(x, layer, w_taps, bias, out=None):
  """layer 1: x = s2d frames [S,6,441,8], w_taps = conv1_w_planes(W) -> [S,20,20,16];
  layer 2: x = h1 [S,20,20,16], w_taps = conv_taps(W, 2) -> [S,9,9,32]  (bias + ReLU fused, bf16 out)."""
  s = x.shape[0]
  shape = (s, 20, 20, 16) if layer == 1 else (s, 9, 9, 32)
  if out is None:
    out = torch.empty(*shape, dtype=torch.bfloat16, device=x.device)
  call("unreal_conv_fwd", ptr(x, torch.bfloat16, "x"), int(layer), ptr(w_taps, torch.bfloat16, "w_taps"),
       ptr(bias, torch.float32, "bias"), ptr(out, torch.bfloat16, "out"), s, stream_ptr())
  return out


def relu_grad(dy, y=None, want_out=True, want_db=True, planes=False):
  """dy [rows, cols] bf16 / f32, y bf16 or None -> (dy * (y > 0) as bf16, column sums f32).
  planes=True: the bf16 output is laid out [cols/8, rows, 8] (8-column chunks as planes)."""
  rows, cols = dy.shape
  if not dy.is_contiguous():
    dy = dy.contiguous()
  out = None
  if want_out:
    out = torch.empty((cols // 8, rows, 8) if planes else (rows, cols), dtype=torch.bfloat16, device=dy.device)
  db = torch.zeros(cols, dtype=torch.float32, device=dy.device) if want_db else None
  call("unreal_relu_grad", ptr(dy, None, "dy"), _lib.dtype_tag(dy), ptr(y, torch.bfloat16, "y"),
       ptr(out, torch.bfloat16, "out"), ptr(db, torch.float32, "db"), rows, cols, 1 if planes else 0, stream_ptr())
  return out, db


def conv1_wgrad(xpp, dy_planes):
  """x'' [S,6,441,8] bf16 (forward's space-to-depth frames), dy_planes [2, S*400, 8] bf16 (masked
  gradient of conv1's output) -> filter gradient in HWIO layout [8,8,3,16] f32."""
  s = xpp.shape[0]
  acc = torch.zeros(4, 16, 48, dtype=torch.float32, device=xpp.device)
  p21 = dy_planes.shape[1] == s * 420          # planes on the 21-pixel row pitch (conv2_dgrad_relu(pitch21=True))
  call("unreal_conv1_wgrad_p21" if p21 else "unreal_conv1_wgrad", ptr(xpp, torch.bfloat16, "xpp"),
       ptr(dy_planes, torch.bfloat16, "dy_planes"), ptr(acc, torch.float32), s, stream_ptr())
  # acc[(by,bx), o, (dy,dx,c)] -> W[4by+dy, 4bx+dx, c, o]
  return acc.view(2, 2, 16, 4, 4, 3).permute(0, 3, 1, 4, 5, 2).reshape(8, 8, 3, 16)


def pc_loss(y8, act, target, mask, num_actions, lam, want_loss=True, want_grad=False, go=None):
  """Pixel-control dueling head + loss on the merged 8-channel deconv output y8 [S, px, 8] f32:
  returns (loss as a 1-element float64 tensor or None, dy8 or None)."""
  s, px = y8.shape[0], y8.shape[1]
  loss = torch.zeros(1, dtype=torch.float64, device=y8.device) if want_loss else None
  dy = torch.empty_like(y8) if want_grad else None
  call("unreal_pc_loss", ptr(y8, torch.float32, "y8"), ptr(act, torch.int32, "act"), ptr(target, torch.float32, "target"),
       ptr(mask, torch.float32, "mask"), int(num_actions), float(lam), s, px, ptr(loss, torch.float64),
       ptr(dy, torch.float32), ptr(go, torch.float32, "go"), stream_ptr())
  return loss, dy


def conv2_wgrad(h1, dy16):
  """h1 [S,20,20,16] (or [S,20,20,8]) bf16, dy16 [S*81, 32] bf16 (masked gradient of conv2's output) -> filter gradient
  in HWIO layout [4,4,16 (8),32] f32, the im2col done by TMA boxes."""
  s, c = h1.shape[0], h1.shape[-1]
  if c not in (16, 8):
    raise ValueError("conv2_wgrad: 16 or 8 input channels")
  acc = torch.zeros(4, 4, c, 32, dtype=torch.float32, device=h1.device)     # the kernel accumulates in HWIO order
  call("unreal_conv2_wgrad" if c == 16 else "unreal_conv2_wgrad_c8", ptr(h1, torch.bfloat16, "h1"),
       ptr(dy16, torch.bfloat16, "dy16"), ptr(acc, torch.float32), s, stream_ptr())
  return acc


def conv2_dgrad_taps(w16):
  """conv2 filter [4,4,16,32] bf16 (HWIO) -> [4 taps, 64 (dy,dx,c), 32 out]: the resident B tiles of
  the transposed-convolution kernel, W[2by+dy, 2bx+dx, c, o]."""
  return w16.reshape(2, 2, 2, 2, 16, 32).permute(0, 2, 1, 3, 4, 5).reshape(4, 64, 32).contiguous()


def conv2_dgrad(dy16, w_dtaps, out=None):
  """dy16 [S*81, 32] bf16 -> gradient w.r.t. conv2's input, dense bf16 [S,20,20,16] (un-masked)."""
  s = dy16.shape[0] // 81
  if out is None:
    out = torch.empty(s, 20, 20, 16, dtype=torch.bfloat16, device=dy16.device)
  call("unreal_conv2_dgrad", ptr(dy16, torch.bfloat16, "dy16"), ptr(w_dtaps, torch.bfloat16, "w_dtaps"),
       ptr(out, torch.bfloat16, "out"), s, stream_ptr())
  return out


def pc_deconv_taps(w8):
  """merged pixel-control deconv filter [4,4,8,32] bf16 ([kh,kw,out,in]) -> [4 taps, 32 (dy,dx,c), 32 in]."""
  return w8.reshape(2, 2, 2, 2, 8, 32).permute(0, 2, 1, 3, 4, 5).reshape(4, 32, 32).contiguous()


def pc_deconv_fwd(h16, w_dtaps, bias8, out=None):
  """h16 bf16 [S,9,9,32] (any view of S*2592) -> relu(conv2d_transpose + bias) f32 [S,20,20,8]."""
  s = h16.numel() // 2592
  if out is None:
    out = torch.empty(s, 20, 20, 8, dtype=torch.float32, device=h16.device)
  call("unreal_pc_deconv_fwd", ptr(h16, torch.bfloat16, "h16"), ptr(w_dtaps, torch.bfloat16, "w_dtaps"),
       ptr(bias8, torch.float32, "bias8"), ptr(out, torch.float32, "out"), s, stream_ptr())
  return out


def conv2_dgrad_relu(dy16, w_dtaps, h1, pitch21=False):
  """conv2's input gradient fused with conv1's ReLU gradient: dy16 [S*81,32] bf16, h1 [S,20,20,16] bf16 ->
  (masked gradient as conv1-wgrad planes [2, S*400, 8] bf16 -- or [2, S*420, 8] on the x'' grid's 21-pixel
  row pitch with a zero column when pitch21 -- and conv1's bias gradient [16] f32)."""
  s = dy16.shape[0] // 81
  planes = torch.empty(2, s * (420 if pitch21 else 400), 8, dtype=torch.bfloat16, device=dy16.device)
  db = torch.zeros(16, dtype=torch.float32, device=dy16.device)
  call("unreal_conv2_dgrad_relu", ptr(dy16, torch.bfloat16, "dy16"), ptr(w_dtaps, torch.bfloat16, "w_dtaps"),
       ptr(h1, torch.bfloat16, "h1"), ptr(planes, torch.bfloat16, "planes"), ptr(db, torch.float32, "db"), s,
       1 if pitch21 else 0, stream_ptr())
  return planes, db


def conv1_fwd_maze(pos, w_taps, bias, out=None):
  """Render-fused conv1 forward for maze frames: pos [S,2] i32 (agent cells) -> h1 bf16 [S,20,20,16]."""
  s = pos.shape[0]
  if out is None:
    out = torch.empty(s, 20, 20, 16, dtype=torch.bfloat16, device=pos.device)
  call("unreal_conv1_fwd_maze", ptr(pos, torch.int32, "pos"), ptr(w_taps, torch.bfloat16, "w_taps"),
       ptr(bias, torch.float32, "bias"), ptr(out, torch.bfloat16, "out"), s, stream_ptr())
  return out


def split_bf16(w32):
  """fp32 tensor -> (hi, lo) bf16 with hi = bf16(w), lo = bf16(w - hi): hi + lo holds w to about 16 mantissa bits."""
  hi = w32.to(torch.bfloat16)
  return hi, (w32 - hi.float()).to(torch.bfloat16)


def s2d_frames_split(frames):
  """frames [S,84,84,3] f32 / u8 -> (x'' hi, x'' lo) bf16 [S,6,441,8] each, as s2d_frames; lo = bf16(x - hi)."""
  s = frames.shape[0]
  if tuple(frames.shape[1:]) != (84, 84, 3):
    raise _lib.UnrealError("s2d_frames_split expects [S,84,84,3] frames")
  hi = torch.empty(s, 6, 441, 8, dtype=torch.bfloat16, device=frames.device)
  lo = torch.empty_like(hi)
  call("unreal_s2d_frames_split", ptr(frames, None, "frames"), _lib.dtype_tag(frames), ptr(hi, torch.bfloat16, "hi"),
       ptr(lo, torch.bfloat16, "lo"), s, stream_ptr())
  return hi, lo


def conv1_fwd_split(xpp_hi, xpp_lo, w_hi, w_lo, bias):
  """Split-bf16 conv1: x'' hi / lo planes [S,6,441,8] (xpp_lo None: the input is exactly bf16), filter planes hi / lo
  (conv1_w_planes of both halves) -> h1 = relu(conv + bias) as (hi, lo) bf16 [S,20,20,16]."""
  s = xpp_hi.shape[0]
  hi = torch.empty(s, 20, 20, 16, dtype=torch.bfloat16, device=xpp_hi.device)
  lo = torch.empty_like(hi)
  call("unreal_conv1_fwd_split", ptr(xpp_hi, torch.bfloat16, "xpp_hi"), ptr(xpp_lo, torch.bfloat16, "xpp_lo"),
       ptr(w_hi, torch.bfloat16, "w_hi"), ptr(w_lo, torch.bfloat16, "w_lo"), ptr(bias, torch.float32, "bias"),
       ptr(hi, torch.bfloat16, "hi"), ptr(lo, torch.bfloat16, "lo"), s, stream_ptr())
  return hi, lo


def conv1_fwd_maze_split(pos, w_hi, w_lo, bias):
  """Split-bf16 render-fused conv1: pos [S,2] i32 -> h1 (hi, lo) bf16 [S,20,20,16]."""
  s = pos.shape[0]
  hi = torch.empty(s, 20, 20, 16, dtype=torch.bfloat16, device=pos.device)
  lo = torch.empty_like(hi)
  call("unreal_conv1_fwd_maze_split", ptr(pos, torch.int32, "pos"), ptr(w_hi, torch.bfloat16, "w_hi"),
       ptr(w_lo, torch.bfloat16, "w_lo"), ptr(bias, torch.float32, "bias"), ptr(hi, torch.bfloat16, "hi"),
       ptr(lo, torch.bfloat16, "lo"), s, stream_ptr())
  return hi, lo


def conv2_fwd_split(h1_hi, h1_lo, w_hi, w_lo, bias):
  """Split-bf16 conv2: h1 hi / lo [S,20,20,16], filters hi / lo (conv_taps of both halves) -> h2 bf16 [S,9,9,32]."""
  s = h1_hi.shape[0]
  out = torch.empty(s, 9, 9, 32, dtype=torch.bfloat16, device=h1_hi.device)
  call("unreal_conv2_fwd_split", ptr(h1_hi, torch.bfloat16, "h1_hi"), ptr(h1_lo, torch.bfloat16, "h1_lo"),
       ptr(w_hi, torch.bfloat16, "w_hi"), ptr(w_lo, torch.bfloat16, "w_lo"), ptr(bias, torch.float32, "bias"),
       ptr(out, torch.bfloat16, "out"), s, stream_ptr())
  return out


def conv1_wgrad_maze(pos, dy_planes21):
  """Render-fused conv1 filter gradient: pos [S,2] i32, dy planes [2, S*420, 8] bf16 -> HWIO [8,8,3,16] f32."""
  s = pos.shape[0]
  if dy_planes21.shape[1] != s * 420:
    raise _lib.UnrealError("conv1_wgrad_maze needs the dY planes on the 21-pixel row pitch")
  acc = torch.zeros(4, 16, 48, dtype=torch.float32, device=pos.device)
  call("unreal_conv1_wgrad_maze", ptr(pos, torch.int32, "pos"), ptr(dy_planes21, torch.bfloat16, "dy_planes"),
       ptr(acc, torch.float32), s, stream_ptr())
  return acc.view(2, 2, 16, 4, 4, 3).permute(0, 3, 1, 4, 5, 2).reshape(8, 8, 3, 16)


def pc_loss_grad16(y8, act, target, mask, num_actions, lam, go):
  """d pixel-control loss / d (pre-ReLU deconv output) as bf16 [S, px, 16] (channels 8..15 zero: conv2's input
  geometry) plus the deconv bias gradient [8] f32."""
  s, px = y8.shape[0], y8.shape[1]
  dy16 = torch.empty(s, px, 16, dtype=torch.bfloat16, device=y8.device)
  db8 = torch.zeros(8, dtype=torch.float32, device=y8.device)
  call("unreal_pc_loss_grad16", ptr(y8, torch.float32, "y8"), ptr(act, torch.int32, "act"), ptr(target, torch.float32, "target"),
       ptr(mask, torch.float32, "mask"), int(num_actions), float(lam), s, px, ptr(dy16, torch.bfloat16),
       ptr(db8, torch.float32), ptr(go, torch.float32, "go"), stream_ptr())
  return dy16, db8


def conv2_fwd_linear(x, w_taps, out=None, scale=None, mask_y=None, want_db=True):
  """conv2's geometry without bias / ReLU: x bf16 [S,20,20,16], w_taps = conv_taps(W [4,4,16,32], 2) -> bf16 [S,9,9,32];
  `scale`: device scalar (f32 [1]) multiplied into the result before rounding.  `mask_y` (bf16, S*2592 elements: the ReLU
  output the result is a gradient of): the result is zeroed where mask_y <= 0 and (out, db f32 [2592] = its sum over
  samples) is returned."""
  s = x.shape[0]
  if out is None:
    out = torch.empty(s, 9, 9, 32, dtype=torch.bfloat16, device=x.device)
  if mask_y is not None:
    if mask_y.numel() != s * 2592:
      raise ValueError("conv2_fwd_linear: mask_y must hold S*2592 elements")
    db = torch.zeros(2592, dtype=torch.float32, device=x.device) if want_db else None
    if x.shape[-1] * 16 != w_taps.shape[1] or x.shape[-1] not in (16, 8):
      raise ValueError("conv2_fwd_linear: x [S,20,20,C] needs w_taps [32, 16*C], C = 16 or 8")
    call("unreal_conv2_fwd_linear_masked", ptr(x, torch.bfloat16, "x"), int(x.shape[-1]), ptr(w_taps, torch.bfloat16, "w_taps"),
         ptr(scale, torch.float32, "scale"), ptr(mask_y, torch.bfloat16, "mask_y"), ptr(out, torch.bfloat16, "out"),
         ptr(db, torch.float32, "db"), s, stream_ptr())
    return out, db
  if scale is not None:
    call("unreal_conv2_fwd_linear_scaled", ptr(x, torch.bfloat16, "x"), ptr(w_taps, torch.bfloat16, "w_taps"),
         ptr(scale, torch.float32, "scale"), ptr(out, torch.bfloat16, "out"), s, stream_ptr())
    return out
  call("unreal_conv2_fwd_linear", ptr(x, torch.bfloat16, "x"), ptr(w_taps, torch.bfloat16, "w_taps"),
       ptr(out, torch.bfloat16, "out"), s, stream_ptr())
  return out


def _pc16(w_dtaps, bias):
  """True for the 16-channel head (8..15 actions): a [16] bias or [4,64,32] deconv taps (conv2_dgrad_taps of [4,4,16,32])."""
  wide = bias.numel() == 16 or tuple(w_dtaps.shape) == (4, 64, 32)
  if wide and not (bias.numel() == 16 and w_dtaps.numel() == 4 * 64 * 32):
    raise _lib.UnrealError("the 16-channel pixel-control head needs a [16] bias and [4,64,32] deconv taps")
  return wide


def pc_deconv_qmax(h16, w_dtaps, bias8, num_actions, out=None):
  """max over actions of the pixel-control Q map, straight from the deconv's epilogue: h16 bf16 [S,9,9,32] -> f32 [S,20,20].
  A [16] bias with [4,64,32] taps selects the 16-channel head (8..15 actions)."""
  s = h16.numel() // 2592
  if out is None:
    out = torch.empty(s, 20, 20, dtype=torch.float32, device=h16.device)
  call("unreal_pc_deconv_qmax16" if _pc16(w_dtaps, bias8) else "unreal_pc_deconv_qmax", ptr(h16, torch.bfloat16, "h16"),
       ptr(w_dtaps, torch.bfloat16, "w_dtaps"),
       ptr(bias8, torch.float32, "bias8"), int(num_actions), s, ptr(out, torch.float32, "qmax"), stream_ptr())
  return out


def pc_deconv_loss(h16, w_dtaps, bias8, act, target, mask, num_actions, lam, c8=False, planes=False):
  """Pixel-control head + loss in one kernel: h16 bf16 [S,9,9,32] (any view of S*2592) -> (loss f64 [1],
  dy16 bf16 [S,400,16] = d loss / d pre-ReLU output, un-scaled by the upstream gradient, db8 [8]).  `c8`: the gradient
  without its 8 zero padding channels, [S,400,8]; `planes`: as four parity planes of the 10 x 10 space-to-depth grid,
  [S,4,100,8] (pc_planes_conv / pc_planes_wgrad).  A [16] bias with [4,64,32] taps selects the 16-channel head (8..15
  actions): dy16 [S,400,16] with every channel real and db [16]; it has no c8 or planes layout."""
  s = h16.numel() // 2592
  loss = torch.zeros(1, dtype=torch.float64, device=h16.device)
  if _pc16(w_dtaps, bias8):
    if c8 or planes:
      raise _lib.UnrealError("the 16-channel pixel-control head writes its loss gradient in conv2's [S,400,16] layout only")
    dy16 = torch.empty(s, 400, 16, dtype=torch.bfloat16, device=h16.device)
    db16 = torch.zeros(16, dtype=torch.float32, device=h16.device)
    call("unreal_pc_deconv_loss16", ptr(h16, torch.bfloat16, "h16"), ptr(w_dtaps, torch.bfloat16, "w_dtaps"),
         ptr(bias8, torch.float32, "bias16"), ptr(act, torch.int32, "act"), ptr(target, torch.float32, "target"),
         ptr(mask, torch.float32, "mask"), int(num_actions), float(lam), s, ptr(loss), ptr(dy16), ptr(db16), stream_ptr())
    return loss, dy16, db16
  if planes:
    dy16 = torch.empty(s, 4, 100, 8, dtype=torch.bfloat16, device=h16.device)
  else:
    dy16 = torch.empty(s, 400, 8 if c8 else 16, dtype=torch.bfloat16, device=h16.device)
  db8 = torch.zeros(8, dtype=torch.float32, device=h16.device)
  call("unreal_pc_deconv_loss_planes" if planes else "unreal_pc_deconv_loss_c8" if c8 else "unreal_pc_deconv_loss", ptr(h16, torch.bfloat16, "h16"), ptr(w_dtaps, torch.bfloat16, "w_dtaps"),
       ptr(bias8, torch.float32, "bias8"), ptr(act, torch.int32, "act"), ptr(target, torch.float32, "target"),
       ptr(mask, torch.float32, "mask"), int(num_actions), float(lam), s, ptr(loss), ptr(dy16), ptr(db8), stream_ptr())
  return loss, dy16, db8


def pc_w_planes(w8):
  """The merged deconv filter [4,4,8,32] bf16 (HWIO) -> the resident B tiles of pc_planes_conv: [4 taps (by,bx)][2 dy][2 dx]
  [32 o][8 c] = W8[2by+dy, 2bx+dx, c, o]."""
  return w8.reshape(2, 2, 2, 2, 8, 32).permute(0, 2, 1, 3, 5, 4).reshape(4, 2, 2, 32, 8).contiguous()


def pc_planes_from_dense(dy8):
  """[S,20,20,8] -> the plane-major layout [S,4,100,8] (tests / tools; the agent's gradient is written that way)."""
  s = dy8.shape[0]
  return dy8.reshape(s, 10, 2, 10, 2, 8).permute(0, 2, 4, 1, 3, 5).reshape(s, 4, 100, 8).contiguous()


def pc_planes_conv(dyp, w_planes, mask_y, scale=None, out=None, want_db=True):
  """The pixel-control head's backward convolution on the plane-major gradient: dyp bf16 [S,4,100,8] -> (d pc_fc1 output
  bf16 [S,9,9,32], masked by mask_y > 0 and scaled by the device scalar `scale`; db f32 [2592])."""
  s = dyp.shape[0]
  if tuple(dyp.shape[1:]) != (4, 100, 8) or mask_y.numel() != s * 2592 or w_planes.numel() != 4096:
    raise ValueError("pc_planes_conv: dyp [S,4,100,8], mask_y S*2592 elements, w_planes = pc_w_planes(W8)")
  if out is None:
    out = torch.empty(s, 9, 9, 32, dtype=torch.bfloat16, device=dyp.device)
  db = torch.zeros(2592, dtype=torch.float32, device=dyp.device) if want_db else None
  call("unreal_pc_planes_conv", ptr(dyp, torch.bfloat16, "dyp"), ptr(w_planes, torch.bfloat16, "w_planes"),
       ptr(scale, torch.float32, "scale"), ptr(mask_y, torch.bfloat16, "mask_y"), ptr(out, torch.bfloat16, "out"),
       ptr(db, torch.float32, "db"), s, stream_ptr())
  return out, db


def pc_planes_wgrad(dyp, hp):
  """dyp bf16 [S,4,100,8], hp bf16 (S*2592 elements, pc_fc1's output) -> the merged deconv filter's gradient [4,4,8,32] f32."""
  s = dyp.shape[0]
  if tuple(dyp.shape[1:]) != (4, 100, 8) or hp.numel() != s * 2592:
    raise ValueError("pc_planes_wgrad: dyp [S,4,100,8], hp S*2592 elements")
  acc = torch.zeros(4, 4, 8, 32, dtype=torch.float32, device=dyp.device)
  call("unreal_pc_planes_wgrad", ptr(dyp, torch.bfloat16, "dyp"), ptr(hp, torch.bfloat16, "hp"), ptr(acc, torch.float32), s,
       stream_ptr())
  return acc


def a3c_head(h, wp, bp, wv, bv, act=None, adv=None, ret=None, mask=None, entropy_beta=0.0, value_coef=0.25,
             want_pi=False, want_v=False, want_sums=False, want_grads=False, v_out=None):
  """Policy / value heads (+ A3C losses) over h [M,256] f32 in one pass.  Returns a dict with the requested
  pi [M,A], v [M], sums f64 [3] (policy, value, entropy), dz [M,A], dv [M]."""
  m = h.shape[0]
  a = 0 if wp is None else wp.shape[1]
  d = h.device
  out = {}
  if want_pi:
    out["pi"] = torch.empty(m, a, dtype=torch.float32, device=d)
  if want_v:     # v_out: a caller-owned [M] buffer (the rollout's value history row) instead of a fresh tensor + a copy
    out["v"] = torch.empty(m, dtype=torch.float32, device=d) if v_out is None else v_out
  if want_sums:
    out["sums"] = torch.zeros(3, dtype=torch.float64, device=d)
  if want_grads:
    if act is not None:
      out["dz"] = torch.empty(m, a, dtype=torch.float32, device=d)
    if ret is not None:
      out["dv"] = torch.empty(m, dtype=torch.float32, device=d)
  call("unreal_a3c_head_loss", ptr(h, torch.float32, "h"), ptr(wp, torch.float32, "wp"), ptr(bp, torch.float32, "bp"),
       ptr(wv, torch.float32, "wv"), ptr(bv, torch.float32, "bv"), ptr(act, torch.int32, "act"),
       ptr(adv, torch.float32, "adv"), ptr(ret, torch.float32, "ret"), ptr(mask, torch.float32, "mask"), m, a,
       float(entropy_beta), float(value_coef), ptr(out.get("pi")), ptr(out.get("v")), ptr(out.get("sums")),
       ptr(out.get("dz")), ptr(out.get("dv")), stream_ptr())
  return out


def a3c_head_bwd(h, wp, wv, dz, dv, go2):
  """-> dh [M,256], dwp [256,A] or None, dbp [A] or None, dwv [256], dbv [1] (fp32)."""
  m = h.shape[0]
  a = 0 if wp is None else wp.shape[1]
  d = h.device
  dh = torch.empty(m, 256, dtype=torch.float32, device=d)
  dwp = torch.zeros(256, a, dtype=torch.float32, device=d) if dz is not None else None
  dbp = torch.zeros(a, dtype=torch.float32, device=d) if dz is not None else None
  dwv = torch.zeros(256, dtype=torch.float32, device=d) if dv is not None else None
  dbv = torch.zeros(1, dtype=torch.float32, device=d) if dv is not None else None
  call("unreal_a3c_head_bwd", ptr(h, torch.float32, "h"), ptr(wp, torch.float32, "wp"), ptr(wv, torch.float32, "wv"),
       ptr(dz, torch.float32, "dz"), ptr(dv, torch.float32, "dv"), ptr(go2, torch.float32, "go2"), m, a, ptr(dh), ptr(dwp),
       ptr(dbp), ptr(dwv), ptr(dbv), stream_ptr())
  return dh, dwp, dbp, dwv, dbv


def cell_gather(table16, pos, out=None):
  """table16 bf16 [49, D], pos i32 [S,2] (agent cells) -> out bf16 [S, D] = table rows of the cells.  `out` may be a
  column slice of a wider row-major buffer (rows out.stride(0) elements apart)."""
  s = pos.shape[0]
  d = table16.shape[1]
  if out is None:
    out = torch.empty(s, d, dtype=torch.bfloat16, device=table16.device)
  if out.dim() != 2 or out.shape[0] != s or out.shape[1] != d or out.stride(1) != 1 or out.dtype != torch.bfloat16:
    raise _lib.UnrealError("cell_gather: out must be bf16 [S, D] with contiguous rows")
  call("unreal_cell_gather", ptr(table16, torch.bfloat16, "table"), ptr(pos, torch.int32, "pos"), out.data_ptr(),
       int(out.stride(0)), s, d, stream_ptr())
  return out


def cell_segment_sum(dy, pos, out=None):
  """dy f32 / bf16 [S,256], pos i32 [S,2] -> f32 [49,256]: rows summed by agent cell (accumulated into `out`)."""
  s = dy.shape[0]
  if out is None:
    out = torch.zeros(49, 256, dtype=torch.float32, device=dy.device)
  call("unreal_cell_segment_sum", ptr(dy, None, "dy"), _lib.dtype_tag(dy), ptr(pos, torch.int32, "pos"),
       ptr(out, torch.float32, "out"), s, dy.shape[1], stream_ptr())
  return out


def rp_loss(logits8, bias, c=None, want_p=False, want_loss=False, want_grad=False, go=None):
  """Reward-prediction softmax / cross-entropy on logits8 [N,8] f32 (columns 0..2; bias [3] added inside):
  -> dict(p [N,3], loss f64 [1], dz16 bf16 [N,8], db [3]) with the requested entries."""
  n = logits8.shape[0]
  d = logits8.device
  out = {}
  if want_p:
    out["p"] = torch.empty(n, 3, dtype=torch.float32, device=d)
  if want_loss:
    out["loss"] = torch.zeros(1, dtype=torch.float64, device=d)
  if want_grad:
    out["dz16"] = torch.empty(n, 8, dtype=torch.bfloat16, device=d)
    out["db"] = torch.zeros(3, dtype=torch.float32, device=d)
  call("unreal_rp_loss", ptr(logits8, torch.float32, "logits8"), ptr(bias, torch.float32, "bias"), ptr(c, torch.float32, "c"),
       n, ptr(out.get("p")), ptr(out.get("loss")), ptr(out.get("dz16")), ptr(out.get("db")), ptr(go, torch.float32, "go"),
       stream_ptr())
  return out


def rollout_lar(last_action, last_reward, num_actions, objective=None, out=None):
  """one-hot(last_action) ++ [last_reward] (++ objective) for every env -> [N, A+1+G] f32."""
  n = last_action.shape[0]
  g = 0 if objective is None else objective.shape[1]
  if out is None:
    out = torch.empty(n, num_actions + 1 + g, dtype=torch.float32, device=last_action.device)
  call("unreal_rollout_lar", ptr(last_action, torch.int32, "last_action"), ptr(last_reward, torch.float32, "last_reward"),
       ptr(objective, torch.float32, "objective"), n, int(num_actions), g, ptr(out, torch.float32, "lar"), stream_ptr())
  return out


def rollout_post(reward, terminal, frame_rec, active, ended, last_rec, episode_reward, lstm_c, lstm_h, stats):
  """The bookkeeping after one env step of the rollout window, in place (see include/unreal_b200.h)."""
  call("unreal_rollout_post", ptr(reward, torch.float32, "reward"), ptr(terminal, torch.uint8, "terminal"),
       ptr(frame_rec, torch.int64, "frame_rec"), reward.shape[0], ptr(active, torch.uint8, "active"),
       ptr(ended, torch.uint8, "ended"), ptr(last_rec, torch.int64, "last_rec"),
       ptr(episode_reward, torch.float32, "episode_reward"), ptr(lstm_c, torch.float32, "lstm_c"),
       ptr(lstm_h, torch.float32, "lstm_h"), ptr(stats, torch.float64, "stats"), stream_ptr())


def maze_eval_act(pi, greedy, streams, state, ep, res, lstm_c, lstm_h, fc_tab, xh, kx, max_steps):
  """One evaluation step after the policy, in place (unreal_maze_eval_act, include/unreal_b200.h): pi f32 [N,A];
  streams: MtStreams (None when greedy); state: MazeState; ep: dict(score f32, length i32, index i32, active u8) [N];
  res: dict(score f32, length i32, finished u8) [N,E]; lstm_c / lstm_h f32 [N,256]; fc_tab bf16 [49,256]; xh bf16
  [N, >= kx + 256] with contiguous rows."""
  n, a = pi.shape
  e = res["score"].shape[1]
  for k, t in res.items():
    if tuple(t.shape) != (n, e):
      raise _lib.UnrealError("maze_eval_act: result %s must be [%d,%d]" % (k, n, e))
  for k, t in ep.items():
    if t.numel() != n:
      raise _lib.UnrealError("maze_eval_act: %s must hold %d entries" % (k, n))
  if state.n != n or tuple(lstm_c.shape) != (n, 256) or tuple(lstm_h.shape) != (n, 256) or tuple(fc_tab.shape) != (49, 256):
    raise _lib.UnrealError("maze_eval_act: maze state [%d], LSTM state [%d,256] and table [49,256] expected" % (n, n))
  xp, ld = _rows2d(xh, xh.shape[1], torch.bfloat16, "xh")
  if xh.shape[0] != n:
    raise _lib.UnrealError("maze_eval_act: xh must have %d rows" % n)
  if streams is None and not greedy:
    raise _lib.UnrealError("maze_eval_act: sampling needs the MT19937 streams")
  call("unreal_maze_eval_act", ptr(pi, torch.float32, "pi"), int(a), 1 if greedy else 0,
       None if streams is None else ptr(streams.mt), None if streams is None else ptr(streams.pos),
       ptr(state.pos, torch.int32), ptr(state.last_action, torch.int32), ptr(state.last_reward, torch.float32),
       ptr(ep["score"], torch.float32, "score"), ptr(ep["length"], torch.int32, "length"),
       ptr(ep["index"], torch.int32, "index"), ptr(ep["active"], torch.uint8, "active"),
       ptr(res["score"], torch.float32, "res score"), ptr(res["length"], torch.int32, "res length"),
       ptr(res["finished"], torch.uint8, "res finished"), int(e), int(max_steps), ptr(lstm_c, torch.float32, "lstm_c"),
       ptr(lstm_h, torch.float32, "lstm_h"), ptr(fc_tab, torch.bfloat16, "fc_tab"), xp, ld, int(kx), n, stream_ptr())


def lstm_cell_act_heads(gates, c_state, h_state, wp, bp, wv, bv, active=None, v_out=None):
  """Acting step of the cell + the policy / value heads in one launch: gates bf16 [N,1024], state f32 [N,256] in place for
  the active envs; wp [256,A], bp [A], wv [256], bv [1] f32 -> (pi f32 [N,A], v f32 [N]; v_out: a caller-owned [N] row)."""
  n, a = gates.shape[0], wp.shape[1]
  pi = torch.empty(n, a, dtype=torch.float32, device=gates.device)
  v = torch.empty(n, dtype=torch.float32, device=gates.device) if v_out is None else v_out
  call("unreal_lstm_cell_act_heads", ptr(gates, torch.bfloat16, "gates"), ptr(c_state, torch.float32, "c_state"),
       ptr(h_state, torch.float32, "h_state"), ptr(active, torch.uint8, "active"), n, ptr(wp, torch.float32, "wp"),
       ptr(bp, torch.float32, "bp"), ptr(wv, torch.float32, "wv"), ptr(bv, torch.float32, "bv"), a, ptr(pi, torch.float32),
       ptr(v, torch.float32, "v_out"), stream_ptr())
  return pi, v


def lstm_cell_act(gates, c_state, h_state, h_out=None, active=None):
  """Acting step of the cell, in place on the persistent state of the active envs; h_out receives the state's h."""
  n = gates.shape[0]
  if gates.dtype == torch.bfloat16:
    call("unreal_lstm_cell_act_g16", ptr(gates, torch.bfloat16, "gates"), ptr(c_state, torch.float32, "c_state"),
         ptr(h_state, torch.float32, "h_state"), ptr(h_out, torch.float32, "h_out"), ptr(active, torch.uint8, "active"), n,
         stream_ptr())
    return h_out
  call("unreal_lstm_cell_act", ptr(gates, torch.float32, "gates"), ptr(c_state, torch.float32, "c_state"),
       ptr(h_state, torch.float32, "h_state"), ptr(h_out, torch.float32, "h_out"), ptr(active, torch.uint8, "active"), n,
       stream_ptr())
  return h_out
