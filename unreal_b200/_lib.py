"""ctypes binding of libunreal_b200.so (the C ABI declared in include/unreal_b200.h).

There is no CPU fallback: if the shared library has not been built, importing this module
raises, and every call that fails on the device raises ``UnrealError`` with the library's
message.  ctypes releases the GIL for the duration of each call.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_uint8, c_uint32, c_void_p

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libunreal_b200.so")

OK = 0
F32 = 0
U8 = 1


class UnrealError(RuntimeError):
  pass


if not os.path.exists(LIB_PATH):
  raise ImportError(
      "%s is missing: build it with `python -m unreal_b200.build` (nvcc, sm_100a). "
      "unreal_b200 has no CPU fallback." % LIB_PATH)

lib = ctypes.CDLL(LIB_PATH)

P = c_void_p  # device pointers travel as void*

# name -> (restype, argtypes); mirrors include/unreal_b200.h one to one
SIGNATURES = {
    "unreal_last_error": (c_char_p, []),
    "unreal_abi_version": (c_int, []),
    "unreal_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "unreal_set_tunable": (c_int, [c_char_p, c_int]),
    "unreal_get_tunable": (c_int, [c_char_p, POINTER(c_int)]),
    "unreal_maze_set_map": (c_int, [c_char_p]),
    "unreal_maze_get_layout": (c_int, [POINTER(c_int)] * 4 + [POINTER(c_uint8)]),
    "unreal_maze_reset": (c_int, [P, P, P, P, c_int, P]),
    "unreal_maze_step": (c_int, [P, P, P, P, P, P, P, P, c_int, P, P, c_int, c_int, P]),
    "unreal_maze_window": (c_int, [P, P, P, P, P, P, P, c_int, P, P, c_int, c_int, c_int, P]),
    "unreal_maze_render": (c_int, [P, P, c_int, c_int, P]),
    "unreal_maze_pixel_change": (c_int, [P, P, P, c_int, P]),
    "unreal_maze_pc_targets": (c_int, [P, P, P, P, c_float, P, c_int, c_int, P]),
    "unreal_maze_rollout_targets": (c_int, [P, P, P, P, c_float, c_float, P, P, P, c_int, c_int, P]),
    "unreal_pixel_change": (c_int, [P, P, c_int, P, c_int, c_int, c_int, c_int, P]),
    "unreal_pixel_change_stream": (c_int, [P, c_int, P, c_int, c_int, c_int, c_int, c_int, P]),
    "unreal_selfcheck_arith": (c_int, [P, P]),
    "unreal_subsample": (c_int, [P, P, c_int, c_int, c_int, c_int, P]),
    "unreal_nstep_returns": (c_int, [P, P, P, P, c_float, P, P, c_int, c_int, P]),
    "unreal_sequence_returns": (c_int, [P, P, P, c_float, P, c_int, c_int, P]),
    "unreal_pc_targets": (c_int, [P, P, P, P, c_float, P, c_int, c_int, P]),
    "unreal_mt_seed": (c_int, [P, P, P, c_int, P]),
    "unreal_choose_action": (c_int, [P, P, P, P, P, c_int, c_int, P]),
    "unreal_mt_randint": (c_int, [P, P, c_uint32, P, c_int, c_int, P]),
    "unreal_replay_create": (c_int, [POINTER(c_void_p), c_int, c_int]),
    "unreal_replay_destroy": (c_int, [c_void_p]),
    "unreal_replay_reset": (c_int, [c_void_p, P]),
    "unreal_replay_add": (c_int, [c_void_p, P, P]),
    "unreal_replay_state": (c_int, [c_void_p, P, P, P, P, P, P]),
    "unreal_replay_copy": (c_int, [c_void_p, c_int, P, P, P, P, P, P]),
    "unreal_replay_sample_sequence": (c_int, [c_void_p, P, P, c_int, P, P, P, P]),
    "unreal_replay_sample_rp": (c_int, [c_void_p, P, P, P, P, P]),
    "unreal_frame_unpack": (c_int, [P, c_int, P, P, P, P, P, P, P, P, P]),
    "unreal_frame_pack": (c_int, [P, P, P, P, P, P, P, c_int, P]),
    "unreal_replay_add_slots": (c_int, [c_void_p, P, P, P]),
    "unreal_ring_store": (c_int, [P, P, P, c_int, c_int, c_int64, P]),
    "unreal_rows_select": (c_int, [P, P, P, P, c_int, c_int64, P]),
    "unreal_replay_gather": (c_int, [c_void_p, P, c_int64, P, P, c_int, c_int, P, P]),
    "unreal_host_frames_ingest": (c_int, [c_int, P, P, c_int, P, P, P, P, P, P, P, P, c_int, P, P, P, P, P, P, P,
                                          c_int, c_int, c_int, c_int, c_int, P]),
    "unreal_rollout_lar": (c_int, [P, P, P, c_int, c_int, c_int, P, P]),
    "unreal_rollout_post": (c_int, [P, P, P, c_int, P, P, P, P, P, P, P, P]),
    "unreal_maze_eval_act": (c_int, [P, c_int, c_int, P, P, P, P, P, P, P, P, P, P, P, P, c_int, c_int, P, P, P, P, c_int64,
                                     c_int, c_int, P]),
    "unreal_grad_sumsq": (c_int, [P, c_int64, P, P]),
    "unreal_rmsprop_update": (c_int, [P, P, P, P, c_int64, P, c_float, c_float, c_float, c_float, c_float,
                                      c_float, P, P]),
    "unreal_rmsprop_update_dlr": (c_int, [P, P, P, P, c_int64, P, c_float, P, c_float, c_float, c_float,
                                          c_float, P, P]),
    "unreal_gemm_bf16": (c_int, [P, c_int64, c_int, P, c_int64, c_int, P, c_int64, c_int, P, P, c_int, c_int, c_int,
                                 c_int, c_int, c_int, P]),
    "unreal_im2col": (c_int, [P, c_int, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "unreal_col2im": (c_int, [P, c_int, P, c_int, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "unreal_lstm_cell_fwd": (c_int, [P, P, P, P, P, c_int, P]),
    "unreal_lstm_cell_fwd_ld": (c_int, [P, P, P, P, P, c_int, c_int, P]),
    "unreal_lstm_cell_act": (c_int, [P, P, P, P, P, c_int, P]),
    "unreal_lstm_cell_fwd_g16": (c_int, [P, P, P, P, P, c_int, c_int, P]),
    "unreal_lstm_cell_act_g16": (c_int, [P, P, P, P, P, c_int, P]),
    "unreal_lstm_cell_act_heads": (c_int, [P, P, P, P, c_int, P, P, P, P, c_int, P, P, P]),
    "unreal_lstm_cell_bwd_g16": (c_int, [P, P, P, P, P, P, P, c_int, P]),
    "unreal_lstm_step_fwd": (c_int, [P, c_int64, P, P, P, P, P, P, P, c_int, P, P, c_int, c_int, c_int, P]),
    "unreal_lstm_step_bwd": (c_int, [P, P, c_int64, P, P, P, P, P, P, P, c_int, c_int, P]),
    "unreal_lstm_cell_bwd": (c_int, [P, P, P, P, P, P, c_int, P]),
    "unreal_lstm_cell_bwd2": (c_int, [P, P, P, P, P, P, P, c_int, P]),
    "unreal_s2d_frames": (c_int, [P, c_int, P, c_int, P]),
    "unreal_conv_fwd": (c_int, [P, c_int, P, P, P, c_int, P]),
    "unreal_relu_grad": (c_int, [P, c_int, P, P, P, c_int64, c_int, c_int, P]),
    "unreal_conv1_wgrad": (c_int, [P, P, P, c_int, P]),
    "unreal_conv2_wgrad": (c_int, [P, P, P, c_int, P]),
    "unreal_conv2_wgrad_c8": (c_int, [P, P, P, c_int, P]),
    "unreal_conv2_dgrad": (c_int, [P, P, P, c_int, P]),
    "unreal_pc_deconv_fwd": (c_int, [P, P, P, P, c_int, P]),
    "unreal_conv2_dgrad_relu": (c_int, [P, P, P, P, P, c_int, c_int, P]),
    "unreal_conv1_wgrad_p21": (c_int, [P, P, P, c_int, P]),
    "unreal_conv1_fwd_maze": (c_int, [P, P, P, P, c_int, P]),
    "unreal_conv1_wgrad_maze": (c_int, [P, P, P, c_int, P]),
    "unreal_s2d_frames_split": (c_int, [P, c_int, P, P, c_int, P]),
    "unreal_conv1_fwd_split": (c_int, [P, P, P, P, P, P, P, c_int, P]),
    "unreal_conv1_fwd_maze_split": (c_int, [P, P, P, P, P, P, c_int, P]),
    "unreal_conv2_fwd_split": (c_int, [P, P, P, P, P, P, c_int, P]),
    "unreal_a3c_head_loss": (c_int, [P, P, P, P, P, P, P, P, P, c_int64, c_int, c_float, c_float, P, P, P, P, P, P]),
    "unreal_a3c_head_bwd": (c_int, [P, P, P, P, P, P, c_int64, c_int, P, P, P, P, P, P]),
    "unreal_pc_loss": (c_int, [P, P, P, P, c_int, c_float, c_int64, c_int, P, P, P, P]),
    "unreal_pc_loss_grad16": (c_int, [P, P, P, P, c_int, c_float, c_int64, c_int, P, P, P, P]),
    "unreal_cell_gather": (c_int, [P, P, P, c_int64, c_int64, c_int, P]),
    "unreal_cell_segment_sum": (c_int, [P, c_int, P, P, c_int64, c_int, P]),
    "unreal_pc_deconv_loss": (c_int, [P, P, P, P, P, P, c_int, c_float, c_int, P, P, P, P]),
    "unreal_pc_deconv_loss_c8": (c_int, [P, P, P, P, P, P, c_int, c_float, c_int, P, P, P, P]),
    "unreal_pc_deconv_loss_planes": (c_int, [P, P, P, P, P, P, c_int, c_float, c_int, P, P, P, P]),
    "unreal_pc_planes_conv": (c_int, [P, P, P, P, P, P, c_int, P]),
    "unreal_pc_planes_wgrad": (c_int, [P, P, P, c_int, P]),
    "unreal_pc_deconv_qmax": (c_int, [P, P, P, c_int, c_int, P, P]),
    "unreal_pc_deconv_loss16": (c_int, [P, P, P, P, P, P, c_int, c_float, c_int, P, P, P, P]),
    "unreal_pc_deconv_qmax16": (c_int, [P, P, P, c_int, c_int, P, P]),
    "unreal_conv2_fwd_linear_scaled": (c_int, [P, P, P, P, c_int, P]),
    "unreal_conv2_fwd_linear_masked": (c_int, [P, c_int, P, P, P, P, P, c_int, P]),
    "unreal_rp_loss": (c_int, [P, P, P, c_int64, P, P, P, P, P, P]),
    "unreal_conv2_fwd_linear": (c_int, [P, P, P, c_int, P]),
}

MISSING = []
for _name, (_res, _args) in SIGNATURES.items():
  try:
    _fn = getattr(lib, _name)
  except AttributeError:
    MISSING.append(_name)
    continue
  _fn.restype = _res
  _fn.argtypes = _args


def last_error():
  return lib.unreal_last_error().decode("utf-8", "replace")


def check(rc, what=""):
  if rc != OK:
    raise UnrealError("%s failed (%d): %s" % (what or "libunreal_b200 call", rc, last_error()))


def call(name, *args):
  check(getattr(lib, name)(*args), name)


def require_device():
  """Raises unless a CUDA device of compute capability 10.x is current."""
  if not torch.cuda.is_available():
    raise UnrealError("unreal_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
  sm, maj, mnr = c_int(), c_int(), c_int()
  check(lib.unreal_device_info(ctypes.byref(sm), ctypes.byref(maj), ctypes.byref(mnr)), "unreal_device_info")
  return sm.value, maj.value, mnr.value


BF16 = 2
_DTYPE_TAG = {torch.float32: F32, torch.uint8: U8, torch.bfloat16: BF16}


def dtype_tag(t):
  try:
    return _DTYPE_TAG[t.dtype]
  except KeyError:
    raise UnrealError("unsupported frame dtype %s (float32 or uint8)" % t.dtype)


def ptr(t, dtype=None, name="tensor"):
  """data_ptr of a contiguous CUDA tensor (None -> NULL), with dtype check."""
  if t is None:
    return None
  if not isinstance(t, torch.Tensor) or not t.is_cuda:
    raise UnrealError("%s must be a CUDA tensor" % name)
  if not t.is_contiguous():
    raise UnrealError("%s must be contiguous" % name)
  if dtype is not None and t.dtype != dtype:
    raise UnrealError("%s must be %s, got %s" % (name, dtype, t.dtype))
  return t.data_ptr()


def host_ptr(t, dtype, name="tensor"):
  """data_ptr of a contiguous pinned host tensor (None -> NULL), with dtype check."""
  if t is None:
    return None
  if not isinstance(t, torch.Tensor) or t.is_cuda or not t.is_pinned():
    raise UnrealError("%s must be a pinned host tensor" % name)
  if not t.is_contiguous():
    raise UnrealError("%s must be contiguous" % name)
  if t.dtype != dtype:
    raise UnrealError("%s must be %s, got %s" % (name, dtype, t.dtype))
  return t.data_ptr()


def stream_ptr(stream=None):
  s = stream if stream is not None else torch.cuda.current_stream()
  return s.cuda_stream


def set_tunable(name, value):
  call("unreal_set_tunable", name.encode(), int(value))


import contextlib
import gc


@contextlib.contextmanager
def graph_capture(graph):
  """`torch.cuda.graph(graph)` with Python's cyclic garbage collector held off for the duration of the capture.
  A collection that runs mid-capture can finalise objects of earlier work whose destructors call cudaFree /
  cudaGraphExecDestroy (library-owned replay rings, old CUDA graphs): a prohibited call during a global-mode
  stream capture, which invalidates it (cudaErrorStreamCaptureInvalidated) -- at a random allocation, i.e. flaky.
  Collect first, then keep the collector off until the capture has ended."""
  gc.collect()
  was_enabled = gc.isenabled()
  gc.disable()
  # with a process group alive, NCCL's watchdog thread polls CUDA events while we capture: in the default global mode
  # any such call from another thread can invalidate (or, with collectives inside the capture, stall) it; thread-local
  # mode scopes the capture's restrictions to this thread
  import torch.distributed as dist
  mode = "thread_local" if (dist.is_available() and dist.is_initialized()) else "global"
  try:
    with torch.cuda.graph(graph, capture_error_mode=mode):
      yield
  finally:
    if was_enabled:
      gc.enable()


# A/B switches for the benchmark scripts without editing them: UNREAL_TUNABLES="name=value,name=value"
for _kv in filter(None, os.environ.get("UNREAL_TUNABLES", "").split(",")):
  _k, _, _v = _kv.partition("=")
  set_tunable(_k.strip(), int(_v))
