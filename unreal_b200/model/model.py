"""UnrealModel: drop-in for model/model.py (vanilla path, segnet_mode == 0), batched over N envs.

Same constructor arguments and `run_*` helper surface as the reference (model.py:46-64, :625-728)
with one documented deviation: there is no TensorFlow session, so the `sess` argument is accepted and
ignored, inputs/outputs are torch CUDA tensors with a leading env axis, and `prepare_loss()` +
the applier's `minimize_local` are replaced by the eager `update(feed, learning_rate, applier)`.

Parameters live in ONE flat fp32 buffer in the reference's variable creation order (20 variables
with all heads, model_test.py:8-20; TF layouts: [in,out] matmul kernels, HWIO conv filters,
[kh,kw,out,in] deconv filters, one BasicLSTMCell kernel [(256+A+1+G)+256, 1024] with gates
i, j, f, o) so that K6 updates them in one launch; a bf16 shadow of the same buffer feeds the
tcgen05 GEMMs (K7).  Each variable starts on an 8-element boundary so the shadow views satisfy
TMA's 16-byte alignment.

The training graph follows model.py:137-598: the base tower unrolls the LSTM over the rollout from
the fed start state; the PC and VR towers unroll from a zero state (:393, :459); RP concatenates
three frames' conv features (:473-488); losses :490-598.  In the reference the batch axis of the
training placeholders is TIME for one env; here tensors are [T, N, ...] and every env is one such
unroll, `mask[t, n]` marking the steps that exist.  total loss = sum over envs (each env is one
reference worker), scaled by `grad_scale` (default 1/N: the synchronous mean of N workers).
"""
from collections import OrderedDict

import numpy as np
import torch

from .. import _lib
from .. import kernels as K
from .layers import (A3CHeadLossFn, CellGatherFn, FlatViewsFn, ConvFn, Deconv8Fn, EncoderFn, LinearFn, LstmFn, PcFusedHeadLossFn, PcHeadLossFn, PcLossFn, PcTowerFusedFn, RpCellLossFn,
                     RpHeadLossFn, split_k_for)


def _variable_specs(A, G, use_pc, use_rp):
  lstm_in = 256 + A + 1 + G
  specs = [
      ("W_base_conv1", (8, 8, 3, 16), 8 * 8 * 3), ("b_base_conv1", (16,), 8 * 8 * 3),
      ("W_base_conv2", (4, 4, 16, 32), 4 * 4 * 16), ("b_base_conv2", (32,), 4 * 4 * 16),
      ("W_base_fc1", (2592, 256), 2592), ("b_base_fc1", (256,), 2592),
      ("lstm_kernel", (lstm_in + 256, 1024), None), ("lstm_bias", (1024,), None),
      ("W_base_fc_p", (256, A), 256), ("b_base_fc_p", (A,), 256),
      ("W_base_fc_v", (256, 1), 256), ("b_base_fc_v", (1,), 256),
  ]
  if use_pc:
    specs += [("W_pc_fc1", (256, 2592), 256), ("b_pc_fc1", (2592,), 256),
              ("W_pc_deconv_v", (4, 4, 1, 32), 4 * 4 * 32), ("b_pc_deconv_v", (1,), 4 * 4 * 32),
              ("W_pc_deconv_a", (4, 4, A, 32), 4 * 4 * 32), ("b_pc_deconv_a", (A,), 4 * 4 * 32)]
  if use_rp:
    specs += [("W_rp_fc1", (7776, 3), 7776), ("b_rp_fc1", (3,), 7776)]
  return specs


class UnrealModel(object):
  def __init__(self, action_size, objective_size, thread_index, use_lstm, use_pixel_change, use_value_replay,
               use_reward_prediction, pixel_change_lambda, entropy_beta, device, segnet_param_dict=None,
               image_shape=(84, 84), is_training=True, n_classes=0, segnet_lambda=0.0, dropout=0.0,
               for_display=False, num_envs=1, seed=0, encoder_precision='bf16'):
    _lib.require_device()
    if encoder_precision not in ('bf16', 'bf16x3'):
      raise _lib.UnrealError("encoder_precision must be 'bf16' or 'bf16x3', got %r" % (encoder_precision,))
    # 'bf16x3': conv1 and conv2 forward on split-bf16 operands (fp32-grade products, the reference's arithmetic); fixed at
    # construction because the filter shadows it needs are built by refresh_shadow and captured by CUDA graphs
    self._encoder_precision = encoder_precision
    segnet_param_dict = segnet_param_dict or {'segnet_mode': 0}
    if segnet_param_dict.get('segnet_mode', 0) != 0:
      raise _lib.UnrealError("segnet_mode != 0 (ErfNet encoder/decoder) is outside the B200 hot path")
    if not use_lstm:
      raise _lib.UnrealError("only the LSTM agent (use_lstm=True, the reference default) is on the B200 hot path")
    if tuple(image_shape) != (84, 84):
      raise _lib.UnrealError("the network is hard-wired to 84x84 frames (model.py:554, 9x9x32 flatten)")
    self._device = torch.device(device if str(device).startswith("cuda") else "cuda:0")
    self._action_size = A = int(action_size)
    self._objective_size = G = int(objective_size)
    self._thread_index = thread_index
    self._use_lstm = use_lstm
    self._use_pixel_change = use_pixel_change
    if use_pixel_change and A > 15:
      raise _lib.UnrealError("pixel control supports up to 15 actions (a 16-channel head: the value and 15 advantages), "
                             "got %d" % A)
    self._use_value_replay = use_value_replay
    self._use_reward_prediction = use_reward_prediction
    self._pixel_change_lambda = float(pixel_change_lambda)
    self._entropy_beta = float(entropy_beta)
    self.segnet_mode = 0
    self.is_training = is_training
    self.for_display = for_display
    self.num_envs = int(num_envs)
    self.lstm_in = 256 + A + 1 + G
    self.kx = (self.lstm_in + 7) // 8 * 8
    self.fused_conv = True    # False: convolutions as explicit im2col + GEMM (A/B switch for benchmarks)
    self.fused_encoder = True # False: conv1 / conv2 as separate autograd nodes (dense gradient + relu_grad pass between them)
    self.fused_heads = True   # False: policy / value heads and their losses as torch ops
    # maze CELL observations (int32 [.,2]): a frame is a pure function of the agent cell, so conv1 -> conv2 -> fc1 of every
    # sample is a row of a 49-entry table computed once per update (and once per rollout for acting), and the encoder's
    # backward pass is a segment sum by cell + a 49-sample backward.  False: the dense render-fused encoder on all samples.
    self.dedup_cells = True
    # update(): the total loss is the SUM over envs (each env is one reference worker); its gradient is scaled by
    # grad_scale before the clip -- None = 1/N, the synchronous mean of N workers; 1.0 = the sum, i.e. N workers each
    # applying its own gradient (the reference's Hogwild, to first order in the step size)
    self.grad_scale = None
    # LSTM gate pre-activations / saved activations as bf16 (False: f32).  The cell kernels are HBM-bound on that buffer.
    self.lstm_gates_bf16 = True
    # one launch per LSTM step of the unroll (needs lstm_gates_bf16): the cell in the step GEMM's epilogue, the cell's
    # backward pass in the epilogue of the recurrent dh GEMM (csrc/lstm_tcgen05.cu), for batches of at least
    # fused_lstm_min_rows env rows (measured per step, profiles/r2_lstm_step_bench.jsonl: forward 20.1 us against 31.0 us
    # for GEMM + cell kernel at 8192 rows and 12.6 / 15.2 at 2048, but 12.4 / 11.6 at 1024 where one tile's latency is
    # the whole launch).  The acting step keeps GEMM + cell kernel: its state is row-major and updated under a mask.
    self.fused_lstm_step = True
    self.fused_lstm_min_rows = 2048
    # pixel-control loss inside the deconv kernel's epilogue (False: deconv -> f32 head output -> separate loss / gradient passes)
    self.fused_pc_loss = True
    # pc_fc1's ReLU / bias gradient in the epilogue of the pixel-control head's backward convolution (PcTowerFusedFn; False:
    # a unreal_relu_grad pass over the dense [S,2592] gradient between the two autograd nodes)
    self.fused_pc_relu = True
    # acting step: the policy / value heads inside the LSTM cell kernel (unreal_lstm_cell_act_heads) instead of a separate head
    # kernel reading h back.  OFF: measured at 8192 envs the fused kernel takes 19.4 us against 12.8 (cell) + 8.7 (heads) inside
    # the captured data phase -- no gain (scripts/act_heads_bench.py); kept as a tested option
    self.fused_act_heads = False
    # ... and the layout of the loss gradient between the fused deconv + loss kernel and the two backward kernels: "planes"
    # (four parity planes of 8 channels, one bulk copy per sample), "c8" ([S,400,8]) or "c16" (conv2's geometry, zero padded).
    # 8..15 actions: the 16-channel head, whose only layout is "c16" (all 16 channels real)
    self.pc_grad_layout = "planes" if A <= 7 else "c16"
    self._cells49 = torch.tensor([[x, y] for y in range(7) for x in range(7)], dtype=torch.int32, device=self._device)
    self._fc_tab_act = torch.zeros(49, 256, dtype=torch.bfloat16, device=self._device)
    self._act_xh = {}         # acting-step [x, h] GEMM operands by batch size (persistent: padding columns stay zero)
    self._build_variables(seed)
    self.reset_state()

  # ---- variables (model.py:752-783 initialisers) --------------------------------------
  def _build_variables(self, seed):
    A, G = self._action_size, self._objective_size
    specs = _variable_specs(A, G, self._use_pixel_change, self._use_reward_prediction)
    offsets, off = [], 0
    for name, shape, _ in specs:
      n = int(np.prod(shape))
      offsets.append((name, shape, off, n))
      off = (off + n + 7) // 8 * 8
    self._padded = (off + 31) // 32 * 32
    self.num_parameters = sum(o[3] for o in offsets)
    rs = np.random.RandomState(seed)
    host = np.zeros(self._padded, np.float32)
    for (name, shape, o, n), (_, _, fan_in) in zip(offsets, specs):
      if name == "lstm_kernel":       # BasicLSTMCell: TF default glorot-uniform kernel, zero bias
        lim = np.sqrt(6.0 / (shape[0] + shape[1]))
        v = rs.uniform(-lim, lim, size=shape)
      elif name == "lstm_bias":
        v = np.zeros(shape)
      else:
        d = 1.0 / np.sqrt(fan_in)
        v = rs.uniform(-d, d, size=shape)
      host[o:o + n] = v.astype(np.float32).reshape(-1)
    self.flat = torch.from_numpy(host).to(self._device).requires_grad_(True)
    self.flat16 = torch.zeros(self._padded, dtype=torch.bfloat16, device=self._device)
    self._offsets = offsets
    self.refresh_shadow()

  @property
  def encoder_precision(self):
    """'bf16' (bf16 operands, fp32 accumulation) or 'bf16x3' (split-bf16 operands in conv1 and conv2's forward pass)."""
    return self._encoder_precision

  def _views(self, flat):
    if torch.is_grad_enabled() and flat.requires_grad:      # one autograd node for all variables (layers.FlatViewsFn)
      return OrderedDict(zip((name for name, _, _, _ in self._offsets), FlatViewsFn.apply(flat, self._offsets)))
    return OrderedDict((name, flat[o:o + n].view(shape)) for name, shape, o, n in self._offsets)

  def refresh_shadow(self):
    """bf16 copy of the parameters for the GEMMs; call after every optimiser step."""
    with torch.no_grad():
      self.flat16.copy_(self.flat)
    self.v16 = self._views(self.flat16)
    # the LSTM kernel in the row layout of the per-step GEMM operand [x (KX columns, zero padded), h]
    wl = self.v16["lstm_kernel"]
    if getattr(self, "wcat16", None) is None:
      self.wcat16 = torch.zeros(self.kx + 256, 1024, dtype=torch.bfloat16, device=self._device)
    self.wcat16[:self.lstm_in].copy_(wl[:self.lstm_in]); self.wcat16[self.kx:].copy_(wl[self.lstm_in:])
    # tap-major filter shadows of the two encoder convolutions (TMA-im2col kernels); refreshed IN PLACE
    # so kernels captured in a CUDA graph keep reading the current filters
    if self.fused_conv:
      t1 = K.conv1_w_planes(self.v16["W_base_conv1"])
      t2 = K.conv_taps(self.v16["W_base_conv2"], 2)
      d2 = K.conv2_dgrad_taps(self.v16["W_base_conv2"])
      if getattr(self, "taps1", None) is None:
        self.taps1, self.taps2 = t1, (t2, d2)
      else:
        self.taps1.copy_(t1); self.taps2[0].copy_(t2); self.taps2[1].copy_(d2)
      if self._encoder_precision == 'bf16x3':
        # the same tap layouts of the rounding residuals bf16(W - bf16(W)) (the hi halves are taps1 / taps2[0])
        with torch.no_grad():
          v32 = self._views(self.flat)
          l1 = K.conv1_w_planes(K.split_bf16(v32["W_base_conv1"])[1])
          l2 = K.conv_taps(K.split_bf16(v32["W_base_conv2"])[1], 2)
        if getattr(self, "taps_lo", None) is None:
          self.taps_lo = (l1, l2)
        else:
          self.taps_lo[0].copy_(l1); self.taps_lo[1].copy_(l2)
    else:
      self.taps1 = self.taps2 = self.taps_lo = None
    if self._use_reward_prediction:
      # W_rp [7776,3] as a bf16 [7776,8] shadow (zero columns 3..7): the B operand of the head's tcgen05 GEMM
      if getattr(self, "rp_w8", None) is None:
        self.rp_w8 = torch.zeros(7776, 8, dtype=torch.bfloat16, device=self._device)
        self.rp_w24 = torch.zeros(2592, 24, dtype=torch.bfloat16, device=self._device)
      self.rp_w8[:, :3].copy_(self.v16["W_rp_fc1"])
      # the same filter by frame for the cell-table path: w24[r, f*8 + k] = W_rp[f*2592 + r, k]
      self.rp_w24.view(2592, 3, 8)[:, :, :3].copy_(self.v16["W_rp_fc1"].view(3, 2592, 3).permute(1, 0, 2))
    if self.fused_conv and self.fused_encoder and getattr(self, "dedup_cells", False):
      # acting-side table fc1(conv2(conv1(frame of cell))) for all 49 cells, refreshed IN PLACE with the parameters
      with torch.no_grad():
        p32 = self._views(self.flat)
        h2 = self._encoder_fn(p32, self._cells49)
        K.gemm_bf16(h2.view(49, 2592), self.v16["W_base_fc1"], out=self._fc_tab_act, b_mn_major=True, bias=p32["b_base_fc1"],
                    relu=True)
    if self._use_pixel_change and self._action_size > 7:
      # 8..15 actions: merged 16-channel shadow (channel 0 = value, 1..A = advantages, the rest zero) in conv2's geometry --
      # the deconv is conv2's transposed-convolution kernel, its backward pass conv2's forward and filter-gradient kernels
      A = self._action_size
      w16 = torch.zeros(4, 4, 16, 32, dtype=torch.bfloat16, device=self._device)
      w16[:, :, 0:1] = self.v16["W_pc_deconv_v"]; w16[:, :, 1:1 + A] = self.v16["W_pc_deconv_a"]
      b16 = torch.zeros(16, dtype=torch.float32, device=self._device)
      with torch.no_grad():
        v32 = self._views(self.flat)
        b16[0:1] = v32["b_pc_deconv_v"]; b16[1:1 + A] = v32["b_pc_deconv_a"]
      t16 = K.conv2_dgrad_taps(w16)
      l16 = K.conv_taps(w16, 2)
      if getattr(self, "pc_taps16", None) is None:
        self.pc_taps16, self.pc_b16, self.pc_lin_taps = t16, b16, l16
      else:
        self.pc_taps16.copy_(t16); self.pc_b16.copy_(b16); self.pc_lin_taps.copy_(l16)
    elif self._use_pixel_change:
      # merged 8-channel shadow of the two pixel-control deconv filters: channel 0 = value, 1..A = advantages
      A = self._action_size
      w8 = torch.zeros(4, 4, 8, 32, dtype=torch.bfloat16, device=self._device)
      w8[:, :, 0:1] = self.v16["W_pc_deconv_v"]; w8[:, :, 1:1 + A] = self.v16["W_pc_deconv_a"]
      b8 = torch.zeros(8, dtype=torch.float32, device=self._device)
      with torch.no_grad():
        v32 = self._views(self.flat)
        b8[0:1] = v32["b_pc_deconv_v"]; b8[1:1 + A] = v32["b_pc_deconv_a"]
      t8 = K.pc_deconv_taps(w8)           # tap-major shadow for the fused tcgen05 deconv forward
      w16 = torch.zeros(4, 4, 16, 32, dtype=torch.bfloat16, device=self._device)
      w16[:, :, :8] = w8                  # the same filter in conv2's geometry: the deconv's input gradient is conv2's forward
      l8 = K.conv_taps(w16, 2)
      l88 = K.conv_taps(w8, 2)            # ... without the 8 padding channels [32, 128], and as the plane kernels' tap tiles
      lpl = K.pc_w_planes(w8)
      if getattr(self, "pc_w8", None) is None:
        self.pc_w8, self.pc_b8, self.pc_taps, self.pc_lin_taps, self.pc_lin_taps8 = w8.view(128, 32), b8, t8, l8, l88
        self.pc_w_planes = lpl
      else:
        self.pc_w8.copy_(w8.view(128, 32)); self.pc_b8.copy_(b8); self.pc_taps.copy_(t8); self.pc_lin_taps.copy_(l8)
        self.pc_lin_taps8.copy_(l88); self.pc_w_planes.copy_(lpl)

  def get_vars(self):
    """The variables in creation order (views of the flat buffer), like model.py:729-730."""
    return list(self._views(self.flat.detach()).values())

  def named_vars(self):
    return self._views(self.flat.detach())

  def get_global_vars(self):
    return self.get_vars()

  def load_vars(self, named):
    """Copy TF-layout arrays (dict name -> array) into the flat buffer."""
    with torch.no_grad():
      views = self._views(self.flat)
      for k, v in named.items():
        views[k].copy_(torch.as_tensor(np.asarray(v), dtype=torch.float32).to(self._device))
    self.refresh_shadow()

  def sync_from(self, src_network, name=None):
    """model.py:735-749: copy the source network's variables (pairing by creation order)."""
    with torch.no_grad():
      self.flat.copy_(src_network.flat)
    self.refresh_shadow()

  # ---- towers -------------------------------------------------------------------------
  def _encoder_fn(self, p32, images):
    """The fused encoder node (EncoderFn) in this model's encoder precision."""
    return EncoderFn.apply(images, p32["W_base_conv1"], p32["b_base_conv1"], p32["W_base_conv2"], p32["b_base_conv2"],
                           self.taps1, self.taps2, self.taps_lo if self._encoder_precision == 'bf16x3' else None)

  def _encoder(self, p32, images):
    """model.py:281-289.  images [S,84,84,3] f32 / u8, x'' planes bf16 [S,6,441,8] or maze cells int32 [S,2]
    -> h2 bf16 [S,9,9,32]."""
    if self.fused_conv and self.fused_encoder:
      return self._encoder_fn(p32, images)
    if self._encoder_precision != 'bf16':
      raise _lib.UnrealError("encoder_precision 'bf16x3' needs the fused encoder (fused_conv and fused_encoder)")
    if images.dtype == torch.int32:
      raise _lib.UnrealError("cell observations (int32 [S,2]) need the fused encoder (fused_conv and fused_encoder)")
    h1 = ConvFn.apply(images, self.v16["W_base_conv1"].view(192, 16), p32["W_base_conv1"], p32["b_base_conv1"], 8, 8, 4,
                      self.taps1)
    h2 = ConvFn.apply(h1, self.v16["W_base_conv2"].view(256, 32), p32["W_base_conv2"], p32["b_base_conv2"], 4, 4, 2,
                      self.taps2)
    return h2

  def _lstm_input(self, p32, h2, t, n):
    """fc1 (model.py:332-340) -> bf16 [T,N,256]; LstmFn packs it with last_action_reward into the step operands (:343)."""
    fc = LinearFn.apply(h2.view(t * n, 2592), self.v16["W_base_fc1"], p32["W_base_fc1"], p32["b_base_fc1"], True, True)
    return fc.view(t, n, 256)

  def _gates_dtype(self):
    return torch.bfloat16 if self.lstm_gates_bf16 else torch.float32

  def _fused_step(self, n):
    return self.fused_lstm_step and self.lstm_gates_bf16 and n >= self.fused_lstm_min_rows

  def _use_tables(self, images):
    return self.dedup_cells and images.dtype == torch.int32 and self.fused_conv and self.fused_encoder

  def _cell_tables(self, p32):
    """(h2 table bf16 [49,2592], fc1 table f32 [49,256]) of the 49 maze cells, inside the autograd graph: every tower of
    the update gathers its rows from them, and their gradients arrive as per-cell sums."""
    h2t = self._encoder_fn(p32, self._cells49).view(49, 2592)
    fct = LinearFn.apply(h2t, self.v16["W_base_fc1"], p32["W_base_fc1"], p32["b_base_fc1"], True, True)
    return h2t, fct.float()

  def _tower(self, p32, images, lar, c0, h0, tables=None):
    """encoder + fc1 + LSTM unroll.  images [T,N,84,84,3], lar [T,N,A+1+G] -> h [T,N,256] f32."""
    t, n = images.shape[:2]
    if tables is not None and self._use_tables(images):
      # the fc1 rows are gathered from the 49-cell table straight into the LSTM step operands
      return LstmFn.apply(tables[1], lar.to(torch.float32), self.wcat16, p32["lstm_kernel"], p32["lstm_bias"], c0, h0,
                          self.lstm_in, self.kx, self._gates_dtype(), self._fused_step(n), images.reshape(t * n, 2)), None
    h2 = self._encoder(p32, images.reshape(t * n, *images.shape[2:]))
    fc = self._lstm_input(p32, h2, t, n)
    return LstmFn.apply(fc, lar.to(torch.float32), self.wcat16, p32["lstm_kernel"], p32["lstm_bias"], c0, h0, self.lstm_in,
                        self.kx, self._gates_dtype(), self._fused_step(n)), h2

  def _policy_value(self, p32, h, v_out=None):
    """model.py:358-377 (tiny [.,256]x[256,A+1] products, fp32).  Without autograd (acting, bootstraps): one fused
    head kernel (logits + softmax + value); with autograd: plain torch ops (the losses use A3CHeadLossFn instead)."""
    if self.fused_heads and not torch.is_grad_enabled() and self._action_size <= 15:
      lead = h.shape[:-1]
      out = K.a3c_head(h.reshape(-1, 256).contiguous(), p32["W_base_fc_p"].contiguous(), p32["b_base_fc_p"],
                       p32["W_base_fc_v"].reshape(256).contiguous(), p32["b_base_fc_v"], want_pi=True, want_v=True,
                       v_out=v_out)
      return out["pi"].view(*lead, self._action_size), out["v"].view(*lead)
    logits = h @ p32["W_base_fc_p"] + p32["b_base_fc_p"]
    v = (h @ p32["W_base_fc_v"] + p32["b_base_fc_v"]).squeeze(-1)
    if v_out is not None:
      v = v_out.copy_(v.reshape(v_out.shape))
    return torch.softmax(logits, dim=-1), v

  def _pc_head(self, p32, h):
    """pc_fc1 + the merged deconv (model.py:411-430): h [S,256] f32 -> y8 [S,20,20,8] f32 after ReLU
    (channel 0 = value stream, 1..A = advantage stream)."""
    A = self._action_size
    if A > 7:
      raise _lib.UnrealError(self._pc16_requirement())
    hp = LinearFn.apply(h, self.v16["W_pc_fc1"], p32["W_pc_fc1"], p32["b_pc_fc1"], True, True)
    return Deconv8Fn.apply(hp, self.pc_w8, self.pc_b8, p32["W_pc_deconv_v"], p32["b_pc_deconv_v"],
                           p32["W_pc_deconv_a"], p32["b_pc_deconv_a"], A, self.pc_taps if self.fused_conv else None)

  def _pc16_requirement(self):
    return ("with %d actions pixel control runs on the 16-channel fused tower only: it needs fused_conv, fused_encoder, "
            "fused_pc_loss and fused_pc_relu on and pc_grad_layout 'c16' (bootstraps: fused_conv and fused_pc_loss)"
            % self._action_size)

  def _pc_q(self, p32, h):
    """model.py:431-441: dueling combine.  h [S,256] f32 -> q [S,20,20,A], q_max [S,20,20]."""
    A = self._action_size
    y8 = self._pc_head(p32, h)
    v, a = y8[..., 0:1], y8[..., 1:1 + A]
    q = v + a - a.mean(dim=3, keepdim=True)
    return q, q.max(dim=3).values

  def _zeros_state(self, n):
    z = torch.zeros(n, 256, device=self._device)
    return z, z

  # ---- acting-side helpers (model.py:625-728), batched over envs ----------------------
  # The acting LSTM state lives in two persistent [N,256] buffers that are only ever updated IN PLACE,
  # so a CUDA graph that captured a rollout keeps reading / writing the live state on every replay.
  @property
  def base_lstm_state_out(self):
    return (self._lstm_c, self._lstm_h)

  @base_lstm_state_out.setter
  def base_lstm_state_out(self, state):
    c, h = state
    with torch.no_grad():
      self._lstm_c.copy_(torch.as_tensor(np.asarray(c.cpu() if isinstance(c, torch.Tensor) else c, dtype=np.float32)).to(self._device).view(-1, 256))
      self._lstm_h.copy_(torch.as_tensor(np.asarray(h.cpu() if isinstance(h, torch.Tensor) else h, dtype=np.float32)).to(self._device).view(-1, 256))

  def reset_state(self, mask=None):
    """model.py:625-628; `mask` [N] selects the envs whose state is zeroed (all when None)."""
    if not hasattr(self, "_lstm_c"):
      self._lstm_c = torch.zeros(self.num_envs, 256, device=self._device)
      self._lstm_h = torch.zeros(self.num_envs, 256, device=self._device)
    if mask is None:
      self._lstm_c.zero_(); self._lstm_h.zero_()
    else:
      keep = (mask == 0).to(torch.float32).unsqueeze(1)
      self._lstm_c.mul_(keep); self._lstm_h.mul_(keep)

  def _images(self, s_t):
    img = s_t['image'] if isinstance(s_t, dict) else s_t
    if not isinstance(img, torch.Tensor):
      img = torch.as_tensor(np.asarray(img, dtype=np.float32))
    img = img.to(self._device)
    return img.reshape(1, -1, *K.obs_shape(img.dtype))

  def _lar(self, last_action_reward, n):
    lar = last_action_reward
    if not isinstance(lar, torch.Tensor):
      lar = torch.as_tensor(np.asarray(lar, dtype=np.float32))
    return lar.to(self._device, torch.float32).reshape(1, n, -1)

  def _step(self, s_t, last_action_reward, state):
    with torch.no_grad():
      p32 = self._views(self.flat)
      img = self._images(s_t)
      n = img.shape[1]
      if self.fused_conv and self.fused_encoder:
        c1 = torch.empty(n, 256, device=self._device); h1 = torch.empty(n, 256, device=self._device)
        gates = self._step_gates(p32, img[0], self._lar(last_action_reward, n)[0], state[1])
        h16 = torch.empty(n, 256, device=self._device, dtype=torch.bfloat16)
        K.lstm_cell_fwd(gates, state[0].contiguous(), c1, h1, h16)
        return p32, h1, (c1, h1)
      (h, c1, h1), _ = self._tower(p32, img, self._lar(last_action_reward, n), state[0], state[1])
      return p32, h[0], (c1, h1)

  def _step_gates(self, p32, images, lar, h_prev, xh=None):
    """One acting step up to the LSTM gate pre-activations, without the training path's glue: fc1 writes straight
    into the [x, h] operand of the step GEMM (`xh`; None: the model's `_act_xh`, persistent, padding columns stay zero),
    the last action / reward vector and h are cast into their columns, one GEMM gives the gates [N,1024] f32."""
    n = images.shape[0]
    if xh is None:
      xh = self._act_xh.get(n)
      if xh is None:
        xh = self._act_xh[n] = torch.zeros(n, self.kx + 256, dtype=torch.bfloat16, device=self._device)
    elif tuple(xh.shape) != (n, self.kx + 256) or xh.dtype != torch.bfloat16:
      raise _lib.UnrealError("xh must be bf16 [%d, %d] with zero padding columns" % (n, self.kx + 256))
    if self._use_tables(images):      # maze cells: fc1's output is a row of the 49-entry table (refresh_shadow)
      K.cell_gather(self._fc_tab_act, images.reshape(n, 2), out=xh[:, :256])
    else:
      h2 = self._encoder_fn(p32, images)
      K.gemm_bf16(h2.view(n, 2592), self.v16["W_base_fc1"], out=xh[:, :256], b_mn_major=True, bias=p32["b_base_fc1"], relu=True)
    xh[:, 256:self.lstm_in].copy_(lar)
    xh[:, self.kx:].copy_(h_prev)
    return self._xh_gates(p32, xh)

  def _xh_gates(self, p32, xh, out=None):
    """The acting step's GEMM: gate pre-activations [N,1024] of a filled [x, h] operand."""
    return K.gemm_bf16(xh, self.wcat16, b_mn_major=True, bias=p32["lstm_bias"], out_dtype=self._gates_dtype(), out=out)

  def _act_cell_heads(self, p32, gates, c, h, active=None, v_out=None):
    """The acting step after the GEMM: the cell in place on the state rows (c, h) [N,256] of the active envs, then the
    policy / value heads -> (pi [N,A], v [N])."""
    if self.fused_heads and self.fused_act_heads and gates.dtype == torch.bfloat16 and self._action_size <= 7:
      # the cell and the heads in one launch: the warp that computes an env's h reduces its logits and value as well
      return K.lstm_cell_act_heads(gates, c, h, p32["W_base_fc_p"].contiguous(), p32["b_base_fc_p"],
                                   p32["W_base_fc_v"].reshape(256).contiguous(), p32["b_base_fc_v"], active, v_out)
    hh = torch.empty(gates.shape[0], 256, device=self._device)
    K.lstm_cell_act(gates, c, h, hh, active)      # in place on the state of the active envs
    return self._policy_value(p32, hh, v_out)

  def act_step(self, s_t, last_action_reward, c, h, active=None, v_out=None, xh=None):
    """run_base_policy_and_value on caller-owned state: the LSTM state rows c, h (f32 [N,256], updated in place for
    the active envs) and, optionally, the step GEMM's operand xh (bf16 [N, kx + 256], zero-initialised; None: the
    model's own per-batch-size operand) -> (pi [N,A], v [N])."""
    if self.fused_conv and self.fused_encoder:
      with torch.no_grad():
        p32 = self._views(self.flat)
        img = self._images(s_t)
        n = img.shape[1]
        gates = self._step_gates(p32, img[0], self._lar(last_action_reward, n)[0], h, xh)
        return self._act_cell_heads(p32, gates, c, h, active, v_out)
    p32, hh, new_state = self._step(s_t, last_action_reward, (c, h))
    with torch.no_grad():
      pi, v = self._policy_value(p32, hh, v_out)
      if active is None:
        c.copy_(new_state[0]); h.copy_(new_state[1])
      else:
        m = active.to(torch.bool).unsqueeze(1)
        c.copy_(torch.where(m, new_state[0], c))
        h.copy_(torch.where(m, new_state[1], h))
    return pi, v

  def run_base_policy_and_value(self, sess, s_t, last_action_reward, active=None, mode="", v_out=None):
    """model.py:630-660: one acting step; advances the LSTM state of the active envs.  `v_out` (f32 [N], contiguous): the
    values are written there (the batched rollout's history row) and returned as that tensor."""
    if v_out is not None and not (v_out.is_contiguous() and v_out.dtype == torch.float32):
      raise _lib.UnrealError("v_out must be a contiguous float32 [N] tensor")
    pi, v = self.act_step(s_t, last_action_reward, self._lstm_c, self._lstm_h, active, v_out)
    return pi, v, None

  def run_base_value(self, sess, s_t, last_action_reward):
    """model.py:687-704: bootstrap value; the LSTM state is NOT advanced."""
    p32, h, _ = self._step(s_t, last_action_reward, self.base_lstm_state_out)
    with torch.no_grad():
      return self._policy_value(p32, h)[1]

  def run_pc_q_max(self, sess, s_t, last_action_reward):
    """model.py:707-712 (zero LSTM state)."""
    img = self._images(s_t)
    p32, h, _ = self._step(s_t, last_action_reward, self._zeros_state(img.shape[1]))
    with torch.no_grad():
      if self.fused_conv and self.fused_pc_loss:
        # pc_fc1 GEMM, then the deconv with the dueling combine + max over actions in its epilogue (no [N,20,20,8] output)
        hp = K.gemm_bf16(h.to(torch.bfloat16), self.v16["W_pc_fc1"], b_mn_major=True, bias=p32["b_pc_fc1"], relu=True,
                         out_dtype=torch.bfloat16)
        if self._action_size > 7:
          return K.pc_deconv_qmax(hp, self.pc_taps16, self.pc_b16, self._action_size)
        return K.pc_deconv_qmax(hp, self.pc_taps, self.pc_b8, self._action_size)
      return self._pc_q(p32, h)[1]

  def run_vr_value(self, sess, s_t, last_action_reward):
    """model.py:715-720 (zero LSTM state)."""
    img = self._images(s_t)
    p32, h, _ = self._step(s_t, last_action_reward, self._zeros_state(img.shape[1]))
    with torch.no_grad():
      return self._policy_value(p32, h)[1]

  def run_rp_c(self, sess, state_history):
    """model.py:723-728: three frames [N,3,84,84,3] -> class probabilities [N,3]."""
    with torch.no_grad():
      return self._rp_c(self._views(self.flat), state_history)

  def _rp_features(self, p32, images):
    """model.py:475-480: the three frames' conv features, concatenated -> bf16 [N, 7776]."""
    n = images.shape[0]
    return self._encoder(p32, images.reshape(n * 3, *images.shape[2:])).reshape(n, 7776)

  def _rp_c(self, p32, images):
    """model.py:482-488 on the device path: tcgen05 GEMM on the padded weight shadow + fused bias / softmax."""
    h2 = self._rp_features(p32, images)
    logits8 = K.gemm_bf16(h2, self.rp_w8, b_mn_major=True, split_k=split_k_for(h2.shape[0], 8, 7776))
    return K.rp_loss(logits8, p32["b_rp_fc1"].contiguous(), want_p=True)["p"]

  # ---- losses (model.py:490-598) -------------------------------------------------------
  def loss(self, feed):
    """Total UNREAL loss summed over envs, and its parts.  feed (all time-major CUDA tensors):
       base: images [T,N,84,84,3], lar [T,N,A+1+G], a [T,N,A] one-hot, adv [T,N], R [T,N],
             mask [T,N], c0 / h0 [N,256]
       pc:   images [L,N,...], lar, a [L,N,A], R [L,N,20,20], mask [L,N]
       vr:   images, lar, R [L,N], mask [L,N]
       rp:   images [N,3,84,84,3], c [N,3] one-hot (zero, positive, negative)"""
    p32 = self._views(self.flat)
    parts = OrderedDict()
    b = feed["base"]
    tables = self._cell_tables(p32) if self._use_tables(b["images"]) else None
    (h, _, _), _ = self._tower(p32, b["images"], b["lar"], b["c0"], b["h0"], tables)
    mask = b["mask"].to(torch.float32)
    if self.fused_heads and self._action_size <= 15:
      t_, n_ = h.shape[:2]
      pol, val, ent = A3CHeadLossFn.apply(
          h.reshape(t_ * n_, 256), p32["W_base_fc_p"], p32["b_base_fc_p"], p32["W_base_fc_v"], p32["b_base_fc_v"],
          b["a"].reshape(t_ * n_, -1).argmax(-1).to(torch.int32), b["adv"].reshape(-1).contiguous(),
          b["R"].reshape(-1).contiguous(), mask.reshape(-1).contiguous(), self._entropy_beta, 0.25)
      parts["policy"], parts["value"], parts["entropy"] = pol, val, ent.detach()
    else:
      pi, v = self._policy_value(p32, h)
      log_pi = torch.log(pi.clamp(1e-20, 1.0))
      entropy = -(pi * log_pi).sum(-1)
      parts["policy"] = -((((log_pi * b["a"]).sum(-1)) * b["adv"] + entropy * self._entropy_beta) * mask).sum()
      parts["value"] = 0.25 * (((b["R"] - v) ** 2) * mask).sum()
      parts["entropy"] = (entropy * mask).sum().detach()
    total = parts["policy"] + parts["value"]
    if self._use_pixel_change and "pc" in feed:
      f = feed["pc"]
      L, n = f["images"].shape[:2]
      (h, _, _), _ = self._tower(p32, f["images"], f["lar"], *self._zeros_state(n), tables)
      act = f["a"].reshape(L * n, -1).argmax(-1).to(torch.int32)
      tgt = f["R"].reshape(L * n, 400).contiguous()
      msk = f["mask"].reshape(L * n).to(torch.float32).contiguous()
      fused_tower = self.fused_conv and self.fused_encoder and self.fused_pc_loss and self.fused_pc_relu
      if self._action_size > 7:
        if not (fused_tower and self.pc_grad_layout == "c16"):
          raise _lib.UnrealError(self._pc16_requirement())
        parts["pc"] = PcTowerFusedFn.apply(h.reshape(L * n, 256), self.v16["W_pc_fc1"], p32["W_pc_fc1"], p32["b_pc_fc1"],
                                           self.pc_taps16, self.pc_b16, self.pc_lin_taps, p32["W_pc_deconv_v"],
                                           p32["b_pc_deconv_v"], p32["W_pc_deconv_a"], p32["b_pc_deconv_a"], act, tgt, msk,
                                           self._action_size, self._pixel_change_lambda)
      elif fused_tower:
        # pc_fc1 + deconv + loss as one node: the ReLU / bias gradient of pc_fc1 leaves the backward convolution's epilogue
        parts["pc"] = PcTowerFusedFn.apply(h.reshape(L * n, 256), self.v16["W_pc_fc1"], p32["W_pc_fc1"], p32["b_pc_fc1"],
                                           self.pc_taps, self.pc_b8,
                                           {"planes": self.pc_w_planes, "c8": self.pc_lin_taps8}.get(self.pc_grad_layout, self.pc_lin_taps),
                                           p32["W_pc_deconv_v"], p32["b_pc_deconv_v"], p32["W_pc_deconv_a"], p32["b_pc_deconv_a"], act, tgt, msk,
                                           self._action_size, self._pixel_change_lambda)
      elif self.fused_conv and self.fused_encoder:
        hp = LinearFn.apply(h.reshape(L * n, 256), self.v16["W_pc_fc1"], p32["W_pc_fc1"], p32["b_pc_fc1"],
                            True, True)
        parts["pc"] = (PcFusedHeadLossFn if self.fused_pc_loss else PcHeadLossFn).apply(hp, self.pc_taps, self.pc_b8, self.pc_lin_taps, p32["W_pc_deconv_v"],
                                         p32["b_pc_deconv_v"], p32["W_pc_deconv_a"], p32["b_pc_deconv_a"], act, tgt, msk,
                                         self._action_size, self._pixel_change_lambda)
      else:
        y8 = self._pc_head(p32, h.reshape(L * n, 256))
        parts["pc"] = PcLossFn.apply(y8, act, tgt, msk, self._action_size, self._pixel_change_lambda)
      total = total + parts["pc"]
    if self._use_value_replay and "vr" in feed:
      f = feed["vr"]
      n = f["images"].shape[1]
      (h, _, _), _ = self._tower(p32, f["images"], f["lar"], *self._zeros_state(n), tables)
      if self.fused_heads:
        l_, n_ = h.shape[:2]
        _, parts["vr"], _ = A3CHeadLossFn.apply(
            h.reshape(l_ * n_, 256), p32["W_base_fc_p"], p32["b_base_fc_p"], p32["W_base_fc_v"], p32["b_base_fc_v"],
            None, None, f["R"].reshape(-1).contiguous(), f["mask"].float().reshape(-1).contiguous(), 0.0, 0.5)
      else:
        parts["vr"] = 0.5 * (((f["R"] - self._policy_value(p32, h)[1]) ** 2) * f["mask"].float()).sum()
      total = total + parts["vr"]
    if self._use_reward_prediction and "rp" in feed:
      f = feed["rp"]
      if tables is not None and self._use_tables(f["images"]):
        cells = f["images"].reshape(-1, 3, 2).to(torch.int64).clamp_(0, 6)
        parts["rp"] = RpCellLossFn.apply(tables[0], self.rp_w24, p32["W_rp_fc1"], p32["b_rp_fc1"],
                                         (cells[..., 1] * 7 + cells[..., 0]).contiguous(), f["c"].to(torch.float32).contiguous())
      else:
        parts["rp"] = RpHeadLossFn.apply(self._rp_features(p32, f["images"]), self.rp_w8, p32["W_rp_fc1"], p32["b_rp_fc1"],
                                         f["c"].to(torch.float32).contiguous())
      total = total + parts["rp"]
    return total, parts

  def loss_and_grads(self, feed, grad_scale=1.0):
    """-> (total, parts, flat gradient [padded P] of grad_scale * total)."""
    self.flat.grad = None
    total, parts = self.loss(feed)
    (total * grad_scale).backward()
    return total.detach(), {k: v.detach() for k, v in parts.items()}, self.flat.grad

  def feed_from_trainer(self, feed):
    """Batched Trainer feed (train/trainer.py of this package: env-major replay sequences as ring
    cells) -> the time-major tensors `loss()` consumes.  Replayed maze frames are re-rendered
    from their cells by K1's render kernel (the ring stores 8-byte records, not frames)."""
    b = feed['base']
    c0, h0 = b['start_lstm_state']
    out = {'base': dict(images=b['si'], lar=b['last_action_rewards'], a=b['a'], adv=b['adv'], R=b['R'],
                        mask=b['active'], c0=c0, h0=h0)}

    dt = b['si'].dtype                      # replayed frames are rendered in the rollout frames' format
    shp = K.obs_shape(dt)

    def seq(f):
      if 'images' in f:       # framed ring (FrameTrainer): the replayed frames themselves, time-major
        l, n = f['images'].shape[:2]
        mask = (torch.arange(l, device=f['images'].device).view(l, 1) < f['length'].view(1, n))
        return dict(images=f['images'], lar=f['last_action_reward'].transpose(0, 1).contiguous(), mask=mask)
      n, l = f['pos'].shape[:2]
      pos = f['pos'].transpose(0, 1).contiguous().view(l * n, 2)
      images = K.maze_render(pos, dtype=dt).view(l, n, *shp)
      mask = (torch.arange(l, device=pos.device).view(l, 1) < f['length'].view(1, n))
      return dict(images=images, lar=f['last_action_reward'].transpose(0, 1).contiguous(), mask=mask)

    if 'pc' in feed:
      f = feed['pc']
      d = seq(f)
      d['a'] = f['a'].transpose(0, 1).contiguous()
      d['R'] = f['R'].transpose(0, 1).contiguous()
      out['pc'] = d
    if 'vr' in feed:
      f = feed['vr']
      d = seq(f)
      d['R'] = f['R'].transpose(0, 1).contiguous()
      out['vr'] = d
    if 'rp' in feed:
      f = feed['rp']
      if 'images' in f:
        out['rp'] = dict(images=f['images'].contiguous(), c=f['c'])
        return out
      n = f['pos'].shape[0]
      out['rp'] = dict(images=K.maze_render(f['pos'].contiguous().view(n * 3, 2), dtype=dt).view(n, 3, *shp), c=f['c'])
    return out

  def update_gradient(self, feed, grad_scale=None):
    """The first half of update(): forward + backward of all heads -> (total, parts, flat gradient).  The learner under
    NCCL replays this as one CUDA graph and runs the gradient exchange + K6 after it (Trainer._update)."""
    if 'si' in feed["base"]:
      feed = self.feed_from_trainer(feed)
    n = feed["base"]["images"].shape[1]
    if grad_scale is None:
      grad_scale = self.grad_scale
    scale = (1.0 / n) if grad_scale is None else grad_scale
    return self.loss_and_grads(feed, scale)

  def update(self, feed, learning_rate, grad_applier, grad_scale=None):
    """One learner step: the reference's `sess.run(apply_gradients, feed_dict)` (trainer.py:543-559)."""
    if 'si' in feed["base"]:
      feed = self.feed_from_trainer(feed)
    n = feed["base"]["images"].shape[1]
    if grad_scale is None:
      grad_scale = self.grad_scale
    scale = (1.0 / n) if grad_scale is None else grad_scale
    total, parts, grad = self.loss_and_grads(feed, scale)
    norm = grad_applier.apply_flat_to(self.flat, grad, learning_rate)
    self.refresh_shadow()
    out = dict(parts)
    out["total"] = total
    out["grad_norm"] = norm
    return out
