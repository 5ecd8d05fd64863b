"""Dense layers of UnrealModel as autograd Functions over the K7 kernels.

Every matrix product -- forward, dgrad and wgrad -- is one call of the tcgen05 GEMM
(`unreal_gemm_bf16`); weights keep TensorFlow's layouts ([in, out] for tf.matmul, HWIO for conv2d,
[kh, kw, out, in] for conv2d_transpose; model/model.py:752-820) and are consumed where they lie:

    forward   y  = x @ W            A = x (K-major),   B = W   as [K, N]  (MN-major)
    dgrad     dx = dy @ W^T         A = dy (K-major),  B = W   as [N', K'] (K-major)
    wgrad     dW = x^T @ dy         A = x (MN-major),  B = dy  (MN-major), split-K over the samples

Activations travel in bf16 between layers (fp32 inside the LSTM cell, the heads and the losses);
gradients are rounded to bf16 only where they become GEMM operands.  torch.autograd is used as the
tape; ReLU masks, bf16 rounding and bias column sums are one fused kernel (`unreal_relu_grad`).
"""
import torch

from .. import kernels as K

_SM = 148


def split_k_for(m, n, k):
  """Split the reduction so that a wgrad (few output tiles, K = samples) fills the 148 SMs in ONE wave: tiles as
  unreal_gemm_bf16 cuts them (128 rows x 256 / 128 / 64 / 32 columns), and the largest split with tiles * split <= 148.
  Measured (profiles/r2_wgrad_split_bench.jsonl): the LSTM's [520,S]x[S,1024] gradient at S = 163 840 takes 242 us at
  split 4 (80 work items), 181 at 7 (140) and 263 at 8 (160: a second, nearly empty wave); fc1's [2592,S]x[S,256] at
  S = 20 480 takes 54 us at 8 and 38 at 7."""
  bn = 256 if n > 128 else (128 if n > 64 else (64 if n > 32 else 32))
  tiles = ((m + 127) // 128) * ((n + bn - 1) // bn)
  kb = (k + 63) // 64
  return max(1, min(_SM // tiles if tiles <= _SM else 1, max(1, kb // 4)))


SEGMENT_SUM_FIRST = True     # LstmFn's fc1-table gradient: segment sums of the gate gradients before the product (A/B switch)


def _wgrad(x16, dy16):
  """x16 [S, K_in], dy16 [S, N_out] (rows contiguous) -> f32 [K_in, N_out]."""
  s, kin = x16.shape
  nout = dy16.shape[1]
  return K.gemm_bf16(x16, dy16, a_mn_major=True, b_mn_major=True, split_k=split_k_for(kin, nout, s))


class FlatViewsFn(torch.autograd.Function):
  """The variables as views of the flat parameter buffer, as ONE autograd node: the backward pass zero-fills one flat
  gradient and copies each variable's gradient into its slice.  Plain slicing makes autograd build a full-size zero
  tensor per variable and add them up one by one (20 fills + 19 adds over 7.6 MB each per update)."""

  @staticmethod
  def forward(ctx, flat, offsets):
    ctx.offsets = offsets
    ctx.numel = flat.numel()
    return tuple(flat[o:o + n].view(shape) for _, shape, o, n in offsets)

  @staticmethod
  def backward(ctx, *grads):
    g = None
    for (_, _, o, n), gi in zip(ctx.offsets, grads):
      if gi is None:
        continue
      if g is None:
        g = torch.zeros(ctx.numel, dtype=gi.dtype, device=gi.device)
      g[o:o + n].copy_(gi.reshape(-1))
    return g, None


class LinearFn(torch.autograd.Function):
  """y = act(x @ W + b): tf.matmul layers (model.py:337-340 fc1, :424 pc_fc1)."""

  @staticmethod
  def forward(ctx, x16, w16, w32, b32, relu, out_bf16):
    # an fp32 input (the LSTM output feeding pc_fc1) is rounded to bf16 here, and its gradient leaves the dgrad GEMM as
    # fp32 -- instead of a cast node whose backward pass is one more pass over the [S,256] gradient
    ctx.x_f32 = x16.dtype == torch.float32
    if ctx.x_f32:
      x16 = x16.to(torch.bfloat16)
    y = K.gemm_bf16(x16, w16, b_mn_major=True, bias=b32, relu=relu,
                    out_dtype=torch.bfloat16 if out_bf16 else torch.float32)
    ctx.relu = relu
    ctx.save_for_backward(x16, w16, y if relu else None)
    return y

  @staticmethod
  def backward(ctx, dy):
    x16, w16, y = ctx.saved_tensors
    dy16, db = K.relu_grad(dy, y if ctx.relu else None)       # mask + bf16 + bias gradient in one pass
    dx = None
    if ctx.needs_input_grad[0]:
      dx = K.gemm_bf16(dy16, w16, out_dtype=torch.float32 if ctx.x_f32 else torch.bfloat16)
    dw = _wgrad(x16, dy16)
    return dx, None, dw, db, None, None


class ConvFn(torch.autograd.Function):
  """relu(conv2d(x, W, stride, VALID) + b) on NHWC input (model.py:283-289, :786-787).

  Forward: the two encoder geometries (8x8x3 stride 4 on frames, 4x4x16 stride 2 on conv1's output)
  run as implicit GEMMs whose im2col is done by the TMA engine (csrc/conv_tcgen05.cu; `taps` is the
  tap-major filter shadow); any other geometry goes through im2col + GEMM.
  Backward: wgrad is a split-K GEMM over the (recomputed) patch matrix, dgrad a GEMM + col2im."""

  @staticmethod
  def forward(ctx, x, w16, w32, b32, kh, kw, stride, taps):
    ctx.fused2 = False
    pre_s2d = x.dtype == torch.bfloat16 and tuple(x.shape[1:]) == (6, 441, 8)   # frames already as x'' planes
    s, h, w, c = (x.shape[0], 84, 84, 3) if pre_s2d else x.shape
    oh, ow = (h - kh) // stride + 1, (w - kw) // stride + 1
    o = w16.shape[1]
    xpp = None
    if pre_s2d:
      if taps is None:
        raise RuntimeError("space-to-depth frames need the fused conv1 kernel (UnrealModel.fused_conv)")
      xpp = x
      y = K.conv_fwd(xpp, 1, taps, b32).view(s * oh * ow, o)
    elif taps is not None and (h, w, c, kh, kw, stride, o) == (84, 84, 3, 8, 8, 4, 16) and x.dtype in (torch.float32, torch.uint8):
      xpp = K.s2d_frames(x)
      y = K.conv_fwd(xpp, 1, taps, b32).view(s * oh * ow, o)
    elif taps is not None and (h, w, c, kh, kw, stride, o) == (20, 20, 16, 4, 4, 2, 32) and x.dtype == torch.bfloat16:
      # conv2: taps = (forward tap filters [32,256], transposed-conv tap filters [4,64,32])
      y = K.conv_fwd(x, 2, taps[0], b32).view(s * oh * ow, o)
      ctx.fused2 = True
      ctx.dtaps = taps[1]
    else:
      cols = K.im2col(x, kh, kw, stride)
      y = K.gemm_bf16(cols, w16, b_mn_major=True, bias=b32, relu=True, out_dtype=torch.bfloat16)
    ctx.geom = (s, h, w, c, kh, kw, stride, oh, ow, o)
    # conv1 keeps its space-to-depth frames (42 KB/frame) for the fused wgrad instead of the frame
    ctx.save_for_backward(x if xpp is None else None, w16, y, xpp)
    return y.view(s, oh, ow, o)

  @staticmethod
  def backward(ctx, dy):
    x, w16, y, xpp = ctx.saved_tensors
    s, h, w, c, kh, kw, stride, oh, ow, o = ctx.geom
    if xpp is not None:      # conv1: tensor-core wgrad straight from x'' and the masked dY planes
      dyp, db = K.relu_grad(dy.reshape(-1, o), y, planes=True)
      return None, None, K.conv1_wgrad(xpp, dyp), db, None, None, None, None
    dy16, db = K.relu_grad(dy.reshape(-1, o), y)
    if ctx.fused2:           # conv2: the filter gradient straight from h1 and dY2 through TMA boxes
      dw = K.conv2_wgrad(x, dy16)
    else:
      cols = K.im2col(x, kh, kw, stride)
      dw = _wgrad(cols, dy16).view(kh, kw, c, o)
    dx = None
    if ctx.needs_input_grad[0]:
      if ctx.fused2:         # transposed convolution as a 4-tap implicit GEMM over zero-filling TMA boxes
        dx = K.conv2_dgrad(dy16, ctx.dtaps)
      else:
        dcols = K.gemm_bf16(dy16, w16, out_dtype=torch.bfloat16)          # [S*OH*OW, KH*KW*C]
        dx = K.col2im(dcols, s, h, w, c, kh, kw, stride, out_dtype=torch.bfloat16)
    return dx, None, dw, db, None, None, None, None


class EncoderFn(torch.autograd.Function):
  """The whole encoder (model.py:281-289: conv 8x8x3->16 stride 4 + ReLU, conv 4x4x16->32 stride 2 + ReLU) as
  ONE autograd node over the fused tcgen05 kernels, so the backward pass can fuse ACROSS the two layers:
  conv2's transposed convolution masks its result by h1 > 0 in the epilogue and writes conv1's wgrad planes
  and bias gradient directly (`unreal_conv2_dgrad_relu`) -- the dense [S,20,20,16] gradient and the separate
  ReLU-gradient pass over it (38 KB per frame of HBM traffic) do not exist.  Frames: f32 / u8 [S,84,84,3], the
  space-to-depth planes bf16 [S,6,441,8], or maze CELLS int32 [S,2] (the conv1 kernels then synthesise their
  input tiles in shared memory: unreal_conv1_fwd_maze / unreal_conv1_wgrad_maze).

  taps_lo = (conv1 planes, conv2 taps) of the filters' rounding residuals bf16(W - bf16(W)): the split-bf16 forward
  (UnrealModel(encoder_precision='bf16x3')).  Frames, conv1's output and the filters enter conv1 and conv2 as hi + lo
  bf16 pairs (three tensor-core passes; two where the input is exactly bf16: maze cells, x'' planes), so the forward
  products are fp32-grade.  Only the hi halves are kept for the backward pass, which is the bf16 one: the gradient
  rounding it adds is far below the forward rounding the split removes."""

  @staticmethod
  def forward(ctx, x, w1_32, b1_32, w2_32, b2_32, taps1, taps2, taps_lo=None):
    pre_s2d = x.dtype == torch.bfloat16 and tuple(x.shape[1:]) == (6, 441, 8)
    s = x.shape[0]
    ctx.cells = x.dtype == torch.int32                          # maze cells [S,2]: render-fused conv1, no frame in HBM
    if taps_lo is not None:
      if ctx.cells:
        xpp = x.contiguous()
        h1, h1_lo = K.conv1_fwd_maze_split(xpp, taps1, taps_lo[0], b1_32)
      else:
        xpp, xpp_lo = (x, None) if pre_s2d else K.s2d_frames_split(x)
        h1, h1_lo = K.conv1_fwd_split(xpp, xpp_lo, taps1, taps_lo[0], b1_32)
      h2 = K.conv2_fwd_split(h1, h1_lo, taps2[0], taps_lo[1], b2_32)
    else:
      if ctx.cells:
        xpp = x.contiguous()
        h1 = K.conv1_fwd_maze(xpp, taps1, b1_32)
      else:
        xpp = x if pre_s2d else K.s2d_frames(x)
        h1 = K.conv_fwd(xpp, 1, taps1, b1_32)                  # bf16 [S,20,20,16]
      h2 = K.conv_fwd(h1.view(s, 20, 20, 16), 2, taps2[0], b2_32)
    ctx.dtaps = taps2[1]
    ctx.save_for_backward(xpp, h1, h2)
    return h2.view(s, 9, 9, 32)

  @staticmethod
  def backward(ctx, dh2):
    xpp, h1, h2 = ctx.saved_tensors
    s = xpp.shape[0]
    dy2, db2 = K.relu_grad(dh2.reshape(-1, 32), h2.view(-1, 32))
    dw2 = K.conv2_wgrad(h1.view(s, 20, 20, 16), dy2)
    dy1_planes, db1 = K.conv2_dgrad_relu(dy2, ctx.dtaps, h1, pitch21=True)
    dw1 = K.conv1_wgrad_maze(xpp, dy1_planes) if ctx.cells else K.conv1_wgrad(xpp, dy1_planes)
    return None, dw1, db1, dw2, db2, None, None, None


class LstmFn(torch.autograd.Function):
  """dynamic_rnn over BasicLSTMCell(256) (model.py:110, :343-351), N envs in lock step.

  Step operand row [KX+256] bf16: columns [0, lstm_in) = concat(fc1 output, last_action_reward), zero padding up
  to KX (lstm_in rounded up to 8 for the TMA row pitch), then h_{t-1}.  `wcat16` [KX+256, 1024] is the cell's
  kernel in that row layout (x rows, zero rows for the padding, h rows).  Each step is ONE GEMM over the
  concatenated operand [x_t, h_{t-1}] (K = KX + 256) whose epilogue adds the bias and writes the gate
  pre-activations once; the cell kernel writes h_t (bf16) straight into step t+1's operand columns.  (The
  earlier form -- one GEMM for all x-parts, then a read-modify-write accumulation of h W_h per step -- moved
  100 MB per step through HBM for the gates at 8192 envs instead of 33.5 MB.)
  """

  @staticmethod
  def forward(ctx, fc16, lar, wcat16, w32, b32, c0, h0, lstm_in, kx, gates_dtype=torch.float32, fused_step=False, pos=None):
    """fc16 [T,N,256] bf16 (fc1 output), lar [T,N,lstm_in-256] f32: packed straight into the step operands.
    pos int32 [T*N,2] (maze cells): fc16 is instead the 49-row fc1 TABLE [49,256] f32 (CellGatherFn's operand) and the
    rows are gathered straight into the operands' fc1 columns -- no [T,N,256] intermediate and no strided copy of it
    (84 MB each way per tower at 8192 envs) -- with the segment sum by cell as the table's gradient.
    gates_dtype bf16: the step GEMM writes the gate pre-activations as bf16 and the cell keeps their activations for the
    backward pass as bf16 (half the traffic of the HBM-bound cell kernels).
    fused_step (needs bf16 gates): one launch per step in both directions -- the cell runs in the step GEMM's epilogue
    (unreal_lstm_step_fwd: the pre-activations never reach HBM, only the bf16 activations the backward pass reads) and
    the cell's backward pass in the epilogue of the recurrent dh GEMM (unreal_lstm_step_bwd)."""
    t, n = lar.shape[:2]
    kc = kx + 256
    dev = fc16.device
    xh = torch.empty(t, n, kc, device=dev, dtype=torch.bfloat16)
    if pos is not None:
      K.cell_gather(fc16.to(torch.bfloat16), pos, out=xh.view(t * n, kc)[:, :256])      # exact: the table holds bf16 values
    else:
      xh[:, :, :256].copy_(fc16)
    xh[:, :, 256:lstm_in].copy_(lar)
    if kx > lstm_in:
      # padding columns: zero, except a ONE in the last of them -- its row of the kernel shadow is zero, so the steps are
      # unchanged, and its row of the wgrad GEMM's result is the column sum of the gate gradients = the bias gradient
      # (instead of a separate pass over the [T*N, 1024] gradient)
      pad = (torch.arange(lstm_in, kx, device=dev) == kx - 1).to(torch.bfloat16)      # device ops only: graph-capture safe
      xh[:, :, lstm_in:kx].copy_(pad)
    xh[0, :, kx:].copy_(h0)
    fused_step = bool(fused_step) and gates_dtype == torch.bfloat16
    # fused steps: c of every step and the gate activations are touched by the step kernels only and live in their tiled
    # layout (kernels.tile32; rows padded to a multiple of 32)
    nt = (n + 31) // 32 * 32 if fused_step else n
    gates = torch.empty(t, nt, 1024, device=dev, dtype=gates_dtype)
    c_all = torch.empty(t + 1, nt, 256, device=dev)
    h_all = torch.empty(t, n, 256, device=dev)
    if fused_step:
      c_all[0].copy_(K.tile32(c0))
      for i in range(t):
        K.lstm_step_fwd(xh[i], wcat16, b32, c_all[i], c_all[i + 1], h_out=h_all[i],
                        h16_out=xh[i + 1, :, kx:] if i + 1 < t else None, acts=gates[i], tiled=True)
      c_last = K.untile32(c_all[t], n).contiguous()
    else:
      h16_last = torch.empty(n, 256, device=dev, dtype=torch.bfloat16)
      c_all[0].copy_(c0)
      for i in range(t):
        K.gemm_bf16(xh[i], wcat16, out=gates[i], b_mn_major=True, bias=b32)
        K.lstm_cell_fwd(gates[i], c_all[i], c_all[i + 1], h_all[i], xh[i + 1, :, kx:] if i + 1 < t else h16_last)
      c_last = c_all[t].clone()
    ctx.fused_step = fused_step
    ctx.lstm_in = lstm_in
    ctx.kx = kx
    ctx.extra = ()
    if pos is not None:       # the fc1 table as the (zero-padded) bf16 operand of the backward pass's 49-row products
      table16 = torch.zeros(64, 256, device=dev, dtype=torch.bfloat16)
      table16[:49].copy_(fc16)
      ctx.extra = (table16,)
    ctx.save_for_backward(xh, wcat16, gates, c_all, pos)
    return h_all, c_last, h_all[t - 1].clone()

  @staticmethod
  def backward(ctx, dh_all, dc_last, dh_last):
    xh, wcat16, gates, c_all, pos = ctx.saved_tensors
    lstm_in, kx = ctx.lstm_in, ctx.kx
    t, n, kc = xh.shape
    dev = xh.device
    dh_all = dh_all.contiguous()
    dgates = torch.empty(t, n, 1024, device=dev, dtype=torch.bfloat16)
    wh = wcat16[kx:]                                     # [256, 1024]: K-major B for dh = dgates @ Wh^T
    dh_rec = None if dh_last is None else dh_last.contiguous()
    if ctx.fused_step:
      dc = torch.zeros(c_all.shape[1], 256, device=dev) if dc_last is None else K.tile32(dc_last)
    else:
      dc = torch.zeros(n, 256, device=dev) if dc_last is None else dc_last.clone().contiguous()
    for i in range(t - 1, -1, -1):
      if ctx.fused_step:
        K.lstm_step_bwd(dgates[i + 1] if i < t - 1 else None, wh, gates[i], c_all[i], c_all[i + 1], dh_all[i], dc, dgates[i],
                        dh2=dh_rec if i == t - 1 else None, tiled=True)
        continue
      K.lstm_cell_bwd(gates[i], c_all[i], c_all[i + 1], dh_all[i], dc, dgates[i], dh_rec)    # dh = dh_all[i] + dh_rec
      if i > 0:
        # small batches: this [N,1024] x [256,1024]^T product is one N tile wide -- split K over more CTAs (measured
        # 10.3 -> 5.1 us at 1024 envs; at 8192 envs the output's zero fill costs what the split saves)
        dh_rec = K.gemm_bf16(dgates[i], wh, split_k=4 if n <= 2048 else 1)
    dg2 = dgates.view(t * n, 1024)
    if pos is not None and SEGMENT_SUM_FIRST and lstm_in - 256 <= 14:
      # table mode (maze cells): sums over samples commute with the products, so the gate gradients are summed BY CELL first --
      # as a tensor-core GEMM against an indicator matrix P [S,64] = [one-hot cell (49) | last action / reward columns of the
      # operand | 1 | 0 ...] (products by 0 / 1 / the operand's own bf16 values, fp32 accumulation; one pass over dgates at
      # HBM speed) -- and everything that involves the operand's x columns comes out of that one [64,1024] result R:
      #   d(fc1 table) = R[:49] . W_x[:256]^T    instead of the [T*N,1024] x [1024,256] GEMM + the segment-sum pass over its result;
      #   dW_x[:256]   = table^T . R[:49]        instead of the fc1 half of the [520,T*N] x [T*N,1024] filter-gradient GEMM;
      #   dW_x[256:]   = R[49:49+nl],  db = R[49+nl]   (the last-action / reward rows and the bias);
      # the big filter-gradient GEMM is left with the 256 h columns: exactly two 128-row tiles.
      (table16,) = ctx.extra
      nl = lstm_in - 256
      xh2 = xh.view(t * n, kc)
      cell = (pos[:, 1].to(torch.int64) * 7 + pos[:, 0].to(torch.int64)).clamp_(0, 48)
      ind = torch.zeros(t * n, 64, device=dev, dtype=torch.bfloat16)
      ind.scatter_(1, cell.view(-1, 1), 1.0)
      ind[:, 49:49 + nl].copy_(xh2[:, 256:lstm_in])
      ind[:, 49 + nl].fill_(1.0)
      r = _wgrad(ind, dg2)                                                           # [64,1024] f32
      gsum16 = r.to(torch.bfloat16)
      dfc = K.gemm_bf16(gsum16, wcat16[:256])[:49].contiguous()                      # [49,256] f32
      dw_fc = _wgrad(table16, gsum16)                                                # [256,1024] f32 (table rows 49..63 are zero)
      dw_h = _wgrad(xh2[:, kx:], dg2)                                                # [256,1024] f32
      dw = torch.cat((dw_fc, r[49:49 + nl], dw_h), dim=0)
      db = r[49 + nl].clone()
      return dfc, None, None, dw, db, None, None, None, None, None, None, None
    dwcat = _wgrad(xh.view(t * n, kc), dg2)              # one wgrad over [x, h]: rows of the x part, padding, h part
    dw = torch.cat((dwcat[:lstm_in], dwcat[kx:]), dim=0)
    if kx > lstm_in:
      db = dwcat[kx - 1].clone()                         # the ones column of the operand (forward)
    else:
      _, db = K.relu_grad(dg2, None, want_out=False)
    # only the 256 fc1 columns carry a gradient (last_action_reward is an input)
    dfc = K.gemm_bf16(dg2, wcat16[:256], out_dtype=torch.bfloat16)
    dfc = dfc.view(t, n, 256) if pos is None else K.cell_segment_sum(dfc, pos)      # table mode: per-cell sums, fp32 [49,256]
    return dfc, None, None, dw, db, None, None, None, None, None, None, None


class Deconv8Fn(torch.autograd.Function):
  """The pixel-control head's two transposed convolutions (value: 1 channel, advantage: A channels;
  model.py:418-430) as ONE 8-channel deconv: y8[..., 0] = relu(deconv_v), y8[..., 1:1+A] =
  relu(deconv_a), channels A+1..7 zero padding.  `w8` is the merged bf16 filter shadow
  [(kh,kw,o8) = 128, 32]; the gradient is split back into the two TF-layout variables.  Forward with
  `taps` (the tap-major shadow): unreal_pc_deconv_fwd, conv2's transposed-convolution tcgen05 kernel at 8
  channels with the bias + ReLU epilogue; without: GEMM into f32 columns + col2im."""

  @staticmethod
  def forward(ctx, h16, w8, b8, wv32, bv32, wa32, ba32, num_actions, taps=None):
    s = h16.shape[0]
    if taps is not None:     # the transposed convolution as a 4-tap implicit GEMM over zero-filling TMA boxes
      y = K.pc_deconv_fwd(h16, taps, b8)                                 # f32 [S,20,20,8]
    else:
      cols = K.gemm_bf16(h16.view(s * 81, 32), w8)                       # f32 [S*81, 128]
      y = K.col2im(cols, s, 20, 20, 8, 4, 4, 2, bias=b8, relu=True)      # f32 [S,20,20,8]
    ctx.num_actions = num_actions
    ctx.save_for_backward(h16, w8)
    return y

  @staticmethod
  def backward(ctx, dy):
    """dy must already be masked by y > 0 (PcLossFn produces it that way)."""
    h16, w8 = ctx.saved_tensors
    a = ctx.num_actions
    s = h16.shape[0]
    dy = dy.contiguous()
    dcols = K.im2col(dy, 4, 4, 2)                                          # bf16 [S*81, 128]
    dh = K.gemm_bf16(dcols, w8, b_mn_major=True, out_dtype=torch.bfloat16).view(s, 2592)
    dw8 = _wgrad(dcols, h16.view(s * 81, 32)).view(4, 4, 8, 32)
    _, db8 = K.relu_grad(dy.view(s * 400, 8), None, want_out=False)
    return (dh, None, None, dw8[:, :, 0:1].contiguous(), db8[0:1].clone(), dw8[:, :, 1:1 + a].contiguous(),
            db8[1:1 + a].clone(), None, None)


class PcLossFn(torch.autograd.Function):
  """lam * 0.5 * sum mask * (R - Q[a])^2 with Q = V + Adv - mean Adv (model.py:431-441, :531-546) in
  one fused pass over y8; the backward pass is the same kernel writing d loss / d (pre-ReLU y8)."""

  @staticmethod
  def forward(ctx, y8, act, target, mask, num_actions, lam):
    loss, _ = K.pc_loss(y8.view(y8.shape[0], 400, 8), act, target, mask, num_actions, lam)
    ctx.cfg = (num_actions, lam)
    ctx.save_for_backward(y8, act, target, mask)
    return loss[0].to(torch.float32)

  @staticmethod
  def backward(ctx, go):
    y8, act, target, mask = ctx.saved_tensors
    a, lam = ctx.cfg
    _, dy = K.pc_loss(y8.view(y8.shape[0], 400, 8), act, target, mask, a, lam, want_loss=False, want_grad=True,
                      go=go.to(torch.float32).reshape(1).contiguous())
    return dy.view_as(y8), None, None, None, None, None


class PcHeadLossFn(torch.autograd.Function):
  """The pixel-control head after pc_fc1 and its loss as ONE autograd node (model.py:418-441, :531-546): merged
  8-channel deconv forward (conv2's transposed-convolution kernel) -> dueling / gather / L2 loss kernel.  The
  backward pass never leaves the encoder's conv2 kernels: the loss gradient is written as conv2-geometry input
  (bf16, 16 channels, with the deconv bias gradient), the input gradient is conv2's FORWARD kernel over it
  (`unreal_conv2_fwd_linear`: d/dx of a transposed convolution is the convolution) and the filter gradient is
  conv2's wgrad kernel with the roles of activation and gradient exchanged -- no im2col, no column matrices."""

  @staticmethod
  def forward(ctx, h16, taps, b8, lin_taps, wv32, bv32, wa32, ba32, act, target, mask, num_actions, lam):
    s = h16.shape[0]
    y8 = K.pc_deconv_fwd(h16, taps, b8)                                 # f32 [S,20,20,8]
    loss, _ = K.pc_loss(y8.view(s, 400, 8), act, target, mask, num_actions, lam)
    ctx.cfg = (num_actions, lam)
    ctx.lin_taps = lin_taps
    ctx.save_for_backward(h16, y8, act, target, mask)
    return loss[0].to(torch.float32)

  @staticmethod
  def backward(ctx, go):
    h16, y8, act, target, mask = ctx.saved_tensors
    a, lam = ctx.cfg
    s = h16.shape[0]
    dy16, db8 = K.pc_loss_grad16(y8.view(s, 400, 8), act, target, mask, a, lam, go.to(torch.float32).reshape(1).contiguous())
    dy16 = dy16.view(s, 20, 20, 16)
    dh = K.conv2_fwd_linear(dy16, ctx.lin_taps).view(s, 2592)
    dw16 = K.conv2_wgrad(dy16, h16.reshape(s * 81, 32))                  # [4,4,16,32]: channels 8..15 are padding
    return (dh, None, None, None, dw16[:, :, 0:1].contiguous(), db8[0:1].clone(), dw16[:, :, 1:1 + a].contiguous(),
            db8[1:1 + a].clone(), None, None, None, None, None)


class PcFusedHeadLossFn(torch.autograd.Function):
  """PcHeadLossFn with the loss fused INTO the deconv kernel (`unreal_pc_deconv_loss`): the f32 head output [S,20,20,8]
  (2.1 GB per update at 8192 envs) is never written -- the epilogue that holds a pixel's 8 channels finishes the dueling /
  gather / L2 loss and writes its gradient as the conv2-geometry bf16 operand of the backward pass directly.  The upstream
  gradient (a device scalar) is applied by the backward convolutions (`unreal_conv2_fwd_linear_scaled`) and to the two
  small filter / bias gradients."""

  @staticmethod
  def forward(ctx, h16, taps, b8, lin_taps, wv32, bv32, wa32, ba32, act, target, mask, num_actions, lam):
    loss, dy16, db8 = K.pc_deconv_loss(h16, taps, b8, act, target, mask, num_actions, lam)
    ctx.num_actions = num_actions
    ctx.lin_taps = lin_taps
    ctx.save_for_backward(h16, dy16, db8)
    return loss[0].to(torch.float32)

  @staticmethod
  def backward(ctx, go):
    h16, dy16, db8 = ctx.saved_tensors
    a = ctx.num_actions
    s = h16.shape[0]
    go32 = go.to(torch.float32).reshape(1).contiguous()
    dy16 = dy16.view(s, 20, 20, 16)
    dh = K.conv2_fwd_linear(dy16, ctx.lin_taps, scale=go32).view(s, 2592)
    dw16 = K.conv2_wgrad(dy16, h16.reshape(s * 81, 32)) * go32           # [4,4,16,32]: channels 8..15 are padding
    db8 = db8 * go32
    return (dh, None, None, None, dw16[:, :, 0:1].contiguous(), db8[0:1].clone(), dw16[:, :, 1:1 + a].contiguous(),
            db8[1:1 + a].clone(), None, None, None, None, None)


class PcTowerFusedFn(torch.autograd.Function):
  """pc_fc1 (model.py:424) + PcFusedHeadLossFn as ONE autograd node, so that pc_fc1's ReLU gradient and bias gradient come
  out of the backward convolution's epilogue instead of a `unreal_relu_grad` pass over the dense [S,2592] gradient (read
  2 x 849 MB + write 849 MB per update at 8192 envs x 20).  `lin_taps` selects the layout the loss gradient travels in
  between the fused deconv + loss kernel and the two backward kernels:
    [32, 256]      conv2's geometry [S,400,16], channels 8..15 zero (`unreal_conv2_fwd_linear_masked`, `unreal_conv2_wgrad`);
    [32, 128]      the 8 real channels [S,400,8] (the same kernels' 8-channel builds);
    [4,2,2,32,8]   (`K.pc_w_planes`) four parity planes [S,4,100,8]: one bulk copy per sample (`unreal_pc_planes_conv`,
                   `unreal_pc_planes_wgrad`) -- what the agent runs."""

  @staticmethod
  def forward(ctx, h, w16, w32, b32, taps, b8, lin_taps, wv32, bv32, wa32, ba32, act, target, mask, num_actions, lam):
    ctx.x_f32 = h.dtype == torch.float32
    x16 = h.to(torch.bfloat16) if ctx.x_f32 else h
    hp = K.gemm_bf16(x16, w16, b_mn_major=True, bias=b32, relu=True, out_dtype=torch.bfloat16)
    ctx.planes = lin_taps.dim() == 5
    ctx.c = 8 if ctx.planes else lin_taps.shape[1] // 16
    loss, dy16, db8 = K.pc_deconv_loss(hp, taps, b8, act, target, mask, num_actions, lam, c8=ctx.c == 8, planes=ctx.planes)
    ctx.num_actions = num_actions
    ctx.lin_taps = lin_taps
    ctx.save_for_backward(x16, w16, hp, dy16, db8)
    return loss[0].to(torch.float32)

  @staticmethod
  def backward(ctx, go):
    x16, w16, hp, dy16, db8 = ctx.saved_tensors
    a = ctx.num_actions
    s = hp.shape[0]
    go32 = go.to(torch.float32).reshape(1).contiguous()
    # d(pc_fc1 output), masked by hp > 0, + pc_fc1's bias gradient; the deconv filters' gradient ([4,4,16 (8),32])
    if ctx.planes:
      dhp, db = K.pc_planes_conv(dy16, ctx.lin_taps, hp, scale=go32)
      dw16 = K.pc_planes_wgrad(dy16, hp) * go32
    else:
      dy16 = dy16.view(s, 20, 20, ctx.c)
      dhp, db = K.conv2_fwd_linear(dy16, ctx.lin_taps, scale=go32, mask_y=hp)
      dw16 = K.conv2_wgrad(dy16, hp.view(s * 81, 32)) * go32
    dhp = dhp.view(s, 2592)
    db8 = db8 * go32
    dx = None
    if ctx.needs_input_grad[0]:
      dx = K.gemm_bf16(dhp, w16, out_dtype=torch.float32 if ctx.x_f32 else torch.bfloat16)
    dw = _wgrad(x16, dhp)
    return (dx, None, dw, db, None, None, None, dw16[:, :, 0:1].contiguous(), db8[0:1].clone(),
            dw16[:, :, 1:1 + a].contiguous(), db8[1:1 + a].clone(), None, None, None, None, None)


class A3CHeadLossFn(torch.autograd.Function):
  """Policy / value heads and their losses as ONE autograd node over two kernels (model.py:358-377, :499-527, :556-565):
  the forward pass computes logits, softmax, value, the policy / value / entropy sums and the gradients w.r.t. logits
  and value in one sweep over h; the backward pass is one more sweep (dh and the four head gradients).  `act` None:
  value loss only (the value-replay tower).  Returns (policy_loss, value_loss, entropy) as fp32 scalars."""

  @staticmethod
  def forward(ctx, h, wp, bp, wv, bv, act, adv, ret, mask, entropy_beta, value_coef):
    h = h.contiguous()
    wv1 = wv.reshape(256).contiguous()
    out = K.a3c_head(h, wp.contiguous() if act is not None else None, bp, wv1, bv, act, adv, ret, mask, entropy_beta,
                     value_coef, want_sums=True, want_grads=True)
    ctx.has_policy = act is not None
    ctx.save_for_backward(h, wp.contiguous() if act is not None else None, wv1, out.get("dz"), out.get("dv"))
    sums = out["sums"].to(torch.float32)
    return sums[0].clone(), sums[1].clone(), sums[2].clone()

  @staticmethod
  def backward(ctx, g_pol, g_val, g_ent):
    h, wp, wv1, dz, dv = ctx.saved_tensors
    zero = torch.zeros((), dtype=torch.float32, device=h.device)
    go2 = torch.stack((g_pol.to(torch.float32) if g_pol is not None else zero,
                       g_val.to(torch.float32) if g_val is not None else zero)).contiguous()
    dh, dwp, dbp, dwv, dbv = K.a3c_head_bwd(h, wp, wv1, dz, dv, go2)
    return (dh, dwp, dbp, None if dwv is None else dwv.view(256, 1), dbv, None, None, None, None, None, None)


class RpHeadLossFn(torch.autograd.Function):
  """The reward-prediction head and its loss as ONE autograd node (model.py:479-488 fc 7776 -> 3 + softmax, :571-575
  cross-entropy with the clipped probabilities): the fc is the tcgen05 GEMM over a bf16 shadow of W_rp padded to 8
  columns (`w8`, [7776, 8]; TMA needs 16-byte rows), split-K so that the 64 row tiles of a 8192-sample batch fill the
  SMs; `unreal_rp_loss` adds the bias and does softmax, loss and d loss / d logits (as the bf16 [N,8] GEMM operand, with
  the bias gradient) in one pass.  Backward: dh2 = dz . W^T and dW = h2^T . dz are two more tcgen05 GEMMs."""

  @staticmethod
  def forward(ctx, h2_16, w8, w32, b32, c):
    n = h2_16.shape[0]
    logits8 = K.gemm_bf16(h2_16, w8, b_mn_major=True, split_k=split_k_for(n, 8, h2_16.shape[1]))
    out = K.rp_loss(logits8, b32, c, want_loss=True)
    ctx.save_for_backward(h2_16, w8, logits8, b32, c)
    return out["loss"][0].to(torch.float32)

  @staticmethod
  def backward(ctx, go):
    h2_16, w8, logits8, b32, c = ctx.saved_tensors
    out = K.rp_loss(logits8, b32, c, want_grad=True, go=go.to(torch.float32).reshape(1).contiguous())
    dz16 = out["dz16"]
    dh2 = K.gemm_bf16(dz16, w8, out_dtype=torch.bfloat16) if ctx.needs_input_grad[0] else None     # [N,8] . [7776,8]^T
    dw = _wgrad(h2_16, dz16)[:, :3].contiguous()
    return dh2, None, dw, out["db"], None


class CellGatherFn(torch.autograd.Function):
  """Maze-cell de-duplication (UnrealModel.dedup_cells): out[s] = table[cell(s)] for the samples' agent cells
  `pos` [S,2]; the backward pass is the segment sum of the per-sample gradient by cell (`unreal_cell_segment_sum`), in
  fp32 -- the table is handed over as fp32 so that autograd adds the towers' gradients in fp32 as well."""

  @staticmethod
  def forward(ctx, table32, pos):
    ctx.save_for_backward(pos)
    return K.cell_gather(table32.to(torch.bfloat16), pos)      # exact: the table holds bf16 values

  @staticmethod
  def backward(ctx, dout):
    (pos,) = ctx.saved_tensors
    return K.cell_segment_sum(dout.contiguous(), pos), None


class RpCellLossFn(torch.autograd.Function):
  """Reward prediction on maze cells (model.py:475-488, :571-575) without materialising the 7776 features of every
  sample: with G[c, f, :] = h2_table[c] . W_rp[f-th 2592-row block] (one 49-row tcgen05 GEMM against the [2592, 24]
  shadow `w24`), a sample's logits are G[cell of frame 0, 0] + G[cell of frame 1, 1] + G[cell of frame 2, 2].  Backward:
  d logits scattered into dG by (cell, frame), then two 49-row GEMMs give dh2_table and dW_rp."""

  @staticmethod
  def forward(ctx, h2t16, w24, w32, b32, idx3, c):
    g = K.gemm_bf16(h2t16, w24, b_mn_major=True).view(49, 3, 8)                     # f32
    logits8 = (g[idx3[:, 0], 0] + g[idx3[:, 1], 1] + g[idx3[:, 2], 2]).contiguous()
    out = K.rp_loss(logits8, b32, c, want_loss=True)
    ctx.save_for_backward(h2t16, w24, logits8, b32, idx3, c)
    return out["loss"][0].to(torch.float32)

  @staticmethod
  def backward(ctx, go):
    h2t16, w24, logits8, b32, idx3, c = ctx.saved_tensors
    out = K.rp_loss(logits8, b32, c, want_grad=True, go=go.to(torch.float32).reshape(1).contiguous())
    dz = out["dz16"].float()
    dg = torch.zeros(49, 3, 8, dtype=torch.float32, device=dz.device)
    for f in range(3):
      dg[:, f].index_add_(0, idx3[:, f], dz)
    dg16 = dg.view(49, 24).to(torch.bfloat16)
    dh = K.gemm_bf16(dg16, w24, out_dtype=torch.bfloat16)                            # [49,24] . [2592,24]^T
    dw24 = _wgrad(h2t16, dg16)                                                       # [2592, 24]
    dw = dw24.view(2592, 3, 8)[:, :, :3].permute(1, 0, 2).reshape(7776, 3)
    return dh, None, dw, out["db"], None, None
