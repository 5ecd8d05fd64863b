"""oracle/model_oracle.py's ModelOracle with the split-bf16 encoder of UnrealModel(encoder_precision='bf16x3').

With `encoder_split=True` the forward operands of conv1 and conv2 (frames, filters, conv1's output) are hi + lo bf16
pairs, hi = bf16(a), lo = bf16(a - hi), instead of bf16 values; the backward pass is unchanged: with `emulate_bf16` it
reads the bf16 operands, as the CUDA path's backward kernels read the hi halves, and rounds the encoder's gradients to
bf16 where the CUDA path stores them.  `encoder_split=False` is ModelOracle itself.
"""
import torch
import torch.nn.functional as F

from oracle import model_oracle as M


def pair(x):
  """x rounded to a split-bf16 pair hi + lo (a constant: no gradient)."""
  x = x.detach()
  hi = x.to(torch.bfloat16).to(x.dtype)
  return hi + (x - hi).to(torch.bfloat16).to(x.dtype)


class SplitEncoderOracle(M.ModelOracle):
  def __init__(self, *args, encoder_split=False, **kwargs):
    super().__init__(*args, **kwargs)
    self.split = encoder_split

  def encoder(self, images):
    if not self.split:
      return super().encoder(images)
    x = images.to(self.dtype).permute(0, 3, 1, 2)
    h1 = F.relu(self._pair_conv(x, "W_base_conv1", "b_base_conv1", 4))
    h1q = M._bf16(h1, self.q)                                # the gradient at h1 as the bf16 path rounds it
    h1 = h1q + (pair(h1) - h1q).detach()
    h2 = F.relu(self._pair_conv(h1, "W_base_conv2", "b_base_conv2", 2))
    return M._bf16(h2.permute(0, 2, 3, 1), self.q)

  def _pair_conv(self, x, wname, bname, stride):
    """conv2d whose value is that of the hi + lo operand pairs and whose gradient is that of the (emulate_bf16) operands."""
    y = F.conv2d(M._bf16(x, self.q), self.w(wname).permute(3, 2, 0, 1), self.p[bname], stride=stride)
    with torch.no_grad():
      ys = F.conv2d(pair(x), pair(self.p[wname]).permute(3, 2, 0, 1), self.p[bname], stride=stride)
    return y + (ys - y).detach()
