import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from unreal_b200 import kernels as K
dev = torch.device("cuda", 0)
n = int(sys.argv[1]) if len(sys.argv) > 1 else 8192
g = torch.Generator(device=dev).manual_seed(0)
kx, kc = 264, 520
xh = torch.randn(2, n, kc, device=dev, generator=g).to(torch.bfloat16)
w = (torch.randn(kc, 1024, device=dev, generator=g) * 0.05).to(torch.bfloat16)
b = torch.zeros(1024, device=dev)
nt = (n + 31) // 32 * 32
c0 = torch.zeros(nt, 256, device=dev); c1 = torch.zeros(nt, 256, device=dev)
h = torch.empty(n, 256, device=dev); acts = torch.empty(nt, 1024, device=dev, dtype=torch.bfloat16)
def timed(fn, reps=50):
  for _ in range(5): fn()
  torch.cuda.synchronize()
  s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  s.record()
  for _ in range(reps): fn()
  e.record(); torch.cuda.synchronize()
  return round(s.elapsed_time(e) * 1e3 / reps, 2)
f_full = lambda: K.lstm_step_fwd(xh[0], w, b, c0, c1, h_out=h, h16_out=xh[1, :, kx:], acts=acts, tiled=True)
f_half = lambda: K.lstm_step_fwd(xh[0, :, kx:], w[kx:], b, c0, c1, h_out=h, h16_out=xh[1, :, kx:], acts=acts, tiled=True)
hc = xh[0, :, kx:].contiguous(); wc = w[kx:].contiguous()
f_half_c = lambda: K.lstm_step_fwd(hc, wc, b, c0, c1, h_out=h, h16_out=xh[1, :, kx:], acts=acts, tiled=True)
res = {"envs": n}
for name, fn in (("k520", f_full), ("k256_view", f_half), ("k256_contiguous", f_half_c), ("k520_again", f_full)):
  res[name + "_eager_us"] = timed(fn)
  gr = torch.cuda.CUDAGraph()
  with torch.cuda.graph(gr):
    for _ in range(20): fn()
  res[name + "_graph_us"] = round(timed(gr.replay, reps=10) / 20, 2)
print(json.dumps(res))
