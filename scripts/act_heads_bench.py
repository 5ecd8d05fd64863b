import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from unreal_b200 import kernels as K
dev = torch.device("cuda", 0)
n, a = 8192, 4
g = torch.Generator(device=dev).manual_seed(0)
gates = torch.randn(n, 1024, device=dev, generator=g).to(torch.bfloat16)
c = torch.randn(n, 256, device=dev, generator=g); h = torch.randn(n, 256, device=dev, generator=g)
wp = torch.randn(256, a, device=dev, generator=g) * 0.1; bp = torch.zeros(a, device=dev)
wv = torch.randn(256, device=dev, generator=g) * 0.1; bv = torch.zeros(1, device=dev)
act = torch.ones(n, device=dev, dtype=torch.uint8)
hout = torch.empty(n, 256, device=dev)
def timed(fn, reps=50):
  for _ in range(5): fn()
  torch.cuda.synchronize()
  s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  s.record()
  for _ in range(reps): fn()
  e.record(); torch.cuda.synchronize()
  return round(s.elapsed_time(e) * 1e3 / reps, 2)
def pair():
  K.lstm_cell_act(gates, c, h, hout, act)
  K.a3c_head(hout, wp, bp, wv, bv, want_pi=True, want_v=True)
print(json.dumps({"cell": timed(lambda: K.lstm_cell_act(gates, c, h, hout, act)), "pair": timed(pair),
                  "fused": timed(lambda: K.lstm_cell_act_heads(gates, c, h, wp, bp, wv, bv, act))}))
