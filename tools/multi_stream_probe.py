import os, sys, time, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, bench
from sdrtrunk_b200 import native
torch.cuda.set_device(0); native.init(0)
S = int(sys.argv[1])
ws = [bench.GpuWorkload("c4fm", r, 0) for r in range(S)]
for w in ws:
    for _ in range(3): w.step_device()
torch.cuda.synchronize()
t0 = time.perf_counter()
K = 10
for _ in range(K):
    for w in ws: w.step_device()
torch.cuda.synchronize()
dt = (time.perf_counter() - t0) / K
print("streams", S, "ms/step", dt * 1e3, "GS/s", S * ws[0].n_complex / dt / 1e9)
