"""Per-kernel timings of the `core` step (old [q ; p.M] read mode), to find a regression."""
import os, sys, time
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch
from pinthememory_b200 import capi, synth
from pinthememory_b200.memory import Memory_sup, _ReadFn, _WriteFn

dev = torch.device("cuda")
K, C, B, h, w, Hm, Wm = 19, 256, 8, 96, 96, 768, 768
mem = Memory_sup(K, C, C, 0.8, 1.0, False).to(dev)
x = synth.make_features(B, C, h, w, device=dev).requires_grad_(True)
f = synth.make_features(B, C, h, w, seed=5, device=dev).abs_().requires_grad_(True)
labels = synth.make_labels(B, Hm, Wm, K, "blocky", seed=2).to(dev)
Gu = synth.make_upstream_grad((B, 2 * C, h, w), device=dev)
gw = [torch.tensor(v, device=dev) for v in (0.02, 0.4, 0.2)]
M0 = mem.m_items.clone()


def step():
    x.grad = None
    f.grad = None
    u, _, _, rl, _ = _ReadFn.apply(x, M0, labels, None, None, 1.0, K)
    Mn, div, cls, _ = _WriteFn.apply(f, labels, M0, mem.clsfier.weight, mem.clsfier.bias, 0.8, K, None)
    torch.autograd.backward([u, rl, div, cls], [Gu, gw[0], gw[1], gw[2]])


for _ in range(5):
    step()
torch.cuda.synchronize()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
t0 = time.perf_counter()
a.record()
for _ in range(50):
    step()
b.record()
torch.cuda.synchronize()
print("core step: gpu %.3f ms, host %.3f ms" % (a.elapsed_time(b) / 50, (time.perf_counter() - t0) * 1e3 / 50))
capi.enable_kernel_timing(True)
capi.reset_counters()
for _ in range(20):
    step()
kt = capi.kernel_timings_ms()
print({k: round(sum(v) / len(v), 4) for k, v in kt.items()})
