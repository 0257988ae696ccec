#!/usr/bin/env python
"""Do the field kernels and the hash kernels really co-run?  Times each alone and both on two streams."""
import ctypes as C, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from presight_b200 import fused, ops, synthetic
from presight_b200._lib import call, ptr, host_floats, host_field_net

dev = "cuda"
n, S, L, F, log2T, A = 32768, 64, 16, 2, 22, 16
g = torch.Generator().manual_seed(0)
rays = synthetic.make_rays(n, seed=1)
o, d = rays["origins"].to(dev), rays["directions"].to(dev)
aabb = [float(v) for v in synthetic.tile_aabb().reshape(-1)]
gg = np.exp((np.log(2048) - np.log(16)) / (L - 1))
grid = fused.GridMeta(tuple(float(np.floor(16 * gg ** l)) for l in range(L)), log2T, F)
table = ((torch.rand(L << log2T, F, generator=g) * 2 - 1) * 1e-3).to(dev)
dims = [(L * F, 64, 80), (64, 64, 64, 64), (31 + A, 64, 64, 3)]
ws, bs = [], []
for dd in dims:
    for i in range(len(dd) - 1):
        ws.append((torch.randn(dd[i + 1], dd[i], generator=g) / dd[i] ** 0.5).to(dev))
        bs.append(torch.zeros(dd[i + 1], device=dev))
eu = (torch.rand(n, S + 1, generator=g) * (40.0 / S) + 0.001).cumsum(-1).to(dev)
app = torch.randn(n, A, generator=g).to(dev)
x01, sel = fused._ray_points(o, d, eu, aabb, True)
feat = fused._hash_fwd(x01, table, grid, level_major=True)
P = n * S
w = torch.empty(n, S, device=dev); rgb = torch.empty(n, 3, device=dev); acc = torch.empty(n, 1, device=dev)
dexp = torch.empty(n, 1, device=dev); dthr = torch.empty(n, 1, device=dev); sem = torch.empty(n, 64, device=dev)
dW = [torch.zeros_like(t) for t in ws]; dB = [torch.zeros_like(t) for t in bs]
net = host_field_net(ws, bs, A, dW, dB)
dfeat = torch.empty_like(feat); dtable = torch.zeros_like(table)
dw = torch.randn(n, S, device=dev) * 1e-3; drgb = torch.randn(n, 3, device=dev); dsem = torch.randn(n, 64, device=dev) * 0.1
dacc = torch.zeros(n, 1, device=dev); ddexp = torch.zeros(n, 1, device=dev)
s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()


def field_fwd(st):
    call("ps_field_level_fwd", C.byref(net), ptr(feat), L, F, ptr(sel), ptr(eu), ptr(d), ptr(app), n, S, 0.5, ptr(w), ptr(rgb),
         ptr(acc), ptr(dexp), ptr(dthr), ptr(sem), None, st.cuda_stream)


def field_bwd(st):
    call("ps_field_level_bwd", C.byref(net), ptr(feat), L, F, ptr(sel), ptr(eu), ptr(d), ptr(app), n, S, ptr(acc), ptr(dexp),
         ptr(dw), ptr(drgb), ptr(dacc), ptr(ddexp), ptr(dsem), ptr(dfeat), None, st.cuda_stream)


def hash_fwd(st):
    call("ps_hash_fwd_lm", ptr(x01), P, ptr(table), host_floats(grid.scalings), L, F, log2T, ptr(feat), st.cuda_stream)


def hash_bwd(st):
    call("ps_hash_bwd_lm", ptr(x01), P, None, host_floats(grid.scalings), L, F, log2T, ptr(dfeat), ptr(dtable), None,
         st.cuda_stream)


def timed(fns):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    s1.wait_stream(torch.cuda.current_stream()); s2.wait_stream(torch.cuda.current_stream())
    ends = []
    for fn, st in fns:
        fn(st)
        e = torch.cuda.Event(enable_timing=True)
        e.record(st)
        ends.append(e)
    torch.cuda.current_stream().wait_stream(s1); torch.cuda.current_stream().wait_stream(s2)
    b.record(); torch.cuda.synchronize()
    timed.ends = [a.elapsed_time(e) for e in ends]          # when each kernel finished
    return a.elapsed_time(b)


for fn in (field_fwd, field_bwd, hash_fwd, hash_bwd):
    fn(s1)
torch.cuda.synchronize()
for name, fns in [("field_fwd", [(field_fwd, s1)]), ("hash_fwd", [(hash_fwd, s2)]), ("field_fwd || hash_fwd", [(field_fwd, s1), (hash_fwd, s2)]),
                  ("field_bwd", [(field_bwd, s1)]), ("hash_bwd", [(hash_bwd, s2)]), ("field_bwd || hash_bwd", [(field_bwd, s1), (hash_bwd, s2)]),
                  ("hash_bwd || field_bwd (hash first)", [(hash_bwd, s2), (field_bwd, s1)])]:
    ts = [timed(fns) for _ in range(3)]
    print(f"{name:40s} {min(ts):.3f} ms   (kernel end times of the last run: {', '.join(f'{t:.3f}' for t in timed.ends)})")
