#!/usr/bin/env python
"""Micro-benchmark of the fused MLP kernels: forward (and backward) per shape and precision at P points."""
import argparse, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from presight_b200 import ops

def timeit(fn, iters=5):
    fn(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters): fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / iters

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", type=int, default=65536 * 64)
    ap.add_argument("--precs", default="0,1")
    ap.add_argument("--bwd", action="store_true")
    args = ap.parse_args()
    P = args.points
    g = torch.Generator().manual_seed(0)
    for (n_in, hidden, n_layers, n_out, act) in [(64, 64, 3, 64, 0), (32, 64, 2, 80, 0), (8, 64, 2, 1, 0), (48, 64, 3, 3, 2)]:
        dims = [n_in] + [hidden] * (n_layers - 1) + [n_out]
        ws = [(torch.randn(dims[i + 1], dims[i], generator=g) / np.sqrt(dims[i])).cuda().requires_grad_(True) for i in range(n_layers)]
        bs = [(torch.randn(dims[i + 1], generator=g) * 0.1).cuda().requires_grad_(True) for i in range(n_layers)]
        x = torch.randn(P, n_in, device="cuda")
        flops = 2 * P * sum(dims[i] * dims[i + 1] for i in range(n_layers))
        for prec in [int(p) for p in args.precs.split(",")]:
            with torch.no_grad():
                t = timeit(lambda: ops.mlp(x, ws, bs, act, prec))
            line = f"{'x'.join(map(str, dims)):16s} prec={prec} fwd {t:7.3f} ms {flops / t / 1e9:8.1f} TFLOP/s"
            if args.bwd:
                xg = x.clone().requires_grad_(True)
                y = ops.mlp(xg, ws, bs, act, prec)
                dy = torch.randn_like(y)
                tb = timeit(lambda: torch.autograd.grad(y, [xg, *ws], dy, retain_graph=True))
                line += f" | bwd {tb:7.3f} ms {3 * flops / tb / 1e9:8.1f} TFLOP/s (fwd recompute not counted)"
            print(line, flush=True)

if __name__ == "__main__":
    main()
