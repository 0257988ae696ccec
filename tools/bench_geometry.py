"""Geometry metrics on one GPU: `ps_depth_metrics` per 1600 x 900 image with M = 2 maps (depth, expected_depth), as a
share of the C2 render time recorded in profiles/render_bench.json, and the nearest-neighbour grid (build, and both
query directions) for 2^24 prior points against 2^26 reference points at r = 0.4 m and 1.0 m.  Prints one JSON line.

    python tools/bench_geometry.py [--reps 20] [--log2-priors 24] [--log2-ref 26] [--out profiles/geometry_bench.json]

Depth metrics: CUDA events around 50 consecutive raw `ps_depth_metrics` calls (inputs and workspace prepared), median
of `--reps` windows; one call reads 12 B per pixel (two fp32 maps and the target; 17.3 MB, so it runs from L2 after
the first call); `geometry.depth_metrics` adds the stack of the maps and the allocations.  Clouds: synthetic
LiDAR-like scenes (ground rings around sensor positions and facades, tests/test_gpu_geometry.lidar_like) in a
200 m x 200 m tile; the reference with 2 cm noise, the priors with 5 cm noise.  How many points share a cell, which
sets the query cost, depends on the scene and r; a trained model's priors against real sweeps will differ.  Each
phase is timed by CUDA events around one call (the build includes its two host reads), median of three runs, the
first of which warms the phase up; points/s = points of the phase / its time.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(os.path.dirname(ROOT), "tests"))

from bench_extract import device_context  # noqa: E402
from test_geometry_host import depth_case  # noqa: E402
from test_gpu_geometry import lidar_like  # noqa: E402


def timed(fn, reps=3):
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts)


def bench_depth(dev, reps):
    from presight_b200 import _lib, geometry
    from presight_b200._lib import call, ptr, stream
    H, W, M = 900, 1600, 2
    preds, t = depth_case(H, W, M, seed=1)
    maps = [torch.from_numpy(p).to(dev) for p in preds]
    tgt = torch.from_numpy(t).to(dev)
    want = geometry.depth_metrics(maps, tgt, 0.0123)
    pred = torch.stack([m.reshape(-1) for m in maps]).contiguous()
    nbytes = C.c_int64(0)
    call("ps_depth_metrics_workspace", M, H * W, C.byref(nbytes))
    ws = torch.empty(int(nbytes.value), dtype=torch.uint8, device=dev)
    out = torch.empty(M, 8, dtype=torch.float64, device=dev)
    lib = _lib.load()

    def raw(n=50):
        for _ in range(n):
            lib.ps_depth_metrics(ptr(pred), M, H * W, ptr(tgt), 0.0123, None, 1.0, 75.0, ptr(ws), ptr(out), stream())

    raw(5)
    per_call = statistics.median(timed(raw, 1) / 50 for _ in range(reps))
    wrapper = statistics.median(timed(lambda: geometry.depth_metrics(maps, tgt, 0.0123), 1) for _ in range(reps))
    torch.cuda.synchronize()
    assert torch.equal(out, want)
    render = json.load(open(os.path.join(os.path.dirname(ROOT), "profiles", "render_bench.json")))
    render_ms = render["c2"]["chunk_32768"]["render_ms_per_image_median"]
    return {"H": H, "W": W, "M": M, "kernel_ms_per_image_median": round(per_call, 4),
            "depth_metrics_ms_per_image_median": round(wrapper, 4),
            "bytes_read_per_call": 12 * H * W, "c2_render_ms_per_image": render_ms,
            "fraction_of_c2_render_time": round(per_call / render_ms, 5),
            "ps_image_metrics_ms_per_image": render["c2"]["metrics_ms_per_image_median"]}


def bench_nn(dev, log2_p, log2_r, r):
    from presight_b200 import geometry
    Np, Nr = 1 << log2_p, 1 << log2_r
    ref = torch.from_numpy(lidar_like(Nr, 21, noise=0.02, extent=200.0)).to(dev)
    prior = torch.from_numpy(lidar_like(Np, 22, noise=0.05, extent=200.0)).to(dev)
    taus = (0.05, 0.1, 0.2) if r < 1 else (0.1, 0.2, 0.5)
    rec = {"r_m": r, "taus_m": list(taus), "prior_points": Np, "reference_points": Nr}
    for name, pts, qs in (("ref_grid", ref, prior), ("prior_grid", prior, ref)):
        holder = {}
        build_ms = timed(lambda: holder.__setitem__("g", geometry.NNGrid(pts, r)))
        g = holder["g"]
        query_ms = timed(lambda: g.query(qs, taus))
        rec[name] = {"build_ms": round(build_ms, 3), "build_points_per_s": round(pts.shape[0] / build_ms * 1e3),
                     "occupied_cells": g.n_cells, "mean_points_per_cell": round(pts.shape[0] / g.n_cells, 2),
                     "query_points": int(qs.shape[0]), "query_ms": round(query_ms, 3),
                     "query_points_per_s": round(qs.shape[0] / query_ms * 1e3),
                     "device_memory_bytes": int(g.points.numel() * 4 + g.cell_keys.numel() * 8
                                                + g.cell_ranges.numel() * 4)}
        del g, holder
    a = geometry.prior_geometry_metrics(prior, ref, r, taus)
    b = geometry.prior_geometry_metrics(prior, ref, r, taus)
    rec["repeat_bit_identical"] = all(torch.equal(a[k], b[k]) for k in a)
    rec["scores"] = {k: (float(v) if v.dim() == 0 else [round(x, 6) for x in v.tolist()]) for k, v in a.items()}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--log2-priors", type=int, default=24)
    ap.add_argument("--log2-ref", type=int, default=26)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_geometry needs a GPU")
    dev = torch.device("cuda")
    res = {"tool": "bench_geometry", **device_context(), "depth_metrics": bench_depth(dev, a.reps)}
    res["nn"] = [bench_nn(dev, a.log2_priors, a.log2_ref, r) for r in (0.4, 1.0)]
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
