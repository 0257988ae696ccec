"""Prior extraction of a whole tile in bounded memory: `PriorExtractor.add` (ps_hits_append) against the per-chunk tail
it replaced (nonzero, two gathers, a zeros tensor and ps_voxel_min_bound), and `TileVoxelizer` over 2^28 and 2^30
synthetic hits.  Prints one JSON line.

    python tools/bench_extract_tile.py [--chunks 24] [--warmup 3] [--hits 28,30] [--out profiles/extract_tile_bench.json]

add(): random-init models of C2 and of the 16-sub-field shape (as tools/bench_extract.py builds them), chunks of 2^17
rays, each chunk timed with CUDA events through the old tail and through `add()` in alternating order; median over the
chunks.  The two stores are compared bit for bit at the end.
TileVoxelizer: point i lies in voxel floor(k^2 / 2^(2 log2 H - 19)) of a 128 x 128 x 32 lattice, k = i * A mod H, so
all 2^19 voxels are hit, from ~H / 2^20 to ~2^(log2 H / 2 + 4.5) times; features and colours are gathered from a
per-voxel table in each slice (standing in for query_priors).  Times: host clock around each phase, ended by a device
synchronise.  Peak: torch.cuda.max_memory_allocated over the voxelizer's lifetime minus the resident points.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_extract import CHUNK, build, bundles, device_context  # noqa: E402


class OldTail:
    """The parent commit's PriorExtractor.add after query_priors, restated: nonzero, gathers, zeros, min_bound."""

    def __init__(self):
        self.points, self.colors, self.min = [], [], None

    @torch.no_grad()
    def add(self, ex, rb):
        from presight_b200.cameras.rays import RayBundle
        from presight_b200.extract import surface_hits
        from presight_b200.priors import PriorVoxelizer
        o, d = rb.origins, rb.directions
        depth = ex.model.get_surface_hits(RayBundle(origins=o, directions=d))["depth"]
        ps, pm, keep = surface_hits(o, d, depth, ex.pose_scale, ex.max_range_m, ex.z_range_m)
        dens, _ = ex.model.query_priors(ps)
        idx = torch.nonzero(keep & (dens > 1)).view(-1)
        self.points.append(ps[idx])
        self.colors.append(torch.zeros(idx.numel(), 3, device=ps.device).to(torch.float32).contiguous())
        self.min = PriorVoxelizer.min_bound(pm[idx], None, self.min)


def time_add(shape, n_chunks, warmup, dev):
    from presight_b200 import synthetic
    from presight_b200.cameras.rays import RayBundle
    from presight_b200.extract import PriorExtractor
    model, _ = build(shape, dev)
    rbs = bundles(n_chunks + warmup, dev, seed0=300)
    fresh = lambda rb: RayBundle(origins=rb.origins, directions=rb.directions)
    old, ex = OldTail(), PriorExtractor(model, synthetic.POSE_SCALE)
    for rb in rbs[:warmup]:
        OldTail().add(ex, fresh(rb))
        PriorExtractor(model, synthetic.POSE_SCALE).add(fresh(rb))
    torch.cuda.synchronize()
    ms = {"old": [], "new": []}
    for i, rb in enumerate(rbs[warmup:]):
        runs = [("old", lambda: old.add(ex, fresh(rb))), ("new", lambda: ex.add(fresh(rb)))]
        for name, fn in (runs if i % 2 == 0 else runs[::-1]):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ms[name].append(a.elapsed_time(b))
    same = (torch.equal(torch.cat(old.points), torch.cat(ex._points)) and torch.equal(old.min, ex._min))
    o, n = statistics.median(ms["old"]), statistics.median(ms["new"])
    return {"old_tail_ms_per_chunk": round(o, 3), "add_ms_per_chunk": round(n, 3),
            "old_tail_rays_per_s": round(CHUNK / (o * 1e-3)), "add_rays_per_s": round(CHUNK / (n * 1e-3)),
            "add_over_old_time": round(n / o, 4), "stores_identical": bool(same), "kept_hits": ex.n_hits,
            "timed_chunks": n_chunks, "rays_per_chunk": CHUNK}


def time_voxelizer(log2_h, dev):
    from presight_b200.priors import TileVoxelizer
    H, V, C, vs, A = 1 << log2_h, 1 << 19, 64, 0.4, 0x9E3779B1
    P_ins, P_acc = 1 << 24, 1 << 22
    shift = 2 * log2_h - 19

    def voxel_of(i0, n):
        k = (torch.arange(i0, i0 + n, device=dev, dtype=torch.int64) * A) & (H - 1)
        return (k * k) >> shift

    def cell(vid):
        return torch.stack([vid & 127, (vid >> 7) & 127, vid >> 14], 1)

    torch.cuda.empty_cache()
    g = torch.Generator(device=dev).manual_seed(0)
    feat_tab = torch.rand(V, C, device=dev, generator=g).half()
    col_tab = torch.rand(V, 3, device=dev, generator=g)
    pts = torch.empty(H, 3, device=dev)
    for i0 in range(0, H, P_ins):
        jit = torch.rand(P_ins, 3, device=dev, generator=g) * 0.8 + 0.1
        pts[i0:i0 + P_ins] = -1.2 + vs * (cell(voxel_of(i0, P_ins)).float() + jit)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t = {}
    t0 = time.perf_counter()
    vox = TileVoxelizer(torch.zeros(3, device=dev), vs, C)
    for i0 in range(0, H, P_ins):
        vox.insert(pts[i0:i0 + P_ins])
    torch.cuda.synchronize()
    t["insert_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    vox.seal()
    torch.cuda.synchronize()
    t["seal_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    for i0 in range(0, H, P_acc):
        vid = voxel_of(i0, P_acc)
        vox.accumulate(pts[i0:i0 + P_acc], feat_tab[vid], col_tab[vid])
    torch.cuda.synchronize()
    t["accumulate_s"] = time.perf_counter() - t0
    hits_total = int(vox.counts.long().sum())
    t0 = time.perf_counter()
    out = vox.finalize(0.2)
    torch.cuda.synchronize()
    t["finalize_s"] = time.perf_counter() - t0
    peak = torch.cuda.max_memory_allocated() - base
    rec = {k: round(v, 3) for k, v in t.items()}
    rec.update({"hits": H, "hits_accumulated": hits_total, "voxels": out["n_voxels"], "kept_voxels": int(out["hits"].numel()),
                "total_s": round(sum(t.values()), 3), "hits_per_s": round(H / sum(t.values())),
                "resident_points_bytes": H * 12, "peak_beyond_points_bytes": int(peak),
                "table_capacity": vox.capacity, "insert_slice": P_ins, "accumulate_slice": P_acc,
                "points_sized_table_bytes_for_comparison": 740 * 2 * H})
    del vox, out, pts
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chunks", type=int, default=24)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="c2,presight")
    ap.add_argument("--hits", default="28,30", help="log2 of the synthetic hit counts for TileVoxelizer")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert args.chunks >= 20, "the median is taken over at least 20 chunks"
    if not torch.cuda.is_available():
        raise SystemExit("bench_extract_tile needs a CUDA device (there is no CPU timing)")
    dev = torch.device("cuda:0")
    rec = {"tool": "bench_extract_tile", **device_context(),
           "note": "add(): random-init fields; TileVoxelizer: synthetic hits with a per-voxel feature table"}
    for s in filter(None, args.shapes.split(",")):
        rec[f"add_{s}"] = time_add(s, args.chunks, args.warmup, dev)
        torch.cuda.empty_cache()
    for h in filter(None, args.hits.split(",")):
        rec[f"tile_voxelizer_2^{int(h)}"] = time_voxelizer(int(h), dev)
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
