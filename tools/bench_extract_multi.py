"""One tile's prior extraction over the GPUs of a box: ShardedPriorExtractor.add and finalize, run under torchrun.
Rank 0 prints one JSON line (and writes it to --out).

    python -m torch.distributed.run --nproc-per-node=G tools/bench_extract_multi.py [--chunks 24] [--tile-hits 28]
        [--out profiles/extract_multi_nG.json]

add(): random-init models of C2 and of the 16-sub-field shape (as tools/bench_extract.py builds them); `--chunks`
chunks of 2^17 rays in all, chunk i on rank i mod G.  Time: host clock from a barrier to the rank's last add() ended by a
device synchronise; rays/s per rank, and in total over the slowest rank's time.
finalize(): phases timed by wrapping the extractor's own steps with a device synchronise and a barrier on each side
(anchor + exchange, voxelize + threshold, gather); the slowest rank's time of each phase.  Bytes moved: the hits every
rank sent to other ranks (24 B each).  Memory: torch.cuda.max_memory_allocated per rank over add() and finalize().
Tile scale (--tile-hits log2 H, C2 model): H stored hits in all, H / G per rank, appended through the extractor's
own ps_hits_append in chunks of 2^20 (uniform in a 200 m x 200 m x 10 m box, colours random), then finalize().
On one GPU, PriorExtractor.finalize runs on a copy of the same store in the same process, and the two results are
compared as tests/test_gpu_tile_extract.assert_same_priors compares them (voxels, threshold and hit counts).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_extract import CHUNK, build, bundles, device_context  # noqa: E402

TILE_CHUNK = 1 << 20


def sync():
    torch.cuda.synchronize()
    dist.barrier()


def slowest(x: float) -> float:
    t = torch.tensor([x], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t)


def gather_ints(x: int):
    t = torch.tensor([x], device="cuda", dtype=torch.int64)
    out = [torch.zeros_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t)
    return [int(v) for v in out]


def timed_finalize(ex, dst=0):
    """finalize() with its steps timed (slowest rank) -> (result, {phase: s})."""
    raw = {}
    for name in ("_anchor", "_exchange", "_voxelize_owned", "_gather"):
        fn = getattr(ex, name)

        def wrap(*a, _fn=fn, _name=name):
            sync()
            t0 = time.perf_counter()
            r = _fn(*a)
            sync()
            raw[_name] = time.perf_counter() - t0
            return r
        setattr(ex, name, wrap)
    sync()
    t0 = time.perf_counter()
    res = ex.finalize(dst)
    sync()
    total = time.perf_counter() - t0
    t = {"exchange_s": slowest(raw["_anchor"] + raw["_exchange"]), "voxelize_s": slowest(raw["_voxelize_owned"]),
         "gather_s": slowest(raw["_gather"]), "finalize_s": slowest(total)}
    return res, {k: round(v, 4) for k, v in t.items()}


def same_store_reference(ex):
    """A PriorExtractor holding a copy of `ex`'s store (one GPU)."""
    from presight_b200.extract import PriorExtractor
    ref = PriorExtractor(ex.model, ex.pose_scale, ex.voxel_size, ex.hit_thr_ratio, ex.max_range_m, ex.z_range_m,
                         ex.chunk_rays, ex.block_hits, ex.insert_slice)
    ref._blocks = [(p.clone(), c.clone()) for p, c in ex._blocks]
    ref._sealed = list(ex._sealed)
    ref._cursor, ref._min, ref._status = ex._cursor.clone(), ex._min.clone(), ex._status.clone()
    return ref


def compare(got, want):
    return {"n_voxels_equal": got["n_voxels"] == want["n_voxels"],
            "hit_thr_equal": float(got["hit_thr"]) == float(want["hit_thr"]),
            "hits_equal": bool(torch.equal(got["hits"], want["hits"])),
            "features_equal": bool(torch.equal(got["features"], want["features"])),
            "points_max_abs_diff": float((got["points"] - want["points"]).abs().max()) if got["hits"].numel() else 0.0}


def finalize_record(ex, world):
    if not sum(gather_ints(ex.n_hits)):              # a random-init C2 field keeps (almost) no hit: nothing to time
        return {"stored_hits": 0, "not_measured": "no stored hit on any rank"}
    ref = same_store_reference(ex) if world == 1 else None     # resident during finalize(): in its peak on one GPU
    torch.cuda.reset_peak_memory_stats()
    stored = gather_ints(ex.n_hits)
    res, t = timed_finalize(ex)
    rec = {**t, "stored_hits_per_rank": stored, "stored_hits": sum(stored),
           "exchanged_bytes": sum(gather_ints(ex.exchanged_bytes)),
           "max_memory_allocated_bytes_per_rank": gather_ints(torch.cuda.max_memory_allocated())}
    if res is not None:
        rec.update({"voxels": res["n_voxels"], "kept_voxels": int(res["hits"].numel())})
    if ref is not None:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        want = ref.finalize()
        torch.cuda.synchronize()
        rec["prior_extractor_finalize_s"] = round(time.perf_counter() - t0, 4)
        rec["same_as_prior_extractor"] = compare(res, want)
    return rec


def run_shape(shape, n_chunks, rank, world, dev):
    from presight_b200 import synthetic
    from presight_b200.cameras.rays import RayBundle
    from presight_b200.extract import ShardedPriorExtractor
    model, _ = build(shape, dev)
    mine = [i for i in range(n_chunks) if i % world == rank]
    rbs = bundles(len(mine) + 1, dev, seed0=500 + 1000 * rank)
    fresh = lambda rb: RayBundle(origins=rb.origins, directions=rb.directions)
    ShardedPriorExtractor(model, synthetic.POSE_SCALE).add(fresh(rbs[0]))        # warm-up
    torch.cuda.reset_peak_memory_stats()
    ex = ShardedPriorExtractor(model, synthetic.POSE_SCALE)
    sync()
    t0 = time.perf_counter()
    for rb in rbs[1:]:
        ex.add(fresh(rb))
    torch.cuda.synchronize()
    t_add = time.perf_counter() - t0
    add_mem = gather_ints(torch.cuda.max_memory_allocated())
    rays = gather_ints(CHUNK * len(mine))
    per_rank = gather_ints(round(CHUNK * len(mine) / t_add))
    rec = {"add_rays_per_s_per_rank": per_rank, "add_rays_per_s_total": round(sum(rays) / slowest(t_add)),
           "add_s": round(slowest(t_add), 4), "rays": sum(rays), "add_max_memory_allocated_bytes_per_rank": add_mem}
    rec["finalize"] = finalize_record(ex, world)
    return rec


def run_tile(log2_h, rank, world, dev):
    from presight_b200 import synthetic
    from presight_b200.extract import ShardedPriorExtractor
    model, _ = build("c2", dev)
    H = 1 << log2_h
    lo, hi = H * rank // world, H * (rank + 1) // world
    ex = ShardedPriorExtractor(model, synthetic.POSE_SCALE, chunk_rays=TILE_CHUNK)
    g = torch.Generator(device=dev).manual_seed(77 + rank)
    box_lo = torch.tensor([-100.0, -100.0, -2.0], device=dev)
    box_ext = torch.tensor([200.0, 200.0, 10.0], device=dev)
    scale = torch.full((1, 3), synthetic.POSE_SCALE, device=dev)
    keep = torch.ones(TILE_CHUNK, device=dev, dtype=torch.uint8)
    dens = torch.full((TILE_CHUNK,), 2.0, device=dev)
    for i in range(lo, hi, TILE_CHUNK):
        n = min(TILE_CHUNK, hi - i)
        pm = box_lo + torch.rand(n, 3, device=dev, generator=g) * box_ext
        ps = (pm * scale).contiguous()
        ex._append(ps, ps / scale, keep[:n], dens[:n], torch.rand(n, 3, device=dev, generator=g))
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return finalize_record(ex, world)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chunks", type=int, default=24, help="chunks of 2^17 rays in all, over the ranks")
    ap.add_argument("--shapes", default="c2,presight")
    ap.add_argument("--tile-hits", type=int, default=28, help="log2 of the stored hits of the tile-scale finalize (0: skip)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_extract_multi needs CUDA devices (there is no CPU timing)")
    dist.init_process_group("nccl")
    rank, world = dist.get_rank(), dist.get_world_size()
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
    dev = torch.device("cuda", torch.cuda.current_device())
    rec = {"tool": "bench_extract_multi", **device_context(), "gpus": world,
           "note": "random-init fields; tile scale: synthetic stored hits, C2 model for finalize's query_priors"}
    for s in filter(None, args.shapes.split(",")):
        rec[s] = run_shape(s, args.chunks, rank, world, dev)
        torch.cuda.empty_cache()
    if args.tile_hits:
        rec[f"tile_2^{args.tile_hits}"] = run_tile(args.tile_hits, rank, world, dev)
    if rank == 0:
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(line + "\n")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
