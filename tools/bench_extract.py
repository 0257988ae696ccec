"""Prior extraction from camera rays: the eval depth pass old (`get_depth_for_camera_ray_bundle`, per-operator final
level) against new (`get_surface_hits`, fused density level), and the whole extractor (`PriorExtractor.add` +
`finalize`), on random-init models of C2 and of PreSight's shipped shape (16 sub-fields).  Prints one JSON line.

    python tools/bench_extract.py [--chunks 24] [--warmup 3] [--out profiles/extract_bench.json]

Rays: `synthetic.make_rays`, chunks of 2^17 rays (the reference's chunk), each timed chunk a different set of rays.
Times: CUDA events around each chunk after a warm-up, median over the timed chunks.  HBM fraction: the algorithmic
bytes of the depth pass (`synthetic.depth_pass_bytes_per_ray`) over the project's measured copy bandwidth.
Random-init fields do not concentrate the samples on surfaces the way a trained scene does, so the proposal levels'
resampling and the kept-hit count differ from a real tile; the numbers are rates of these inputs, not of a city scan.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_GBS = 6554.9          # measured bf16 copy bandwidth of one B200 (BASELINE.md)
CHUNK = 1 << 17


def device_context():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip()
    except Exception as e:                     # the number stays unlabelled rather than wrong
        out = f"unavailable ({type(e).__name__})"
    return {"device": name, "power_limit_and_max_sm_clock": out}


def build(shape: str, dev):
    from presight_b200 import synthetic
    from presight_b200.model import NerfactoNuscMSModel
    torch.manual_seed(0)
    if shape == "c2":
        cfg = synthetic.config_c2("b200")
        cen, aabbs = torch.zeros(1, 3), synthetic.tile_aabb()
    else:
        cfg = synthetic.config_presight("b200")
        cen, aabbs = synthetic.sub_field_layout(16)
    model = NerfactoNuscMSModel(cfg, cen, aabbs)
    with torch.no_grad():                      # init-scale tables give a featureless field (as smoke() does)
        for name, p in model.named_parameters():
            if name.endswith("hash_table"):
                p.mul_(300.0)
    return model.to(dev).eval(), cfg


def bundles(n_chunks: int, dev, seed0: int):
    from presight_b200 import synthetic
    from presight_b200.cameras.rays import RayBundle
    out = []
    for i in range(n_chunks):
        h = synthetic.make_rays(CHUNK, seed=seed0 + i)
        out.append(RayBundle(origins=h["origins"].to(dev), directions=h["directions"].to(dev)))
    return out


def timed(fn, items, warmup):
    for it in items[:warmup]:
        fn(it)
    torch.cuda.synchronize()
    ms = []
    for it in items[warmup:]:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn(it)
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return statistics.median(ms), ms


def run_shape(shape: str, n_chunks: int, warmup: int, dev):
    from presight_b200 import synthetic
    from presight_b200.cameras.rays import RayBundle
    from presight_b200.extract import PriorExtractor
    model, cfg = build(shape, dev)
    model.config.eval_num_rays_per_chunk = CHUNK          # the reference's chunk for get_depth_for_camera_ray_bundle
    rbs = bundles(n_chunks + warmup, dev, seed0=100)
    assert model.field.supports_level_depth(cfg.num_nerf_samples_per_ray)

    def fresh(rb):
        return RayBundle(origins=rb.origins, directions=rb.directions)
    with torch.no_grad():
        old_ms, _ = timed(lambda rb: model.get_depth_for_camera_ray_bundle(fresh(rb)), rbs, warmup)
        new_ms, _ = timed(lambda rb: model.get_surface_hits(fresh(rb)), rbs, warmup)
        agree = []
        for rb in rbs[warmup:]:
            a = model.get_depth_for_camera_ray_bundle(fresh(rb))["depth"]
            b = model.get_surface_hits(fresh(rb))["depth"]
            agree.append(float(((a - b).abs() <= 1e-4 * a.abs().max()).float().mean()))
    # end to end: add every timed chunk, then finalize; hits kept per ray reported for context
    for rb in rbs[:warmup]:
        ex = PriorExtractor(model, synthetic.POSE_SCALE)
        ex.add(fresh(rb))
    torch.cuda.synchronize()
    ex = PriorExtractor(model, synthetic.POSE_SCALE)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for rb in rbs[warmup:]:
        ex.add(fresh(rb))
    res = ex.finalize()
    b.record()
    b.synchronize()
    e2e_ms = a.elapsed_time(b)
    n_rays = CHUNK * n_chunks
    bpr = synthetic.depth_pass_bytes_per_ray(cfg)
    bound_rays_s = HBM_GBS * 1e9 / bpr
    new_rays_s = CHUNK / (new_ms * 1e-3)
    return {
        "depth_pass_bytes_per_ray": bpr,
        "old_get_depth_ms_per_chunk": round(old_ms, 3), "old_rays_per_s": round(CHUNK / (old_ms * 1e-3)),
        "new_surface_hits_ms_per_chunk": round(new_ms, 3), "new_rays_per_s": round(new_rays_s),
        "speedup": round(old_ms / new_ms, 3),
        "hbm_bound_rays_per_s": round(bound_rays_s), "new_fraction_of_hbm_bound": round(new_rays_s / bound_rays_s, 4),
        "threshold_depth_agreement_min": round(min(agree), 5), "threshold_depth_agreement_mean": round(sum(agree) / len(agree), 5),
        "extractor_e2e_ms": round(e2e_ms, 2), "extractor_e2e_rays_per_s": round(n_rays / (e2e_ms * 1e-3)),
        "kept_hits": ex.n_hits, "voxels": int(res["n_voxels"]), "timed_chunks": n_chunks, "rays_per_chunk": CHUNK,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chunks", type=int, default=24)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="c2,presight")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert args.chunks >= 20, "the median is taken over at least 20 chunks"
    if not torch.cuda.is_available():
        raise SystemExit("bench_extract needs a CUDA device (there is no CPU timing)")
    dev = torch.device("cuda:0")
    rec = {"tool": "bench_extract", **device_context(),
           "note": "random-init fields: samples are not concentrated on surfaces as in a trained scene"}
    for s in args.shapes.split(","):
        rec[s] = run_shape(s, args.chunks, args.warmup, dev)
        torch.cuda.empty_cache()
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
