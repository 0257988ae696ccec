"""Rendering whole camera images and scoring them: `get_outputs_for_camera_ray_bundle` on 1600 x 900 images at two
chunk sizes, and `ps_image_metrics` (PSNR + SSIM) per image, on random-init models of C2 and of PreSight's shipped shape
(16 sub-fields).  Prints one JSON line.

    python tools/bench_render.py [--frames 2] [--out profiles/render_bench.json]

Images: every camera of the first `--frames` frames of `synthetic.make_cameras` (6 per frame), rays from
`RayGenerator.image_rays`, generated before the timed window.  Render time: CUDA events around each image's
`get_outputs_for_camera_ray_bundle`, median over the images after one warm-up image, with `eval_num_rays_per_chunk` at
the config default (2^15) and at 2^17.  HBM fraction: the forward hash bytes of the render pass, which are those of the
depth pass (`synthetic.depth_pass_bytes_per_ray`), over the project's measured copy bandwidth.  Metrics time: CUDA events
around `metrics.image_metrics` on one (render, random target) pair, cycling over all the rendered images so that the
35 MB a pair reads mostly comes from HBM rather than L2 (the images together exceed the 126 MB L2 from 4 images up).
Random-init fields do not concentrate samples on surfaces the way a trained scene does; the numbers are rates of these
inputs, not of a city scan.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench_extract import HBM_GBS, build, device_context  # noqa: E402

CHUNKS = (1 << 15, 1 << 17)
METRIC_REPS = 60


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def run_shape(shape: str, n_frames: int, dev):
    from presight_b200 import metrics, synthetic
    from presight_b200.cameras.ray_generator import RayGenerator
    model, cfg = build(shape, dev)
    cams = synthetic.make_cameras(seed=42, n_frames=n_frames)
    H, W = cams["H"], cams["W"]
    gen = RayGenerator(cams["camera_to_worlds"], cams["fx"], cams["fy"], cams["cx"], cams["cy"]).to(dev)
    n_img = cams["camera_to_worlds"].shape[0]
    bundles = [gen.image_rays(i, H, W) for i in range(n_img)]
    bpr = synthetic.depth_pass_bytes_per_ray(cfg)
    bound_rays_s = HBM_GBS * 1e9 / bpr
    rec = {"images": n_img, "timed_images": n_img - 1, "H": H, "W": W, "depth_pass_bytes_per_ray": bpr,
           "hbm_bound_rays_per_s": round(bound_rays_s)}
    renders = None
    for chunk in CHUNKS:
        model.config.eval_num_rays_per_chunk = chunk
        outs, ms = [], []
        for i, rb in enumerate(bundles):
            box = {}
            t = event_ms(lambda: box.update(out=model.get_outputs_for_camera_ray_bundle(rb)))
            outs.append(box["out"]["rgb"])
            if i > 0:                                # image 0 warms this chunk size up
                ms.append(t)
        med = statistics.median(ms)
        rays_s = H * W / (med * 1e-3)
        rec[f"chunk_{chunk}"] = {"render_ms_per_image_median": round(med, 3), "render_ms_min": round(min(ms), 3),
                                 "render_ms_max": round(max(ms), 3), "rays_per_s": round(rays_s),
                                 "fraction_of_hbm_bound": round(rays_s / bound_rays_s, 4)}
        if renders is None:
            renders = outs
        else:                                        # the chunk size changes only the per-chunk expected-depth clip
            rec[f"chunk_{chunk}"]["rgb_equal_to_chunk_{}".format(CHUNKS[0])] = all(
                torch.equal(a, b) for a, b in zip(renders, outs))
        del outs
    g = torch.Generator(device=dev).manual_seed(0)
    targets = [torch.rand(H, W, 3, device=dev, generator=g) for _ in range(n_img)]
    metrics.image_metrics(renders[0], targets[0])     # warm-up
    torch.cuda.synchronize()
    ms = [event_ms(lambda: metrics.image_metrics(renders[i % n_img], targets[i % n_img])) for i in range(METRIC_REPS)]
    met = statistics.median(ms)
    render_default = rec[f"chunk_{CHUNKS[0]}"]["render_ms_per_image_median"]
    rec["metrics_ms_per_image_median"] = round(met, 4)
    rec["metrics_fraction_of_render_time"] = round(met / render_default, 5)
    rec["metrics_bytes_per_image_min"] = 2 * H * W * 3 * 4
    rec["metrics_effective_gb_per_s"] = round(2 * H * W * 3 * 4 / (met * 1e-3) / 1e9, 1)
    psnr, ssim, _ = metrics.image_metrics(renders[1], targets[1])
    rec["example_psnr_ssim_vs_random_target"] = [round(float(psnr[0]), 4), round(float(ssim[0]), 6)]
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=2)
    ap.add_argument("--shapes", default="c2,presight")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert args.frames >= 1
    if not torch.cuda.is_available():
        raise SystemExit("bench_render needs a CUDA device (there is no CPU timing)")
    dev = torch.device("cuda:0")
    rec = {"tool": "bench_render", **device_context(),
           "note": "random-init fields: samples are not concentrated on surfaces as in a trained scene"}
    for s in args.shapes.split(","):
        with torch.no_grad():
            rec[s] = run_shape(s, args.frames, dev)
        torch.cuda.empty_cache()
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
