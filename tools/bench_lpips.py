"""LPIPS of evaluation images: `metrics.LPIPS` (`ps_lpips`) per 1600 x 900 pair at B = 1 and B = 6 (one frame's six
cameras), its kernels one by one, the same definition through F.conv2d (cuDNN, TF32: what torchmetrics costs on the
device), and one C2 render at the default chunk for LPIPS's share of an evaluation image.  Prints one JSON line.

    python tools/bench_lpips.py [--reps 30] [--out profiles/lpips_bench.json]

Weights: seeded random AlexNet / lin weights (the time does not depend on their values).  Images: six C2 renders of the
first frame of `synthetic.make_cameras` (random-init field) against random targets.  Pair time: CUDA events around each
call, median over `--reps` calls after a warm-up, B = 1 cycling over the six pairs.  A pair's activations (~140 MB)
exceed the 126 MB L2, so each call mostly starts from HBM.  Kernel times: torch.profiler with CUDA activities in a pass
of its own (after the timed passes), mean per call.  FLOPs: `metrics.lpips_flops` (multiply-adds x 2 of the five
convolutions, 82.0 G per 1600 x 900 pair); the TF32 rate is set against NVIDIA's data-sheet figure for one B200,
1,125 TFLOP/s dense, which is not a measured peak.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from bench_extract import build, device_context  # noqa: E402
from bench_render import event_ms  # noqa: E402

TF32_DATASHEET_TFLOPS = 1125.0
SHIFT = (-0.030, -0.088, -0.188)
SCALE = (0.458, 0.448, 0.450)
LAYERS = ((0, 4, 2, False), (3, 1, 2, True), (6, 1, 1, True), (8, 1, 1, False), (10, 1, 1, False))


def random_weights(seed=0):
    """AlexNet `features` and LPIPS lin weights in the state-dict layouts `LPIPS.from_state_dicts` reads."""
    from presight_b200.metrics import _expected_keys
    g = torch.Generator().manual_seed(seed)
    alex, lin = {}, {}
    for k, shape in _expected_keys().items():
        if k.startswith("lin"):
            lin[k] = torch.rand(shape, generator=g) * (2.0 / shape[1])
        elif k.endswith("weight"):
            fan_in = shape[1] * shape[2] * shape[3]
            alex[k] = torch.randn(shape, generator=g) * (2.0 / fan_in) ** 0.5
        else:
            alex[k] = torch.randn(shape, generator=g) * 0.01
    return alex, lin


def cudnn_lpips(pred, gt, alex, lin):
    """The definition on [B,H,W,3] pairs through F.conv2d / F.max_pool2d on the device (fp32 tensors, TF32 allowed),
    as torchmetrics runs it -> [B]."""
    shift = torch.tensor(SHIFT, device=pred.device)[None, :, None, None]
    scale = torch.tensor(SCALE, device=pred.device)[None, :, None, None]
    x = torch.cat([pred, gt]).permute(0, 3, 1, 2)
    x = (2 * x - 1 - shift) / scale
    B = pred.shape[0]
    total = 0
    for k, (i, stride, pad, pool) in enumerate(LAYERS):
        if pool:
            x = F.max_pool2d(x, 3, 2)
        x = F.relu(F.conv2d(x, alex[f"features.{i}.weight"], alex[f"features.{i}.bias"], stride=stride, padding=pad))
        n = x / (torch.sqrt((x * x).sum(1, keepdim=True)) + 1e-10)
        d = (n[:B] - n[B:]) ** 2
        total = total + F.conv2d(d, lin[f"lin{k}.model.1.weight"]).mean((1, 2, 3))
    return total


def kernel_times(fn, calls):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if "lpips_" in ev.key:
            name = ev.key.replace("ps::(anonymous namespace)::", "").replace("void ", "").split("(")[0]
            out[name] = round(getattr(ev, "device_time_total", 0) / calls / 1e3, 4)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_lpips needs a CUDA device (there is no CPU timing)")
    from presight_b200 import metrics, synthetic
    from presight_b200.cameras.ray_generator import RayGenerator
    dev = torch.device("cuda:0")
    rec = {"tool": "bench_lpips", **device_context(), "tf32_datasheet_tflops": TF32_DATASHEET_TFLOPS,
           "cudnn_allow_tf32": torch.backends.cudnn.allow_tf32}

    with torch.no_grad():
        model, _ = build("c2", dev)
        cams = synthetic.make_cameras(seed=42, n_frames=1)
        H, W = cams["H"], cams["W"]
        gen = RayGenerator(cams["camera_to_worlds"], cams["fx"], cams["fy"], cams["cx"], cams["cy"]).to(dev)
        bundles = [gen.image_rays(i, H, W) for i in range(6)]
        renders, render_ms = [], []
        for i, rb in enumerate(bundles):
            box = {}
            t = event_ms(lambda: box.update(out=model.get_outputs_for_camera_ray_bundle(rb)))
            renders.append(box["out"]["rgb"].clamp(0, 1).contiguous())
            if i > 0:
                render_ms.append(t)
        del model
        torch.cuda.empty_cache()
        g = torch.Generator(device=dev).manual_seed(0)
        targets = [torch.rand(H, W, 3, device=dev, generator=g) for _ in range(6)]
        pred6, gt6 = torch.stack(renders), torch.stack(targets)
        flops_pair = 2 * metrics.lpips_flops(H, W)
        render = statistics.median(render_ms)
        rec.update({"H": H, "W": W, "gflop_per_pair": round(flops_pair / 1e9, 3),
                    "c2_render_ms_default_chunk": round(render, 3),
                    "c2_eval_num_rays_per_chunk": synthetic.config_c2("b200").eval_num_rays_per_chunk})

        alex, lin = random_weights(0)
        net = metrics.LPIPS.from_state_dicts(alex, lin, device=dev)
        alex_d = {k: v.to(dev) for k, v in alex.items()}
        lin_d = {k: v.to(dev) for k, v in lin.items()}

        def timed(fn, per):
            fn()
            torch.cuda.synchronize()
            ms = [event_ms(lambda i=i: fn(i)) for i in range(args.reps)]
            med = statistics.median(ms) / per
            return {"ms_per_pair_median": round(med, 4), "ms_per_pair_min": round(min(ms) / per, 4),
                    "tflops": round(flops_pair / (med * 1e-3) / 1e12, 2),
                    "fraction_of_tf32_datasheet": round(flops_pair / (med * 1e-3) / 1e12 / TF32_DATASHEET_TFLOPS, 4),
                    "fraction_of_c2_render": round(med / render, 4)}

        rec["ps_lpips_B1"] = timed(lambda i=0: net(renders[i % 6], targets[i % 6]), 1)
        rec["ps_lpips_B6"] = timed(lambda i=0: net(pred6, gt6), 6)
        rec["cudnn_tf32_B1"] = timed(lambda i=0: cudnn_lpips(pred6[i % 6:i % 6 + 1], gt6[i % 6:i % 6 + 1], alex_d, lin_d), 1)
        rec["cudnn_tf32_B6"] = timed(lambda i=0: cudnn_lpips(pred6, gt6, alex_d, lin_d), 6)

        ours = net(pred6, gt6)
        ref = cudnn_lpips(pred6, gt6, alex_d, lin_d).double()
        rec["values_ps_lpips"] = [float(v) for v in ours]
        rec["max_rel_diff_vs_cudnn_tf32"] = float(((ours - ref).abs() / ref.abs()).max())
        rec["kernel_ms_per_call_B1"] = kernel_times(lambda: net(renders[0], targets[0]), 20)
        rec["kernel_ms_per_call_B6"] = kernel_times(lambda: net(pred6, gt6), 5)
        rec["goal_ms_per_pair"] = 3.6
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
