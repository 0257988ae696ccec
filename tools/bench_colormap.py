"""Colormapped evaluation images and the eval-split loop: `ps_colormap` per 1600 x 900 image with M = 3 depth-like maps
(depth, prop_depth_0, prop_depth_1), the same definition run by torch (nerfstudio's colormaps, host reads included),
and `evaluate.average_eval_image_metrics` per C2 image.  Prints one JSON line.

    python tools/bench_colormap.py [--reps 20] [--out profiles/colormap_bench.json]

Byte model of one call: 8 M HW read for the maps (min / max pass and map pass), 4 HW for the accumulation and
12 (M + 1) HW written, 109.4 MB at 1600 x 900 with M = 3; its share of the HBM byte bound is set against NVIDIA's
data-sheet 7.7 TB/s for one B200, which is not a measured peak.  One call's working set (~92 MB) fits the 126 MB L2, so
the timed calls cycle over four input / output sets (~370 MB) and each call starts from HBM.  Kernel call time: CUDA
events around 50 consecutive raw `ps_colormap` calls (stacked maps and workspace prepared), median of `--reps` windows;
`colormap_images` adds the stack of the maps and the allocations.  Torch restatement: host clock around one image's
four colormaps and a device synchronise (it reads min / max to the host per depth map), median of `--reps`.  Eval loop:
host clock around `average_eval_image_metrics` over five 1600 x 900 C2 frames with `model.colormap` and `model.lpips`
(random weights) set, after one warm-up frame; random-init field.  Kernel times: torch.profiler in a pass of its own.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(os.path.dirname(ROOT), "tests"))

from bench_extract import build, device_context  # noqa: E402
from bench_lpips import random_weights  # noqa: E402

HBM_DATASHEET_TBS = 7.7
SETS = 4


def bytes_per_call(M: int, HW: int) -> int:
    return 8 * M * HW + 4 * HW + 12 * (M + 1) * HW


def kernel_times(fn, calls):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if "colormap_" in ev.key:
            name = ev.key.replace("ps::(anonymous namespace)::", "").replace("void ", "").split("(")[0]
            out[name] = round(getattr(ev, "device_time_total", 0) / calls / 1e3, 4)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_colormap needs a CUDA device (there is no CPU timing)")
    from presight_b200 import _lib, evaluate, metrics, synthetic
    from presight_b200.cameras.ray_generator import RayGenerator
    from test_gpu_colormap import apply_colormap, apply_depth_colormap
    dev = torch.device("cuda:0")
    H, W, M = 900, 1600, 3
    HW = H * W
    nbytes = bytes_per_call(M, HW)
    rec = {"tool": "bench_colormap", **device_context(), "H": H, "W": W, "M": M, "bytes_per_call": nbytes,
           "hbm_datasheet_tbs": HBM_DATASHEET_TBS, "input_sets_cycled": SETS}
    g = torch.Generator(device=dev).manual_seed(0)
    lut = torch.rand(256, 3, device=dev, generator=g)
    sets = []
    for _ in range(SETS):
        maps = [0.5 + 80 * torch.rand(H, W, 1, device=dev, generator=g) ** 2 for _ in range(M)]
        acc = torch.rand(H, W, 1, device=dev, generator=g)
        stacked = torch.stack([m.reshape(HW) for m in maps])
        out = torch.empty(M + 1, HW, 3, device=dev)
        sets.append((maps, acc, stacked, out))
    ws_bytes = C.c_int64(0)
    _lib.call("ps_colormap_workspace", M, HW, C.byref(ws_bytes))
    ws = torch.empty(ws_bytes.value, dtype=torch.uint8, device=dev)
    lib, st = _lib.load(), _lib.stream()

    def raw(i):
        _, acc, stacked, out = sets[i % SETS]
        return lib.ps_colormap(stacked.data_ptr(), M, HW, acc.data_ptr(), lut.data_ptr(), ws.data_ptr(),
                               out.data_ptr(), st)

    def events(fn, n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(n):
            fn(i)
        b.record()
        b.synchronize()
        return a.elapsed_time(b) / n

    with torch.no_grad():
        # correctness at the timed size: the kernel against torch's definition, bit for bit
        acc_img, depth_imgs = metrics.colormap_images(sets[0][0], sets[0][1], lut)
        rec["bit_identical_to_torch"] = bool(
            torch.equal(acc_img, apply_colormap(sets[0][1], lut))
            and all(torch.equal(d, apply_depth_colormap(m, sets[0][1], lut)) for d, m in zip(depth_imgs, sets[0][0])))

        _lib.check(raw(0), "ps_colormap")
        for _ in range(3):
            events(raw, 50)
        ms = [events(raw, 50) for _ in range(args.reps)]
        med = statistics.median(ms)
        rec["ps_colormap"] = {"ms_per_image_median": round(med, 5), "ms_per_image_min": round(min(ms), 5),
                              "gb_per_s": round(nbytes / (med * 1e-3) / 1e9, 1),
                              "fraction_of_hbm_byte_bound": round(nbytes / (HBM_DATASHEET_TBS * 1e12) / (med * 1e-3), 4)}

        def wrapped(i):
            maps, acc, _, _ = sets[i % SETS]
            metrics.colormap_images(maps, acc, lut)
        events(wrapped, 10)
        rec["colormap_images_ms_per_image_median"] = round(statistics.median(events(wrapped, 20)
                                                                              for _ in range(args.reps)), 5)

        def torch_restatement(i):
            maps, acc, _, _ = sets[i % SETS]
            torch.cuda.synchronize()
            t = time.perf_counter()
            apply_colormap(acc, lut)
            for m in maps:
                apply_depth_colormap(m, acc, lut)
            torch.cuda.synchronize()
            return (time.perf_counter() - t) * 1e3
        for i in range(5):
            torch_restatement(i)
        tms = [torch_restatement(i) for i in range(args.reps)]
        rec["torch_restatement"] = {"ms_per_image_median": round(statistics.median(tms), 4),
                                    "ms_per_image_min": round(min(tms), 4), "host_reads_per_image": 2 * M}
        rec["speedup_vs_torch"] = round(statistics.median(tms) / med, 1)
        rec["kernel_ms_per_call"] = kernel_times(lambda: raw(0), 50)
        del sets
        torch.cuda.empty_cache()

    # the eval loop on C2 at 1600 x 900
    model, _ = build("c2", dev)
    alex, lin = random_weights(0)
    model.lpips = metrics.LPIPS.from_state_dicts(alex, lin, device=dev)
    model.colormap = lut
    cams = synthetic.make_cameras(seed=42, n_frames=1)
    gen = RayGenerator(cams["camera_to_worlds"], cams["fx"], cams["fy"], cams["cx"], cams["cy"]).to(dev)
    gimg = torch.Generator(device=dev).manual_seed(1)
    frames = [(i, torch.rand(cams["H"], cams["W"], 3, device=dev, generator=gimg)) for i in range(6)]
    evaluate.average_eval_image_metrics(model, gen, frames[:1])
    torch.cuda.synchronize()
    t = time.perf_counter()
    avg = evaluate.average_eval_image_metrics(model, gen, frames[1:], get_std=True)
    loop_ms = (time.perf_counter() - t) * 1e3 / 5
    rec["eval_loop_c2"] = {"frames": 5, "ms_per_image": round(loop_ms, 2), "H": cams["H"], "W": cams["W"],
                           "eval_num_rays_per_chunk": model.config.eval_num_rays_per_chunk,
                           "metrics": {k: round(v, 6) for k, v in avg.items()},
                           "ps_colormap_fraction_of_loop": round(med / loop_ms, 5)}
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
