#!/usr/bin/env python
"""Headline benchmark: train rays/s of the PreSight city-NeRF inner loop (BASELINE.json config 2).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config c2|c1] [--fp32] [--strong]
                    [--dump-outputs DIR]

One step = encode + MLP + sample + composite, forward and backward (update step: proposal nets get gradients),
plus the gradient all-reduce for N > 1; the optimizer is excluded (SURVEY §8d).  Prints ONE JSON line.
  value     device-resident inputs, CUDA-event timed, max over ranks
  e2e       the same step through the public model API with HOST (pinned) ray batches copied in every step and the
            loss read back every step
  roofline  dominant memory kernel (main-grid hash scatter-add), algorithmic bytes / CUDA-event duration vs measured HBM
            peak; the kernel runs once per ray slice of the final level, concurrently with the field backward
  cpu_baseline  the oracle port of the reference's torch path, timed on this box's host cores on a bounded sample
`--impl reference` times that CPU path alone (the reference arm of the harness).
`--dump-outputs DIR` also writes what the last timed step computed (rank 0) as DIR/<name>.npy, see step_results().
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

METRIC = "train_rays_per_s"
UNIT = "rays/s"

DUMP_RAYS = 4096              # rays sampled from every per-ray output by --dump-outputs
DUMP_GRAD_ENTRIES = 32768     # entries sampled from every larger parameter gradient
DUMP_BYTES = 64 << 20


# ------------------------------------------------------------------------------------------------ helpers
def roofline_traffic(kernel: str, config: str, rays: int) -> dict:
    """{"traffic": dram bytes per launch of `kernel` or None, "traffic_source": ...} from profiles/roofline_traffic.json
    (written from an `ncu --set full` capture of this command, see DESIGN §5)."""
    path = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        with open(path) as f:
            t = json.load(f)
        if t.get("kernel") == kernel and t.get("config") == config and int(t.get("rays_per_gpu", -1)) == rays:
            return {"traffic": float(t["dram_bytes_per_launch"]), "traffic_source": t.get("source")}
    except Exception:
        pass
    return {"traffic": None, "traffic_source": None}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int) -> None:
        super().__init__(daemon=True)
        self.index, self.samples, self._stop_evt = index, [], threading.Event()

    def run(self) -> None:
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) == 6:
                    self.samples.append(parts)
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.samples)}


def build_config(name: str, impl: str):
    from presight_b200 import synthetic
    return {"c1": synthetic.config_c1, "c3": synthetic.config_c1, "c2": synthetic.config_c2, "c5": synthetic.config_c2,
            "presight": synthetic.config_presight}[name](impl)


def workload_name(name: str) -> str:
    return {"c2": "PreSight city NeRF train step: 16-level 2^22-entry hash grid F2 + props L8 F1 2^20 (128/64/64 "
                  "samples), 6-cam nuScenes-shaped rays",
            "c1": "nerfacto-style hash-grid field: main L16 F2 2^19 + props L5 F2 2^17 (256/96/48 samples)",
            "c3": "proposal-heavy sampling: nerfacto-style field, 2 proposal nets (256/96) + 48 NeRF samples/ray",
            "c5": "prior extraction: dense density/feature query on a 400x200x16 BEV voxel grid per tile (C2 model), "
                  "tiles sharded over the GPUs, no communication",
            "presight": "PreSight shipped shape: 16 sub-fields (nearest-centroid routing), main L10 F4 2^20 16->16384 each "
                        "+ props L8 F1 2^20 (128/64/64 samples), 6-cam nuScenes-shaped rays"}[name]


def build_model(config_name: str, cfg, host, dev):
    """Random-init model of the named configuration (16 routed sub-fields for `presight`, one otherwise)."""
    from presight_b200 import synthetic
    from presight_b200.model import NerfactoNuscMSModel
    if config_name == "presight":
        centroids, aabbs = synthetic.sub_field_layout(16)
    else:
        centroids, aabbs = torch.zeros(1, 3), synthetic.tile_aabb()
    return NerfactoNuscMSModel(cfg, centroids, aabbs, host["n_cameras"], host["n_videos"]).to(dev)


# ------------------------------------------------------------------------------------------------ C5: prior query
def time_prior_query(model, dev, rank, world, iters, tiles_total=8, with_e2e=True):
    """BASELINE config 5: `model.query_priors` on the 400x200x16 grid of each of this rank's tiles (8 tiles, sharded by
    tile with no communication — extract_priors.py:151-154 concatenates on the host).  -> dict with device-resident and
    host-buffer (points copied in from pinned memory, densities + fp16 features copied out) timings, max over ranks."""
    from presight_b200 import synthetic
    from presight_b200.parallel import shard_range
    lo, hi = shard_range(tiles_total, rank, world)
    if world > tiles_total:
        lo, hi = rank % tiles_total, rank % tiles_total + 1
    host_grids = [synthetic.prior_tile_grid(t).pin_memory() for t in range(lo, hi)]
    grids = [g.to(dev, non_blocking=True) for g in host_grids]
    M = host_grids[0].shape[0]
    for g in grids:
        model.query_priors(g)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        for g in grids:
            model.query_priors(g)
    b.record()
    torch.cuda.synchronize()
    t_dev = a.elapsed_time(b) / 1e3
    t_e2e = float("nan")
    if with_e2e:
        out_mean = torch.empty(M, dtype=torch.float32).pin_memory()
        out_feat = torch.empty(M, 64, dtype=torch.float16).pin_memory()
        if world > 1:
            dist.barrier()
        a.record()
        for _ in range(iters):
            for hg in host_grids:
                mean, feats = model.query_priors(hg.to(dev, non_blocking=True))
                out_mean.copy_(mean, non_blocking=True)
                out_feat.copy_(feats, non_blocking=True)
        b.record()
        torch.cuda.synchronize()
        t_e2e = a.elapsed_time(b) / 1e3
    if world > 1:
        tt = torch.tensor([t_dev, t_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_dev, t_e2e = float(tt[0]), float(tt[1])
    n_tiles = max(1, hi - lo)
    pts = M * n_tiles * iters * world
    faithful, elided = synthetic.prior_query_bytes_per_point(model.config)
    return {"points_per_s": pts / t_dev, "e2e_points_per_s": pts / t_e2e, "points_per_tile": M, "tiles": n_tiles * world,
            "ms_per_tile": t_dev / (iters * n_tiles) * 1e3, "e2e_ms_per_tile": t_e2e / (iters * n_tiles) * 1e3,
            "h2d_bytes_per_tile": M * 12, "d2h_bytes_per_tile": M * (4 + 128),
            "algorithmic_bytes_per_point": {"reference_count": faithful, "duplicate_encode_elided": elided},
            "GBps_per_gpu_reference_count": faithful * pts / t_dev / 1e9 / world,
            "GBps_per_gpu_elided_count": elided * pts / t_dev / 1e9 / world}


# ------------------------------------------------------------------------------------------------ loss
def step_loss(model, out, batch):
    """The loss dict of a camera-only training step — rgb MSE, sky BCE, semantic MSE, (z-anti-aliased) interlevel,
    distortion — summed as the trainer does (nerfacto_nusc_ms.py:558-645 with the multipliers of :127-133,167,192;
    trainer.py:498 `functools.reduce(torch.add, loss_dict.values())`)."""
    loss_dict = model.get_loss_dict(out, batch)
    loss = None
    for v in loss_dict.values():
        loss = v if loss is None else loss + v
    return loss


def step_results(out, loss, model, n_rays: int) -> dict:
    """What a training step hands its caller, as host float32 / float64 arrays: the loss, the model outputs (weights and
    euclidean bin edges per sampler level) of a fixed seeded sample of DUMP_RAYS rays, and every parameter gradient (a
    fixed seeded sample of DUMP_GRAD_ENTRIES entries of a larger one).  The samples depend on the shapes alone, so two
    builds run with the same arguments write files that compare entry for entry."""
    g = torch.Generator().manual_seed(0)
    rows = torch.randperm(n_rays, generator=g)[:DUMP_RAYS].sort().values.to(loss.device)
    res = {"loss": loss}
    for k, v in out.items():
        if k == "weights_list":
            res.update({f"weights_{i}": w[rows] for i, w in enumerate(v)})
        elif k == "ray_samples_list":
            res.update({f"eu_bins_{i}": rs.frustums.eu_bins[rows] for i, rs in enumerate(v)})
        else:
            res[k] = v[rows]
    for name, p in model.named_parameters():
        if p.grad is None:
            continue
        gr = p.grad.reshape(-1)
        if gr.numel() > DUMP_GRAD_ENTRIES:
            gr = gr[torch.randint(gr.numel(), (DUMP_GRAD_ENTRIES,), generator=g).to(gr.device)]
        res[f"grad.{name}"] = gr
    arrays = {k: v.detach().to("cpu", torch.float64 if v.dtype == torch.float64 else torch.float32).numpy()
              for k, v in res.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_BYTES, f"--dump-outputs would write {total} bytes (limit {DUMP_BYTES})"
    return arrays


# ------------------------------------------------------------------------------------------------ CPU reference arm
def oracle_model_from(model, cfg):
    """Build the oracle's parameter containers from the product model's state dict (CPU copies)."""
    import oracle as O
    from oracle import state as OS
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    fmeta = dict(num_levels=cfg.num_levels, base_res=cfg.base_res, max_res=cfg.max_res,
                 log2_hashmap_size=cfg.log2_hashmap_size, use_semantics=cfg.use_semantics,
                 semantic_dim=cfg.semantic_dim)
    nf = len(model.field.fields)
    fields = [OS.ngp_from_state(sd, f"field.fields.{i}.", fmeta, True) for i in range(nf)]
    props = []
    for lvl, net in enumerate(model.proposal_networks):
        a = cfg.proposal_net_args_list[min(lvl, len(cfg.proposal_net_args_list) - 1)]
        pm = dict(num_levels=a["num_levels"], base_res=a.get("base_res", 16), max_res=a["max_res"],
                  log2_hashmap_size=a["log2_hashmap_size"], use_linear=a.get("use_linear", False))
        props.append([OS.prop_from_state(sd, f"proposal_networks.{lvl}.fields.{i}.", pm, True) for i in range(nf)])
    sky = None
    if cfg.use_sky_model:
        sky = [OS.sky_from_state(sd, f"sky_model.fields.{i}.", cfg.use_semantics, True) for i in range(nf)]
    ocfg = O.ModelCfg(num_proposal_samples=tuple(cfg.num_proposal_samples_per_ray),
                      num_nerf_samples=cfg.num_nerf_samples_per_ray, near=cfg.near_plane, far=cfg.far_plane,
                      piecewise_thr=cfg.piecewise_sampler_threshold)
    emb = {k: sd[k] for k in sd if "embedding.embedding.weight" in k}
    return O.Model(ocfg, model.centroids.cpu(), fields, props, sky), emb


def cpu_reference_step(omodel, emb, cfg, batch, n):
    """One fwd+bwd of the oracle port on `n` rays (torch CPU, all host threads)."""
    import oracle as O
    o, d = batch["origins"][:n], batch["directions"][:n]
    parts = []
    if cfg.appearance_embed_dim > 0:
        parts.append(emb["appearance_embedding.embedding.weight"][batch["camera_indices"][:n, 0]])
    if cfg.video_embed_dim > 0:
        parts.append(emb["video_embedding.embedding.weight"][batch["video_ids"][:n, 0]])
    app = torch.cat(parts, dim=-1) if parts else None
    jit = [torch.rand(n, 1) for _ in range(len(cfg.num_proposal_samples_per_ray) + 1)]
    out = O.model_outputs(omodel, o, d, app, jit)
    loss = O.rgb_loss(batch["rgb"][:n], out["rgb"])
    if cfg.use_sky_model:
        loss = loss + 0.001 * O.sky_loss(out["accumulation"].view(-1, 1), batch["sky"][:n].view(-1, 1))
    if cfg.use_semantics:
        loss = loss + 0.5 * O.semantic_loss(out["semantics"], batch["features"][:n])
    sp = [b[0] for b in out["bins_list"]]
    if cfg.enable_z_anti_aliasing:
        loss = loss + cfg.interlevel_loss_mult * O.z_anti_aliasing_interlevel_loss(out["weights_list"], sp, cfg.pulse_width)
    else:
        loss = loss + cfg.interlevel_loss_mult * O.interlevel_loss(out["weights_list"], sp)
    loss = loss + cfg.distortion_loss_mult * O.distortion_loss(out["weights_list"], sp)
    params = [f.grid.table for f in omodel.fields] + [p.grid.table for lvl in omodel.props for p in lvl]
    for p in params:
        p.grad = None
    loss.backward()
    return float(loss.detach())


def time_cpu_reference(model, cfg, batch, sample_rays, steps, warmup):
    torch.set_num_threads(os.cpu_count() or 1)
    omodel, emb = oracle_model_from(model, cfg)
    for _ in range(warmup):
        cpu_reference_step(omodel, emb, cfg, batch, sample_rays)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        cpu_reference_step(omodel, emb, cfg, batch, sample_rays)
        ts.append(time.perf_counter() - t0)
    return sample_rays / statistics.median(ts), statistics.median(ts)


def cpu_hash_only(cfg, n_points=1 << 16):
    """The figure BASELINE.md §3 promises beside the step: the reference-style torch HashEncoding (oracle port of
    encodings.py:343-384, main grid) forward + backward alone on the host cores -> points/s."""
    import oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    grid = O.HashGrid(table=((torch.rand((cfg.num_levels << cfg.log2_hashmap_size), cfg.features_per_level) * 2 - 1)
                             * 1e-3).requires_grad_(True),
                      scalings=O.hash_scalings(cfg.num_levels, cfg.base_res, cfg.max_res), log2_T=cfg.log2_hashmap_size)
    x = torch.rand(n_points, 3)
    ts = []
    for _ in range(3):
        grid.table.grad = None
        t0 = time.perf_counter()
        O.hash_encode(x, grid).sum().backward()
        ts.append(time.perf_counter() - t0)
    return n_points / statistics.median(ts)


def main_c5(args, model, cfg, host, dev, rank, world):
    """`--config c5`: the prior query as the benchmarked step (one step = one tile's 1.28 M-point query)."""
    from presight_b200 import ops, synthetic
    model.eval()
    clocks = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    clocks.start()
    ops.PROBE = ops.KernelProbe()
    l0 = ops.launch_count()
    r = time_prior_query(model, dev, rank, world, max(args.steps, 1))
    launches = ops.launch_count() - l0
    probe = ops.PROBE.summary()
    ops.PROBE = None
    clock_info = clocks.stop()
    if rank == 0:
        peak, peak_src = measured_peaks()
        L, F = cfg.num_levels, cfg.features_per_level
        kname = f"hash_fwd_L{L}F{F}T{cfg.log2_hashmap_size}"
        n_launch, k_mean = probe.get(kname, (0, float("nan")))
        algo = synthetic.hash_bytes_fwd(L, F) * r["points_per_tile"]
        line = {"metric": "prior_query_points_per_s", "value": r["points_per_s"], "unit": "points/s", "n_gpus": world,
                "steps": args.steps, "warmup": 1, "ms_per_step": r["ms_per_tile"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32 hash + bf16 MLP, fp16 features", "data": "synthetic",
                "config": {"workload": workload_name("c5"), "points_per_tile": r["points_per_tile"], "tiles": r["tiles"],
                           "parallelism": f"tiles sharded over {world} GPU(s), no communication",
                           "l2": "inputs larger than L2 (576 MiB of hash tables)"},
                "e2e": {"value": r["e2e_points_per_s"], "unit": "points/s", "h2d_bytes_per_step": r["h2d_bytes_per_tile"],
                        "d2h_bytes_per_step": r["d2h_bytes_per_tile"], "ms_per_step": r["e2e_ms_per_tile"]},
                "gpu_launches": int(launches), "clocks": clock_info,
                "roofline": {"bound": "hbm", "kernel": kname, "achieved": algo / (k_mean * 1e-3) / 1e9 if n_launch else None,
                             "peak": peak, "unit": "GB/s",
                             "frac": algo / (k_mean * 1e-3) / 1e9 / peak if n_launch else None, "traffic": None,
                             "peak_source": peak_src, "kernel_ms": k_mean,
                             "step_GBps_reference_count": r["GBps_per_gpu_reference_count"],
                             "step_GBps_elided_count": r["GBps_per_gpu_elided_count"],
                             "step_frac_of_hbm_roofline_reference_count": r["GBps_per_gpu_reference_count"] / peak},
                "kernels_ms_per_launch": {k: round(v[1], 4) for k, v in sorted(probe.items())}}
        if world == 1 and not args.no_cpu_baseline:
            import oracle as O
            torch.set_num_threads(os.cpu_count() or 1)
            om, _ = oracle_model_from(model, cfg)
            n = 16384
            pts = synthetic.prior_tile_grid(0)[:n]
            t0 = time.perf_counter()
            O.prior_query(om, pts)
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": n / dt, "unit": "points/s", "cores": os.cpu_count() or 1, "kind": "port",
                                    "sample": f"{n} points of tile 0, oracle port of extract_priors.py:130-138 (torch CPU fp32)"}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ main
_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line of the contract, written to the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main() -> None:
    # stdout carries exactly one JSON line: anything libraries print while the run is going on (NCCL writes its
    # "NCCL version ..." banner to stdout when NCCL_DEBUG is set) is sent to stderr at the file-descriptor level
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=["c1", "c2", "c3", "c5", "presight"],
                    help="c2 = the headline workload (BASELINE config 2 / 4); c1 / c3 = nerfacto-style shapes (config 1 / 3); "
                         "c5 = prior query per tile; presight = the shipped 16-sub-field shape")
    ap.add_argument("--no-extras", action="store_true",
                    help="default c2 run only: skip the short extra measurements folded into the line "
                         "(C5 prior query per tile, strong-scaling step for N > 1)")
    ap.add_argument("--rays", type=int, default=65536, help="rays per GPU (weak scaling) or global (--strong)")
    ap.add_argument("--fp32", action="store_true", help="3xTF32 MLPs (1e-3 parity class) instead of bf16")
    ap.add_argument("--strong", action="store_true", help="fixed global batch split across ranks (reference semantics)")
    ap.add_argument("--cpu-sample-rays", type=int, default=1024)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the end-to-end leg (short runs under ncu)")
    ap.add_argument("--optimizer", default="none", choices=["none", "torch", "fused"],
                    help="also take an Adam step inside the timed step (SURVEY 8f-2; the headline metric excludes it): "
                         "torch.optim.Adam or presight_b200.optim.FusedAdam with PreSight's hyper-parameters")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's loss, sampled outputs and sampled gradients (rank 0) as DIR/<name>.npy, "
                         "so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.config == "c5" or args.steps < 1):
        ap.error("--dump-outputs needs the training step of the b200 arm (not --impl reference or --config c5) and --steps >= 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    impl = "b200+fp32" if args.fp32 else "b200"
    from presight_b200 import synthetic
    cfg = build_config(args.config, impl)

    # ---------------------------------------------------------------- reference arm: CPU only, rank 0 only
    if args.impl == "reference":
        if rank != 0:
            return
        from presight_b200.model import NerfactoNuscMSModel
        torch.manual_seed(42)
        batch = synthetic.make_rays(max(args.cpu_sample_rays, 1), seed=42)
        model = NerfactoNuscMSModel(cfg, torch.zeros(1, 3), synthetic.tile_aabb(), batch["n_cameras"], batch["n_videos"])
        t_start = time.perf_counter()
        rps, med = time_cpu_reference(model, cfg, batch, args.cpu_sample_rays, max(1, args.steps), max(1, args.warmup))
        cores = os.cpu_count() or 1
        sample = f"{args.cpu_sample_rays} rays/step of the same workload, torch CPU fp32, {cores} threads"
        emit({
            "impl": "reference", "metric": METRIC, "value": rps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": med * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args.config), "rays_per_step": args.cpu_sample_rays},
            "cpu_baseline": {"value": rps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": rps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": time.perf_counter() - t_start})
        return

    # ---------------------------------------------------------------- b200 arm
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback for the b200 path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        from presight_b200.parallel import init_nccl
        init_nccl(dev, high_priority=os.environ.get("PS_NCCL_PRIO", "1") == "1")
    from presight_b200 import ops
    from presight_b200.cameras.rays import RayBundle
    from presight_b200.model import VIDEO_ID, NerfactoNuscMSModel
    from presight_b200.parallel import GradSynchronizer

    rays_per_rank = args.rays // world if args.strong else args.rays
    torch.manual_seed(42)                                        # identical weights on every rank
    host = synthetic.make_rays(rays_per_rank, seed=42 + rank)    # reference seeds data with seed + rank (train.py:99)
    model = build_model(args.config, cfg, host, dev)
    if args.config == "c5":
        return main_c5(args, model, cfg, host, dev, rank, world)
    model.train()
    params = [p for p in model.parameters() if p.requires_grad]
    sync = None
    if world > 1:
        # The 512 MiB main-table gradient is complete only when its last level has been scattered, at the very end of the
        # backward.  It is exchanged level group by level group from inside the backward (parallel.py), so all but the last
        # group travel under the remaining scatter and the proposal levels' backward, which keep their single-GPU schedule.
        # PS_PARTIAL_AR=0: whole-table all-reduce, hidden under the proposal levels' backward run after the final level.
        from presight_b200 import fused
        from presight_b200.parallel import level_groups
        partial = []
        if os.environ.get("PS_PARTIAL_AR", "1") == "1":
            cuts = os.environ.get("PS_AR_CUTS")
            for n, m in model.named_modules():
                if n.endswith("mlp_base_grid") and hasattr(m, "hash_table") and "proposal" not in n:
                    partial.append((m.hash_table, level_groups(m.num_levels, None if cuts is None else
                                                               [int(c) for c in cuts.split(",")], world)))
        # PS_EXCHANGE=peer: the pieces on the copy engines between IPC-mapped buffers (peer_exchange.py) instead of NCCL
        # all-reduces (parity-tested; at 2 GPUs no faster than NCCL, profiles/r2_e_n2_variants.txt, so not the default)
        sync = GradSynchronizer(params, overlap=True, partial_tables=partial,
                                peer=os.environ.get("PS_EXCHANGE", "nccl") == "peer")
        if not partial:
            fused.set_overlap_prop_bwd(False)
    optimizer = None
    if args.optimizer == "torch":
        optimizer = torch.optim.Adam(params, lr=1e-2, eps=1e-15, weight_decay=1e-5)
    elif args.optimizer == "fused":
        from presight_b200.optim import FusedAdam
        optimizer = FusedAdam(params, lr=1e-2, eps=1e-15, weight_decay=1e-5)

    tensor_keys = ("origins", "directions", "camera_indices", "video_ids", "rgb", "features", "sky")
    pinned = {k: host[k].pin_memory() for k in tensor_keys}
    resident = {k: pinned[k].to(dev, non_blocking=True) for k in tensor_keys}
    h2d_bytes = sum(pinned[k].numel() * pinned[k].element_size() for k in tensor_keys)

    def run_step(batch, keep=None):
        for p in params:
            p.grad = None
        rb = RayBundle(origins=batch["origins"], directions=batch["directions"],
                       camera_indices=batch["camera_indices"], metadata={VIDEO_ID: batch["video_ids"]})
        model.proposal_sampler._step = 0                 # update step: proposal nets receive gradients
        out = model(rb)
        loss = step_loss(model, out, batch)
        loss.backward()
        if sync is not None:
            sync.finish()
        if optimizer is not None:
            optimizer.step()
        if keep is not None:
            keep.update(out=out, loss=loss)
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up
    for _ in range(max(args.warmup, 3)):
        run_step(resident)
    barrier()

    # ---- timed: device-resident inputs
    clocks = ClockSampler(local_rank)
    clocks.start()
    ops.PROBE = ops.KernelProbe()
    launches0 = ops.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_host0 = time.perf_counter()
    run_step(resident)                               # one more warm-up step, timed on the HOST with an empty launch queue:
    t_host = time.perf_counter() - t_host0          # the Python / launch cost of a step (the GPU must exceed it to stay busy)
    barrier()
    last_step = {} if args.dump_outputs else None
    ev0.record()
    for i in range(args.steps):
        run_step(resident, last_step if i == args.steps - 1 else None)
    ev1.record()
    barrier()
    dump = None
    if last_step is not None and rank == 0:          # read before the end-to-end leg replaces the gradients
        dump = step_results(last_step["out"], last_step["loss"], model, rays_per_rank)
    last_step = None
    launches = ops.launch_count() - launches0
    probe = ops.PROBE.summary()
    ops.PROBE = None
    t_dev = ev0.elapsed_time(ev1) / 1e3

    # ---- timed: end to end.  Every step: this step's batch is copied from pinned host memory (double-buffered on a copy
    # stream, so the copy of batch k+1 travels under the compute of batch k) and the step's loss is read back to the host
    # (asynchronously into pinned memory; the host consumes it one step later, as a trainer's logger does).
    from presight_b200.prefetch import DevicePrefetcher
    pf = DevicePrefetcher(dev, tensor_keys)
    loss_host = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ready = [torch.cuda.Event(), torch.cuda.Event()]

    def e2e_loop(n_steps):
        last_ = 0.0
        pf.push(pinned)
        for i in range(n_steps):
            batch = pf.pop()
            if i + 1 < n_steps:
                pf.push(pinned)                      # next step's inputs: host -> device while this step computes
            loss_ = run_step(batch)
            pf.release()
            loss_host[i % 2].copy_(loss_.detach(), non_blocking=True)      # device -> host read of the step's result
            loss_ready[i % 2].record()
            if i > 0:
                loss_ready[(i - 1) % 2].synchronize()
                last_ = float(loss_host[(i - 1) % 2])
        loss_ready[(n_steps - 1) % 2].synchronize()
        return float(loss_host[(n_steps - 1) % 2])
    if args.no_e2e:
        t_e2e, last = float("nan"), float("nan")
    else:
        e2e_loop(2)
        barrier()
        ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev2.record()
        last = e2e_loop(args.steps)
        ev3.record()
        barrier()
        t_e2e = ev2.elapsed_time(ev3) / 1e3
    clock_info = clocks.stop()

    # ---- the roofline kernel alone: the main-grid scatter on the step's own final-level sample points (same ray slices
    # as the step, nothing else on the device), CUDA events on its stream.  In the step it shares the SMs with the
    # field / proposal backward kernels, so its in-step event time measures the pipeline, not the kernel.
    alone_ms = None
    if rank == 0 and cfg.num_levels * cfg.features_per_level <= 48:
        from presight_b200 import fused
        from presight_b200._lib import call, host_floats, ptr, stream
        with torch.no_grad():
            rb = RayBundle(origins=resident["origins"], directions=resident["directions"],
                           camera_indices=resident["camera_indices"], metadata={VIDEO_ID: resident["video_ids"]})
            eu = model(rb)["ray_samples_list"][-1].frustums.eu_bins.contiguous()
        f0 = model.field.fields[0]
        enc = f0.mlp_base_grid
        x01, _ = fused._ray_points(resident["origins"], resident["directions"], eu, f0.aabb_host(),
                                   f0.spatial_distortion is not None)
        S_, L_, F_, T_ = eu.shape[1] - 1, cfg.num_levels, cfg.features_per_level, cfg.log2_hashmap_size
        dfeat = torch.randn(x01.shape[0] * L_ * F_, device=dev) * 1e-3
        dtab = torch.zeros_like(enc.hash_table)
        bounds = fused._chunk_bounds(rays_per_rank, S_)

        def scatter_all():
            P_ = x01.shape[0]
            for (c0, c1) in bounds:      # level-major gradient of a slice = [L][slice points][F]: rebuild the view
                n_ = (c1 - c0) * S_
                call("ps_hash_bwd_lm", ptr(x01[c0 * S_:c1 * S_]), n_, None, host_floats(enc._scalings_host), L_, F_, T_,
                     ptr(dfeat[:n_ * L_ * F_]), ptr(dtab), None, stream())
        scatter_all()
        torch.cuda.synchronize()
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record()
        for _ in range(5):
            scatter_all()
        eb.record()
        torch.cuda.synchronize()
        alone_ms = ea.elapsed_time(eb) / 5
        del dfeat, dtab, x01

    # ---- extras folded into the default line (short; all ranks take part): the strong-scaling variant of the step — the
    # reference's semantics, train_num_rays_per_batch // world_size per rank (my_datamanager.py:206) — and BASELINE
    # config 5, the prior query per tile with tiles sharded over the ranks
    extras = {}
    if args.config == "c2" and not args.no_extras and optimizer is None:
        if world > 1 and not args.strong:
            n_s = args.rays // world
            hs = synthetic.make_rays(n_s, seed=1042 + rank)
            res_s = {k: hs[k].to(dev) for k in tensor_keys}
            for _ in range(3):
                run_step(res_s)
            barrier()
            es0, es1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k_s = max(5, min(args.steps, 20))
            es0.record()
            for _ in range(k_s):
                run_step(res_s)
            es1.record()
            barrier()
            ts = torch.tensor([es0.elapsed_time(es1) / 1e3], device=dev, dtype=torch.float64)
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
            extras["strong"] = {"metric": METRIC, "value": n_s * world * k_s / float(ts), "unit": UNIT,
                                "global_rays": n_s * world, "rays_per_gpu": n_s, "ms_per_step": float(ts) / k_s * 1e3,
                                "steps": k_s, "scaling": "strong"}
            del res_s
        model.eval()
        c5 = time_prior_query(model, dev, rank, world, 5)
        model.train()
        extras["c5_prior_query"] = c5

    if world > 1:
        t = torch.tensor([t_dev, t_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_dev, t_e2e = float(t[0]), float(t[1])
    total_rays = rays_per_rank * world
    value = total_rays * args.steps / t_dev
    e2e = total_rays * args.steps / t_e2e

    if rank == 0:
        peak, peak_src = measured_peaks()
        L, F = cfg.num_levels, cfg.features_per_level
        points = rays_per_rank * cfg.num_nerf_samples_per_ray
        kname = f"hash_bwd_L{L}F{F}T{cfg.log2_hashmap_size}"
        n_launch, k_mean = probe.get(kname, (0, float("nan")))
        # the final level is processed in ray slices (presight_b200/fused.py): the kernel's time per step is the sum of
        # its launches in that step; the slices overlap the field-backward kernel of the next slice on another stream
        k_ms = n_launch * k_mean / args.steps if n_launch else float("nan")
        algo_bytes = synthetic.hash_bytes_bwd(L, F) * points
        achieved = algo_bytes / (k_ms * 1e-3) / 1e9 if n_launch else None
        step_bytes = synthetic.step_bytes_per_ray(cfg, True)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": t_dev / args.steps * 1e3, "higher_is_better": True,
            "scaling": "strong" if args.strong else "weak", "vs_baseline": None,
            "dtype": "f32 (hash/compositing) + " + ("tf32x3 MLP" if args.fp32 else "bf16 MLP, fp32 accumulate"),
            "data": "synthetic",
            "config": {"workload": workload_name(args.config), "rays_per_gpu": rays_per_rank, "global_rays": total_rays,
                       "parallelism": f"dp{world}",
                       "step": "update step (proposal nets trained), " + ("optimizer excluded" if optimizer is None
                                                                          else f"Adam step included ({args.optimizer})"),
                       "l2": "inputs larger than L2 (576 MiB of hash tables + grads re-zeroed every step)"},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                    "ms_per_step": t_e2e / args.steps * 1e3},
            "gpu_launches": int(launches), "host_enqueue_ms_per_step": t_host * 1e3,
            "clocks": clock_info,
            "roofline": {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None,
                         # dram__bytes_read + write of ONE launch of this kernel from the ncu --set full capture of this
                         # same command, kept in profiles/roofline_traffic.json with its source file (null when the
                         # run's shape is not the captured one)
                         **roofline_traffic(kname, args.config, rays_per_rank),
                         "peak_source": peak_src,
                         "kernel_ms": k_ms, "launches_per_step": (n_launch / args.steps) if n_launch else None,
                         "algorithmic_bytes_per_launch": algo_bytes / max(1.0, n_launch / args.steps) if n_launch else None,
                         "algorithmic_bytes_per_step": algo_bytes,
                         "step_frac_of_hbm_roofline": (step_bytes * total_rays / world) / (t_dev / args.steps) / 1e9 / peak,
                         # the same launches with the device to themselves (see above)
                         "alone": None if not alone_ms else {
                             "kernel_ms": alone_ms, "achieved": algo_bytes / (alone_ms * 1e-3) / 1e9,
                             "frac": algo_bytes / (alone_ms * 1e-3) / 1e9 / peak}},
            "kernels_ms_per_step": {k: round(v[0] * v[1] / args.steps, 4) for k, v in sorted(probe.items())},
            "loss": last,
        }
        if extras:
            line["extras"] = extras
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            n = args.cpu_sample_rays
            rps, med = time_cpu_reference(model, cfg, host, n, 3, 1)
            line["cpu_baseline"] = {"value": rps, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"{n} rays/step of the same workload ({args.config}) and weights: the oracle "
                                              f"port of the reference's torch path (the reference modules themselves "
                                              f"cannot travel to this box), torch CPU fp32, {cores} threads, median of 3 "
                                              f"steps ({med:.2f} s/step)",
                                    "hash_only_points_per_s": cpu_hash_only(cfg)}
        if dump is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dump.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
