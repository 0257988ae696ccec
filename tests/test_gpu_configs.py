"""Parity at the NAMED configurations of BASELINE.json / SURVEY §8 — real grid and network sizes, reduced ray counts:

  C1 / C3  nerfacto-style field (main L16 F2 T2^19, props L5 F2 T2^17 hidden 16, samples 256/96/48): the stand-alone
           kernels serve every level (the fused tcgen05 kernels do not cover these sample counts);
  C2 / C4  PreSight train step (main L16 F2 T2^22, props L8 F1 T2^20 hidden 64, samples 128/64/64, 64-d semantics, sky):
           the fused tcgen05 proposal / field kernels serve every level (bf16 class) — C4 is the same step per rank, its
           gradient exchange is covered on CPU by tests/test_parallel_cpu.py;
  C5       prior query on the 400 x 200 x 16 voxel grid of one tile.

The checker is the CPU oracle run on the product model's own weights, rays and jitters.  Tolerances are the north
star's: 1e-3 scale-relative for the fp32 class ("b200+fp32"), 1e-2 for the bf16-MLP class ("b200").
"""
import os
import sys

import pytest
import torch

import oracle as O
from helpers import assert_close

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402  (oracle_model_from: oracle containers built from a product state dict)

pytestmark = pytest.mark.gpu
DEV = "cuda"


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def build(cfg_name, impl, n_rays):
    from presight_b200 import synthetic
    from presight_b200.model import NerfactoNuscMSModel
    cfg = bench.build_config(cfg_name, impl)
    torch.manual_seed(42)
    host = synthetic.make_rays(n_rays, seed=7)
    model = NerfactoNuscMSModel(cfg, torch.zeros(1, 3), synthetic.tile_aabb(), host["n_cameras"], host["n_videos"])
    with torch.no_grad():      # random-init tables are +-1e-3: scale them so that densities and colours are not trivial
        for f in model.field.fields:
            f.mlp_base_grid.hash_table.mul_(300.0)
        for p in model.proposal_networks:
            for f in p.fields:
                f.encoding.hash_table.mul_(300.0)
    return model.to(DEV).train(), cfg, host


def run_both(cfg_name, impl, n_rays):
    """-> (product outputs, oracle outputs, product model, oracle model) for one training-mode forward + backward of
    rgb MSE (+ semantic MSE) + interlevel loss, same weights / rays / jitters on both sides."""
    from presight_b200 import losses
    from presight_b200.cameras.rays import RayBundle
    from presight_b200.model import VIDEO_ID
    model, cfg, host = build(cfg_name, impl, n_rays)
    omodel, emb = bench.oracle_model_from(model, cfg)
    g = torch.Generator().manual_seed(3)
    jit = [torch.rand(n_rays, 1, generator=g) for _ in range(3)]
    rb = RayBundle(origins=host["origins"].to(DEV), directions=host["directions"].to(DEV),
                   camera_indices=host["camera_indices"].to(DEV), metadata={VIDEO_ID: host["video_ids"].to(DEV)})
    model.proposal_sampler._step = 0
    out = model(rb, jitters=[j.to(DEV) for j in jit])
    parts = []
    if cfg.appearance_embed_dim > 0:
        parts.append(emb["appearance_embedding.embedding.weight"][host["camera_indices"][:, 0]])
    if cfg.video_embed_dim > 0:
        parts.append(emb["video_embedding.embedding.weight"][host["video_ids"][:, 0]])
    app = torch.cat(parts, dim=-1) if parts else None
    oo = O.model_outputs(omodel, host["origins"], host["directions"], app, jit)

    loss = ((out["rgb"] - host["rgb"].to(DEV)) ** 2).mean()
    oloss = O.rgb_loss(host["rgb"], oo["rgb"])
    if cfg.use_semantics:
        loss = loss + 0.5 * ((out["semantics"] - host["features"].to(DEV).clip(0, 1)) ** 2).mean()
        oloss = oloss + 0.5 * O.semantic_loss(oo["semantics"], host["features"])
    loss = loss + losses.interlevel_loss(out["weights_list"], [rs.sp_bins for rs in out["ray_samples_list"]])
    oloss = oloss + O.interlevel_loss(oo["weights_list"], [b[0] for b in oo["bins_list"]])
    loss.backward()
    oloss.backward()
    assert_close(loss.detach().cpu(), oloss.detach(), 1e-3 if impl.endswith("fp32") else 1e-2, "loss")
    return out, oo, model, omodel


def frac_off(a, b, tol):
    """fraction of elements whose error exceeds tol x max|b|"""
    a, b = a.detach().cpu().double(), b.detach().double()
    return float(((a - b).abs() > tol * b.abs().max()).double().mean())


def check_outputs(out, oo, tol, keys):
    for k in keys:
        assert_close(out[k].detach().cpu(), oo[k], tol, k)
    # first level: identical bins by construction
    assert_close(out["weights_list"][0].detach().cpu(), oo["weights_list"][0], tol, "weights 0")
    # later levels: a weight that differs in the last bits can move a sample across a cdf edge (SURVEY §7), after which
    # that ray's bins differ; everything else must agree
    for i in (1, 2):
        assert frac_off(out["weights_list"][i], oo["weights_list"][i], tol) < 0.02, f"weights {i}"


@pytest.mark.parametrize("impl,tol,gtol", [("b200+fp32", 1e-3, 5e-3), ("b200", 1e-2, 5e-2)])
def test_c1_shapes_match_oracle(impl, tol, gtol):
    """C1 / C3: samples 256 / 96 / 48, hidden-16 proposal nets, no semantics, no sky model."""
    out, oo, model, om = run_both("c1", impl, 384)
    check_outputs(out, oo, tol, ("rgb", "accumulation", "expected_depth"))
    g = dict(model.named_parameters())
    assert rel_l2(g["field.fields.0.mlp_base_grid.hash_table"].grad.cpu(), om.fields[0].grid.table.grad) < gtol
    assert rel_l2(g["proposal_networks.0.fields.0.encoding.hash_table"].grad.cpu(), om.props[0][0].grid.table.grad) < gtol
    assert rel_l2(g["field.fields.0.rgb_head.layers.0.weight"].grad.cpu(), om.fields[0].rgb.weights[0].grad) < gtol


@pytest.mark.parametrize("impl,tol,gtol", [("b200+fp32", 1e-3, 5e-3), ("b200", 1e-2, 5e-2)])
def test_c2_config_matches_oracle(impl, tol, gtol):
    """C2 / C4: 2^22-entry main grid, samples 128 / 64 / 64, 64-d semantics, sky model; "b200" = the fused tcgen05
    proposal and field kernels (asserted), "b200+fp32" = the stand-alone kernels."""
    out, oo, model, om = run_both("c2", impl, 512)
    if impl == "b200":
        assert model.field.supports_fused()
    check_outputs(out, oo, tol, ("rgb", "accumulation", "expected_depth", "semantics"))
    g = dict(model.named_parameters())
    assert rel_l2(g["field.fields.0.mlp_base_grid.hash_table"].grad.cpu(), om.fields[0].grid.table.grad) < gtol
    assert rel_l2(g["proposal_networks.0.fields.0.encoding.hash_table"].grad.cpu(), om.props[0][0].grid.table.grad) < gtol
    assert rel_l2(g["field.fields.0.semantic_head.layers.2.weight"].grad.cpu(), om.fields[0].sem.weights[2].grad) < gtol
    assert rel_l2(g["field.fields.0.rgb_head.layers.0.weight"].grad.cpu(), om.fields[0].rgb.weights[0].grad) < gtol


def test_c2_loss_dict_matches_oracle():
    """`get_loss_dict` (rgb / sky / semantic / z-anti-aliased interlevel / distortion kernels) at C2 shapes: every term
    against the oracle's restatement of the reference's loss function evaluated on the SAME rendered outputs, weights
    and bins (so the comparison isolates the loss kernels from the sampling), fp32 tolerances."""
    from presight_b200.cameras.rays import RayBundle
    from presight_b200.model import VIDEO_ID
    n = 256
    model, cfg, host = build("c2", "b200", n)
    rb = RayBundle(origins=host["origins"].to(DEV), directions=host["directions"].to(DEV),
                   camera_indices=host["camera_indices"].to(DEV), metadata={VIDEO_ID: host["video_ids"].to(DEV)})
    model.proposal_sampler._step = 0
    out = model(rb)
    batch = {k: host[k].to(DEV) for k in ("rgb", "sky", "features")}
    ld = model.get_loss_dict(out, batch)
    assert set(ld) == {"rgb_loss", "sky_loss", "semantic_loss", "interlevel_loss", "distortion_loss"}
    wl = [w.detach().cpu() for w in out["weights_list"]]
    sp = [rs.sp_bins.detach().cpu() for rs in out["ray_samples_list"]]
    rgb, acc, sem = (out[k].detach().cpu() for k in ("rgb", "accumulation", "semantics"))
    want = {"rgb_loss": O.rgb_loss(host["rgb"], rgb),
            "sky_loss": cfg.sky_loss_mult * O.sky_loss(acc.view(-1, 1), host["sky"].view(-1, 1)),
            "semantic_loss": cfg.semantic_loss_mult * O.semantic_loss(sem, host["features"]),
            "interlevel_loss": cfg.interlevel_loss_mult * O.z_anti_aliasing_interlevel_loss(wl, sp, cfg.pulse_width),
            "distortion_loss": cfg.distortion_loss_mult * O.distortion_loss(wl, sp)}
    for k, v in want.items():
        assert_close(ld[k].detach().cpu(), v, 1e-4, k)
    sum(ld.values()).backward()
    grads = {k: p.grad for k, p in model.named_parameters() if p.grad is not None}
    assert len(grads) >= 30 and all(bool(torch.isfinite(g).all()) for g in grads.values())
    assert "proposal_networks.0.fields.0.encoding.hash_table" in grads and "field.fields.0.mlp_base_grid.hash_table" in grads


@pytest.mark.parametrize("lidar", [False, True])
def test_c2_loss_dict_with_depth_supervision(lidar):
    """`get_loss_dict` with a depth target (nerfacto_nusc_ms.py:577-629): expected-depth and line-of-sight terms from
    `ps_depth_losses` against the oracle's restatements on the SAME rendered depth / weights / bins, in the mono-depth
    and the LiDAR variant (which, as in the reference, wins when both are enabled and ignores the sky mask); the step
    drives the line-of-sight schedules; a missing pose scale factor is an error."""
    from presight_b200.cameras.rays import RayBundle
    from presight_b200.model import VIDEO_ID
    n = 256
    model, cfg, host = build("c2", "b200", n)
    cfg.use_monodepth_loss = True
    cfg.use_lidar_loss = lidar
    model.step = 12000                      # past line_of_sight_start_step: mult = 0.1 / 2^2, sigma between max and min
    scale = 0.05
    rb = RayBundle(origins=host["origins"].to(DEV), directions=host["directions"].to(DEV),
                   camera_indices=host["camera_indices"].to(DEV),
                   metadata={VIDEO_ID: host["video_ids"].to(DEV),
                             "pose_scale_factor": torch.full((n, 1), scale, device=DEV)})
    model.proposal_sampler._step = 0
    out = model(rb)
    g = torch.Generator().manual_seed(11)
    depth = torch.rand(n, generator=g) * 90.0
    batch = {k: host[k].to(DEV) for k in ("rgb", "sky", "features")}
    batch["depth"] = depth.to(DEV)
    ld = model.get_loss_dict(out, batch)
    assert {"expected_depth_loss", "line_of_sight_loss"} <= set(ld)
    last = out["ray_samples_list"][-1]
    eu = last.frustums.eu_bins.detach().cpu()
    steps = ((eu[:, :-1] + eu[:, 1:]) / 2 / scale)[..., None]
    pred = out["expected_depth"].detach().cpu() / scale
    w = out["weights_list"][-1].detach().cpu()
    sky = host["sky"].view(-1, 1)
    sigma, mult = O.line_of_sight_sigma(12000), O.line_of_sight_mult(12000)
    if lidar:
        want_e = O.expected_depth_loss(depth.view(-1, 1), pred, cfg.lidar_depth_upperbound)
        want_l = O.line_of_sight_loss(w, depth.view(-1, 1), steps, sigma, None, cfg.lidar_depth_upperbound)
    else:
        want_e = O.expected_monodepth_loss(depth.view(-1, 1), pred, sky, cfg.monodepth_depth_upperbound, False)
        want_l = O.line_of_sight_loss(w, depth.view(-1, 1), steps, sigma, sky, cfg.monodepth_depth_upperbound)
    assert_close(ld["expected_depth_loss"].detach().cpu(), cfg.expected_depth_loss_mult * want_e, 1e-4, "expected depth")
    assert_close(ld["line_of_sight_loss"].detach().cpu(), mult * want_l, 1e-4, "line of sight")
    sum(ld.values()).backward()
    assert all(bool(torch.isfinite(p.grad).all()) for p in model.parameters() if p.grad is not None)
    rb2 = RayBundle(origins=rb.origins, directions=rb.directions, camera_indices=rb.camera_indices,
                    metadata={VIDEO_ID: host["video_ids"].to(DEV)})
    out2 = model(rb2)
    with pytest.raises(KeyError, match="pose_scale_factor"):
        model.get_loss_dict(out2, batch)


@pytest.mark.parametrize("impl,tol", [("b200+fp32", 1e-3), ("b200", 1e-2)])
def test_c5_prior_query_full_grid(impl, tol):
    """C5: the 400 x 200 x 16 grid of one tile (1.28 M points) through query_priors; the oracle checks a random
    20 000-point subset, and the subset queried on its own must reproduce the full run's rows exactly (points are
    independent units — what lets tiles / slabs shard over GPUs with no communication)."""
    model, cfg, _ = build("c2", impl, 8)
    model.eval()
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from bench_prior_query import tile_grid
    pts = tile_grid(0, DEV)
    assert pts.shape == (400 * 200 * 16, 3)
    mean, feats = model.query_priors(pts)
    assert mean.shape == (pts.shape[0],) and feats.shape == (pts.shape[0], 64) and feats.dtype == torch.float16
    assert bool(torch.isfinite(mean).all()) and float(feats.float().min()) >= 0.0 and float(feats.float().max()) <= 1.0
    idx = torch.randperm(pts.shape[0], generator=torch.Generator().manual_seed(0))[:20000].to(DEV)
    m2, f2 = model.query_priors(pts[idx].contiguous())
    assert torch.equal(m2, mean[idx]) and torch.equal(f2, feats[idx])
    omodel, _ = bench.oracle_model_from(model, cfg)
    om, of = O.prior_query(omodel, pts[idx].cpu())
    assert_close(m2.cpu(), om, tol, "mean density")
    assert_close(f2.float().cpu(), of.float(), tol, "semantic features")
