"""Geometry metrics on the device: `ps_depth_metrics` against the fp64 oracle, the nearest-neighbour grid against
cKDTree (random, adversarial and LiDAR-like clouds, up to 2^22 x 2^24 points), chunking and repeatability, the ABI's
argument checks, and the depth keys of the model's evaluation hooks."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import geometry_oracle as GO
from test_geometry_host import assert_depth_close, depth_case

pytestmark = pytest.mark.gpu
DEV = "cuda"


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


# ---- depth metrics --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M", [1, 2, 4])
@pytest.mark.parametrize("H,W", [(31, 31), (97, 173), (900, 1600)])
def test_depth_metrics_match_oracle(H, W, M):
    from presight_b200 import geometry
    preds, t = depth_case(H, W, M, seed=H * 7 + M)
    got = geometry.depth_metrics([dev(p) for p in preds], dev(t), 0.0123)
    assert got.dtype == torch.float64 and got.shape == (M, 8) and got.is_cuda
    assert_depth_close(got.cpu().numpy(), GO.depth_metrics(preds, t, 0.0123), rel=1e-9)
    # the pose scale as a device scalar gives the same bits
    again = geometry.depth_metrics([dev(p) for p in preds], dev(t), torch.tensor([0.0123], device=DEV))
    assert torch.equal(got, again)


def test_depth_metrics_repeatable_shapes_and_no_valid_pixel():
    from presight_b200 import geometry
    preds, t = depth_case(900, 1600, 2, seed=5)
    maps = [dev(p)[..., None] for p in preds]                 # [H,W,1] as the renderer returns them
    a = geometry.depth_metrics(maps, dev(t), 0.0123)
    b = geometry.depth_metrics(maps, dev(t)[..., None], 0.0123)
    assert torch.equal(a, b)
    assert torch.equal(geometry.depth_metrics(maps[0], dev(t), 0.0123), a[:1])
    none = geometry.depth_metrics(maps, torch.zeros(900, 1600, device=DEV), 0.0123)
    assert torch.isnan(none[:, :7]).all() and (none[:, 7] == 0).all()
    lo = geometry.depth_metrics(maps, dev(t), 0.0123, min_m=2.0, max_m=40.0)
    assert_depth_close(lo.cpu().numpy(), GO.depth_metrics(preds, t, 0.0123, 2.0, 40.0), rel=1e-9)
    with pytest.raises(ValueError):
        geometry.depth_metrics(maps * 3, dev(t), 1.0)
    with pytest.raises(ValueError):
        geometry.depth_metrics(maps, dev(t)[:10], 1.0)
    with pytest.raises(ValueError):
        geometry.depth_metrics(maps, dev(t), 0.0)
    with pytest.raises(ValueError):
        geometry.depth_metrics(maps, dev(t), 1.0, min_m=0.0)


def test_depth_metrics_abi_checks():
    from presight_b200 import _lib
    lib = _lib.load()
    nbytes = C.c_int64(0)
    assert lib.ps_depth_metrics_workspace(2, 1440000, C.byref(nbytes)) == 0 and nbytes.value > 0
    assert lib.ps_depth_metrics_workspace(0, 10, C.byref(nbytes)) == 1
    assert lib.ps_depth_metrics_workspace(5, 10, C.byref(nbytes)) == 1
    assert lib.ps_depth_metrics_workspace(1, 0, C.byref(nbytes)) == 1
    x = torch.ones(2, 100, device=DEV)
    ws = torch.empty(1 << 16, dtype=torch.uint8, device=DEV)
    out = torch.empty(2, 8, dtype=torch.float64, device=DEV)
    good = dict(pred=x.data_ptr(), M=2, HW=100, t=x.data_ptr(), s=1.0, sd=None, lo=1.0, hi=75.0, ws=ws.data_ptr(),
                out=out.data_ptr())

    def run(**kw):
        a = dict(good, **kw)
        return lib.ps_depth_metrics(a["pred"], a["M"], a["HW"], a["t"], a["s"], a["sd"], a["lo"], a["hi"], a["ws"],
                                    a["out"], _lib.stream())

    assert run() == 0
    torch.cuda.synchronize()
    for kw, msg in [(dict(M=0), b"M must be"), (dict(M=5), b"M must be"), (dict(HW=0), b"HW must be"),
                    (dict(pred=None), b"null"), (dict(t=None), b"null"), (dict(ws=None), b"null"),
                    (dict(out=None), b"null"), (dict(s=0.0), b"pose scale"), (dict(lo=0.0), b"min_m"),
                    (dict(lo=80.0), b"min_m"), (dict(hi=float("inf")), b"min_m")]:
        assert run(**kw) == 1, kw
        assert msg in lib.ps_last_error(), (kw, lib.ps_last_error())


# ---- nearest neighbours ---------------------------------------------------------------------------------------------
def lidar_like(n, seed, noise=0.02, extent=60.0):
    """Points as a LiDAR sees a street: rings on the ground around a few sensor positions, and facades (vertical planes),
    plus noise; metres, f32."""
    rng = np.random.default_rng(seed)
    n_ring = n // 2
    centres = rng.uniform(-extent / 2, extent / 2, (8, 2))
    c = centres[rng.integers(0, 8, n_ring)]
    rad = rng.choice(np.geomspace(2.0, extent / 2, 32), n_ring)
    ang = rng.uniform(0, 2 * np.pi, n_ring)
    ground = np.stack([c[:, 0] + rad * np.cos(ang), c[:, 1] + rad * np.sin(ang), np.full(n_ring, -1.8)], 1)
    n_wall = n - n_ring
    side = rng.integers(0, 4, n_wall)
    u, h = rng.uniform(-extent / 2, extent / 2, n_wall), rng.uniform(-1.8, 12.0, n_wall)
    pos = np.where(side % 2 == 0, extent / 2, -extent / 2)
    walls = np.where((side < 2)[:, None], np.stack([pos, u, h], 1), np.stack([u, pos, h], 1))
    pts = np.concatenate([ground, walls]) + rng.normal(0, noise, (n, 3))
    return pts[rng.permutation(n)].astype(np.float32)


def adversarial(kind, r, seed=0):
    """(queries, reference) with points on cell faces, edges and corners of the grid, or everything in one cell."""
    rng = np.random.default_rng(seed)
    if kind == "faces_corners":
        g = np.arange(-4, 5) * r
        lattice = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
        ref = np.concatenate([lattice, lattice[::3] + np.array([r / 2, 0, 0]), lattice[::5] + np.array([0, r / 2, r / 2])])
        q = np.concatenate([lattice + rng.choice([-1, 0, 1], lattice.shape) * r / 4, lattice[::2] + r * 0.999,
                            rng.uniform(-5 * r, 5 * r, (500, 3))])
        return q.astype(np.float32), ref.astype(np.float32)
    if kind == "one_cell":
        ref = rng.uniform(0, r * 0.999, (3000, 3))
        q = rng.uniform(-r, 2 * r, (2000, 3))
        return q.astype(np.float32), ref.astype(np.float32)
    if kind == "far_queries":                       # queries outside the reference's extent, below and above
        ref = rng.uniform(0, 5 * r, (1000, 3))
        q = np.concatenate([rng.uniform(-3 * r, 0, (300, 3)), rng.uniform(5 * r, 8 * r, (300, 3)),
                            np.array([[-1e6, 0, 0], [1e6, 1e6, 1e6]])])
        return q.astype(np.float32), ref.astype(np.float32)
    pts = lidar_like(20000, seed)
    return lidar_like(8000, seed + 1, noise=0.05), pts


def check_nn(q, ref, r, taus, chunk=1 << 22):
    from presight_b200 import geometry
    grid = geometry.NNGrid(dev(ref), r)
    mean, counts, d = grid.query(dev(q), taus, chunk=chunk, return_distances=True)
    want = GO.nn_distances(q, ref, r)
    got = d.cpu().numpy()
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)
    assert counts.tolist() == [int((want < t).sum()) for t in taus]
    assert float(mean) == pytest.approx(want.mean(), rel=1e-12)
    return grid, mean, counts, d


@pytest.mark.parametrize("r", [0.4, 1.0])
@pytest.mark.parametrize("kind", ["random", "faces_corners", "one_cell", "far_queries", "lidar"])
def test_nn_distances_match_ckdtree(kind, r):
    if kind == "random":
        rng = np.random.default_rng(3)
        q, ref = rng.uniform(-5, 5, (7000, 3)).astype(np.float32), rng.uniform(-5, 5, (9000, 3)).astype(np.float32)
    else:
        q, ref = adversarial(kind, r)
    check_nn(q, ref, r, (r / 8, r / 3, r / 2, r))


def test_nn_one_point_and_duplicates():
    ref = np.array([[1.0, -2.0, 3.0]], np.float32)
    q = np.concatenate([ref, ref + 0.3, ref + 5.0]).astype(np.float32)
    check_nn(q, ref, 0.6, (0.1, 0.6))
    dup = np.repeat(lidar_like(500, 9), 4, axis=0)
    check_nn(lidar_like(700, 10), dup, 0.5, (0.05, 0.5))


def test_chunked_queries_equal_one_shot_and_are_repeatable():
    from presight_b200 import geometry
    q, ref = lidar_like(50000, 4, noise=0.05), lidar_like(80000, 5)
    grid, mean, counts, d = check_nn(q, ref, 0.4, (0.05, 0.1, 0.2))
    for chunk in (1024, 3 * 1024, 5000):
        m2, c2, d2 = grid.query(dev(q), (0.05, 0.1, 0.2), chunk=chunk, return_distances=True)
        assert torch.equal(m2, mean) and torch.equal(c2, counts) and torch.equal(d2, d), chunk
    a = geometry.prior_geometry_metrics(dev(q), dev(ref), 0.4, (0.05, 0.1, 0.2))
    b = geometry.prior_geometry_metrics(dev(q), dev(ref), 0.4, (0.05, 0.1, 0.2), chunk=2048)
    assert a.keys() == b.keys() and all(torch.equal(a[k], b[k]) for k in a)


def test_prior_geometry_metrics_large():
    """2^22 priors against 2^24 reference points, both directions against cKDTree."""
    from presight_b200 import geometry
    ref = lidar_like(1 << 24, 21, extent=120.0)
    prior = lidar_like(1 << 22, 22, noise=0.05, extent=120.0)
    taus = (0.05, 0.1, 0.2)
    got = geometry.prior_geometry_metrics(dev(prior), dev(ref), 0.4, taus, return_distances=True)
    want = GO.prior_geometry_metrics(prior, ref, 0.4, taus)
    for k in ("prior_to_ref", "ref_to_prior"):
        np.testing.assert_allclose(got[k].cpu().numpy(), want[k], rtol=1e-12, atol=0)
    for k in ("accuracy", "completeness"):
        assert float(got[k]) == pytest.approx(float(want[k]), rel=1e-12)
    for k in ("precision", "recall"):
        assert got[k].tolist() == want[k].tolist(), k         # counts are exact, so the fractions are equal
    np.testing.assert_allclose(got["fscore"].cpu().numpy(), want["fscore"], rtol=1e-14)


def test_prior_geometry_metrics_errors_and_abi():
    from presight_b200 import _lib, geometry
    pts = dev(lidar_like(100, 1))
    for args in ((pts[:0], pts), (pts, pts[:0])):
        with pytest.raises(ValueError, match="empty"):
            geometry.prior_geometry_metrics(*args, 0.4, (0.1,))
    with pytest.raises(ValueError, match="threshold"):
        geometry.prior_geometry_metrics(pts, pts, 0.4, (0.5,))
    with pytest.raises(ValueError, match="at most"):
        geometry.prior_geometry_metrics(pts, pts, 0.4, (0.1,) * 9)
    wide = pts.clone()
    wide[0, 0] = 1e6
    with pytest.raises(RuntimeError, match="2\\^21"):
        geometry.NNGrid(wide, 0.4)
    m = geometry.prior_geometry_metrics(pts, pts, 0.4, (0.1,))
    assert float(m["accuracy"]) == float(m["completeness"]) == 0.0 and m["fscore"].tolist() == [1.0]
    lib = _lib.load()
    assert lib.ps_nn_grid_reduce(None, None, 0, 0, 1, None, None, None) == 1
    assert lib.ps_nn_grid_query(None, None, 1, 0, None, 0, None, None, None, None) == 1


# ---- model hooks ----------------------------------------------------------------------------------------------------
def rendered_c2(H=48, W=64, cam=2):
    from test_gpu_extract import c2_model
    from test_gpu_render import ray_generator
    model, cfg = c2_model()
    out = model.get_outputs_for_camera_ray_bundle(ray_generator().image_rays(cam, H, W))
    return model, cfg, out


def lidar_image(out, scale, seed):
    """A target near the rendered depth, in metres, with holes."""
    g = torch.Generator().manual_seed(seed)
    d = out["depth"][..., 0].cpu() / scale
    t = d * torch.exp(0.1 * torch.randn(d.shape, generator=g))
    t[torch.rand(d.shape, generator=g) < 0.3] = 0.0
    return t.to(DEV)


def test_model_hook_depth_keys():
    from presight_b200 import geometry
    model, cfg, out = rendered_c2()
    H, W = out["rgb"].shape[:2]
    gt = torch.rand(H, W, 3, generator=torch.Generator().manual_seed(3)).to(DEV)
    scale = float(out["depth"].median()) / 30.0               # the median rendered depth at 30 m
    target = lidar_image(out, scale, 1)
    base_m, base_imgs = model.get_image_metrics_and_images(out, {"rgb": gt})
    m, imgs = model.get_image_metrics_and_images(out, {"rgb": gt, "depth": target, "pose_scale_factor": scale})
    dm = geometry.depth_metrics([out["depth"], out["expected_depth"]], target, scale, 1.0, cfg.lidar_depth_upperbound)
    names = geometry.DEPTH_METRICS[:7]
    assert 0 < float(dm[0, 7]) < H * W
    want = {f"{p}_{n}": float(dm[i, j]) for i, p in enumerate(("depth", "expected_depth")) for j, n in enumerate(names)}
    assert m == {**base_m, **want}
    assert imgs.keys() == base_imgs.keys() and all(torch.equal(imgs[k], base_imgs[k]) for k in imgs)
    # a device pose scale and an [H,W,1] target give the same numbers
    m2, _ = model.get_image_metrics_and_images(out, {"rgb": gt, "depth": target[..., None],
                                                     "pose_scale_factor": torch.tensor([[scale]], device=DEV)})
    assert m2 == m
    with pytest.raises(KeyError, match="pose_scale_factor"):
        model.get_image_metrics_and_images(out, {"rgb": gt, "depth": target})


def test_eval_loop_with_depth_frames():
    from presight_b200 import evaluate
    from test_gpu_render import ray_generator
    model, _, _ = rendered_c2()
    gen = ray_generator()
    H, W = 40, 48
    scale = float(model.get_outputs_for_camera_ray_bundle(gen.image_rays(1, H, W))["depth"].median()) / 30.0
    g = torch.Generator().manual_seed(8)
    frames = []
    for i in range(3):
        cam = 2 * i + 1
        out = model.get_outputs_for_camera_ray_bundle(gen.image_rays(cam, H, W))
        frames.append((cam, torch.rand(H, W, 3, generator=g).to(DEV), lidar_image(out, scale, 10 + i)))
    per = []
    for cam, img, depth in frames:
        out = model.get_outputs_for_camera_ray_bundle(gen.image_rays(cam, H, W))
        per.append(model.get_image_metrics_and_images(out, {"rgb": img, "depth": depth, "pose_scale_factor": scale})[0])
    got = evaluate.average_eval_image_metrics(model, gen, frames, pose_scale_factor=scale)
    assert "depth_abs_rel" in got and "expected_depth_a3" in got and "psnr" in got
    for k in per[0]:
        assert got[k] == float(torch.mean(torch.tensor([p[k] for p in per]))), k
    two = evaluate.average_eval_image_metrics(model, gen, [f[:2] for f in frames])
    two_scaled = evaluate.average_eval_image_metrics(model, gen, [f[:2] for f in frames], pose_scale_factor=scale)
    plain = [model.get_image_metrics_and_images(
        model.get_outputs_for_camera_ray_bundle(gen.image_rays(cam, H, W)), {"rgb": img})[0] for cam, img, _ in frames]
    assert set(two) == set(two_scaled) == {"psnr", "ssim", "num_rays_per_sec", "fps"}
    for k in ("psnr", "ssim"):
        assert two[k] == two_scaled[k] == float(torch.mean(torch.tensor([p[k] for p in plain]))), k
    with pytest.raises(ValueError, match="with and without depth"):
        evaluate.average_eval_image_metrics(model, gen, [frames[0], frames[1][:2]], pose_scale_factor=scale)
