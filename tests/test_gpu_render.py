"""Rendering whole camera images and scoring them on the device: ps_image_metrics against the numpy oracle, the chunked
`get_outputs_for_camera_ray_bundle` against `forward` on the same slices, `RayGenerator.image_rays`, and the model's
metric hooks (`get_image_metrics_and_images`, `get_metrics_dict`)."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import metrics_oracle as MO
from test_gpu_extract import c2_model, presight_model
from test_metrics_host import image_pair

pytestmark = pytest.mark.gpu
DEV = "cuda"


def on_dev(*arrays):
    return [torch.from_numpy(a).to(DEV) for a in arrays]


@pytest.mark.parametrize("kind", ["random", "smooth", "edge"])
@pytest.mark.parametrize("H,W", [(11, 11), (12, 37), (900, 1600)])
def test_image_metrics_match_oracle(kind, H, W):
    from presight_b200 import metrics
    pred, gt = image_pair(kind, H, W, seed=H + W)
    psnr, ssim, sse = metrics.image_metrics(*on_dev(pred, gt))
    assert psnr.dtype == torch.float32 and ssim.dtype == sse.dtype == torch.float64 and psnr.shape == (1,)
    d = (pred - gt).astype(np.float64)
    assert float(sse[0]) == pytest.approx(float(np.sum(d * d)), rel=1e-12)
    assert abs(float(psnr[0]) - MO.psnr(pred, gt)) <= 1e-4
    assert abs(float(ssim[0]) - MO.ssim(pred, gt)) <= 1e-5
    assert float(metrics.psnr(*on_dev(pred, gt))) == float(psnr[0])
    assert float(metrics.ssim(*on_dev(pred, gt))) == float(ssim[0])


def test_batch_gives_each_image_its_own_data_range():
    from presight_b200 import metrics
    pairs = [image_pair(k, 70, 90, seed=i) for i, k in enumerate(("random", "smooth", "edge"))]
    # different spreads per image: the SSIM constants follow each image's own range
    pairs = [(p * s + o, g * s + o) for (p, g), s, o in zip(pairs, (1.0, 0.3, 2.0), (0.0, 0.5, -1.0))]
    pred = np.stack([p for p, _ in pairs]).astype(np.float32)
    gt = np.stack([g for _, g in pairs]).astype(np.float32)
    psnr, ssim, _ = metrics.image_metrics(*on_dev(pred, gt))
    assert psnr.shape == ssim.shape == (3,)
    for i in range(3):
        assert abs(float(psnr[i]) - MO.psnr(pred[i], gt[i])) <= 1e-4
        assert abs(float(ssim[i]) - MO.ssim(pred[i], gt[i])) <= 1e-5
        alone = metrics.image_metrics(*on_dev(pred[i], gt[i]))
        assert float(alone[1][0]) == float(ssim[i])


def test_repeated_launches_are_bit_identical_and_special_values():
    from presight_b200 import metrics
    pred, gt = on_dev(*image_pair("random", 900, 1600, seed=1))
    a, b = metrics.image_metrics(pred, gt), metrics.image_metrics(pred, gt)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    psnr, ssim, sse = metrics.image_metrics(gt, gt)
    assert float(sse[0]) == 0.0 and float(psnr[0]) == float("inf") and float(ssim[0]) == 1.0
    c = torch.full((30, 40, 3), 0.3, device=DEV)
    assert torch.isnan(metrics.ssim(c, torch.full_like(c, 0.7)))


def test_invalid_shapes_are_rejected():
    from presight_b200 import _lib, metrics
    lib = _lib.load()
    pred, gt = on_dev(*image_pair("random", 12, 12, seed=0))
    ws = torch.empty(1 << 16, dtype=torch.uint8, device=DEV)
    out32, out64 = torch.empty(1, device=DEV), torch.empty(2, dtype=torch.float64, device=DEV)
    for H, W in ((10, 12), (12, 10), (0, 12)):
        rc = lib.ps_image_metrics(pred.data_ptr(), gt.data_ptr(), 1, H, W, 1.0, ws.data_ptr(), None, out32.data_ptr(),
                                  out64.data_ptr(), _lib.stream())
        assert rc == 1, (H, W)
        assert b"11" in lib.ps_last_error() or b"empty" in lib.ps_last_error()
    nbytes = C.c_int64(0)
    assert lib.ps_image_metrics_workspace(1, -1, 12, C.byref(nbytes)) == 1
    with pytest.raises(RuntimeError, match="11 x 11"):
        metrics.ssim(pred[:10], gt[:10])
    with pytest.raises(ValueError):
        metrics.image_metrics(pred, gt[:11])
    # PSNR alone takes any size, e.g. a ray batch
    assert abs(float(metrics.psnr(pred[:3, :2], gt[:3, :2])) - MO.psnr(pred[:3, :2].cpu().numpy(),
                                                                         gt[:3, :2].cpu().numpy())) <= 1e-4


def ray_generator():
    from presight_b200 import synthetic
    from presight_b200.cameras.ray_generator import RayGenerator
    cams = synthetic.make_cameras(seed=42, n_frames=4)
    return RayGenerator(cams["camera_to_worlds"], cams["fx"], cams["fy"], cams["cx"], cams["cy"]).to(DEV)


def test_image_rays_equal_forward_on_explicit_indices():
    gen = ray_generator()
    H, W, cam = 45, 61, 7
    rb = gen.image_rays(cam, H, W)
    rr, cc = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    idx = torch.stack([torch.full((H, W), cam), rr, cc], dim=-1).reshape(-1, 3).to(DEV)
    want = gen(idx)
    assert rb.origins.shape == (H, W, 3) and rb.camera_indices.shape == (H, W, 1)
    for name in ("origins", "directions", "pixel_area", "camera_indices"):
        assert torch.equal(getattr(rb, name).reshape(H * W, -1), getattr(want, name)), name
    assert torch.equal(rb.metadata["directions_norm"].reshape(H * W, -1), want.metadata["directions_norm"])
    assert int(rb.camera_indices.min()) == int(rb.camera_indices.max()) == cam


@pytest.mark.parametrize("shape", ["c2", "presight16"])
def test_camera_ray_bundle_is_forward_on_consecutive_slices(shape):
    from presight_b200.cameras.rays import RayBundle
    model, _ = c2_model() if shape == "c2" else presight_model()
    model.config.eval_num_rays_per_chunk = 1000
    H, W = 37, 53                                            # 1961 rays: one full chunk and a partial one
    rb = ray_generator().image_rays(5, H, W)
    out = model.get_outputs_for_camera_ray_bundle(rb)
    flat = {k: v.reshape(H * W, -1) for k, v in (("o", rb.origins), ("d", rb.directions), ("a", rb.pixel_area),
                                                 ("c", rb.camera_indices), ("n", rb.metadata["directions_norm"]))}
    parts = []
    with torch.no_grad():
        for i in range(0, H * W, 1000):
            s = slice(i, i + 1000)
            parts.append(model(RayBundle(origins=flat["o"][s], directions=flat["d"][s], pixel_area=flat["a"][s],
                                         camera_indices=flat["c"][s], metadata={"directions_norm": flat["n"][s]})))
    assert set(out) == {k for k, v in parts[0].items() if torch.is_tensor(v)}
    for k, v in out.items():
        want = torch.cat([p[k] for p in parts])
        assert v.shape[:2] == (H, W)
        assert torch.equal(v.reshape(want.shape), want), k
    assert out["rgb"].shape == (H, W, 3) and out["depth"].shape == (H, W, 1)


def test_image_metrics_and_images_of_a_rendered_image():
    model, _ = c2_model()
    H, W = 48, 64
    out = model.get_outputs_for_camera_ray_bundle(ray_generator().image_rays(2, H, W))
    gt = torch.rand(H, W, 3, generator=torch.Generator().manual_seed(3)).to(DEV)
    m, imgs = model.get_image_metrics_and_images(out, {"rgb": gt})
    pred = out["rgb"].cpu().numpy()
    assert set(m) == {"psnr", "ssim"} and all(isinstance(v, float) for v in m.values())
    assert abs(m["psnr"] - MO.psnr(pred, gt.cpu().numpy())) <= 1e-4
    assert abs(m["ssim"] - MO.ssim(pred, gt.cpu().numpy())) <= 1e-5
    assert torch.equal(imgs["img"], torch.cat([gt, out["rgb"]], dim=1)) and imgs["img"].shape == (H, 2 * W, 3)
    assert imgs["accumulation"].shape == imgs["depth"].shape == (H, W, 1)


def test_metrics_dict_is_a_device_scalar():
    model, _ = c2_model()
    g = torch.Generator().manual_seed(4)
    rgb = torch.rand(10000, 3, generator=g).to(DEV).requires_grad_(True)
    target = torch.rand(10000, 3, generator=g).to(DEV)
    d = model.get_metrics_dict({"rgb": rgb}, {"rgb": target})
    assert set(d) == {"psnr"} and d["psnr"].is_cuda and d["psnr"].dim() == 0
    assert abs(float(d["psnr"]) - MO.psnr(rgb.detach().cpu().numpy(), target.cpu().numpy())) <= 1e-4
