"""The evaluation outputs on the device: `ps_colormap` bit for bit against torch running nerfstudio's colormaps, its
ABI checks, the model's `colormap` hook on a rendered image, and `average_eval_image_metrics` against the per-frame
metrics it averages."""
import ctypes as C

import pytest
import torch

from test_colormap_host import colormap_case, seeded_lut, torchvision_and_lin
from test_gpu_extract import c2_model

pytestmark = pytest.mark.gpu
DEV = "cuda"


# nerfstudio 0.3.3 utils/colormaps.py with default ColormapOptions, restated literally in torch (the LUT passed in)
def apply_float_colormap(x, lut):                      # x [H,W,1]
    x = torch.nan_to_num(x, 0)
    return lut[(x * 255).long()[..., 0]]


def apply_colormap(x, lut):                            # normalize=False, colormap_min=0, colormap_max=1, invert=False
    return apply_float_colormap(torch.clip(x * (1.0 - 0.0) + 0.0, 0, 1), lut)


def apply_depth_colormap(depth, accumulation, lut):
    near, far = float(torch.min(depth)), float(torch.max(depth))
    depth = torch.clip((depth - near) / (far - near + 1e-10), 0, 1)
    c = apply_colormap(depth, lut)
    return c * accumulation + (1 - accumulation)


def oracle(maps, acc, lut):
    return apply_colormap(acc, lut), [apply_depth_colormap(d, acc, lut) for d in maps]


def case_on_dev(kind, H, W, M, seed):
    maps, acc = colormap_case(kind, H, W, M, seed=seed)
    return [torch.from_numpy(m[..., None].copy()).to(DEV) for m in maps], torch.from_numpy(acc[..., None]).to(DEV)


@pytest.mark.parametrize("M", [0, 1, 3])
@pytest.mark.parametrize("H,W", [(37, 53), (900, 1600)])
@pytest.mark.parametrize("kind", ["random", "constant", "boundaries", "special"])
def test_colormap_equals_torch(kind, H, W, M):
    from presight_b200 import metrics
    maps, acc = case_on_dev(kind, H, W, M, seed=H + M)
    lut = torch.from_numpy(seeded_lut(M)).to(DEV)
    acc_img, depth_imgs = metrics.colormap_images(maps, acc, lut)
    want_acc, want_depths = oracle(maps, acc, lut)
    assert acc_img.shape == (H, W, 3) and len(depth_imgs) == M
    assert torch.equal(acc_img, want_acc)
    for m in range(M):
        assert torch.equal(depth_imgs[m], want_depths[m]), (kind, m)


def test_repeated_calls_are_bit_identical_and_abi_checks():
    from presight_b200 import _lib, metrics
    maps, acc = case_on_dev("random", 900, 1600, 3, seed=1)
    lut = torch.from_numpy(seeded_lut(1)).to(DEV)
    a, b = metrics.colormap_images(maps, acc, lut), metrics.colormap_images(maps, acc, lut)
    assert torch.equal(a[0], b[0]) and all(torch.equal(x, y) for x, y in zip(a[1], b[1]))

    lib = _lib.load()
    nbytes = C.c_int64(0)
    assert lib.ps_colormap_workspace(3, 900 * 1600, C.byref(nbytes)) == 0 and 0 < nbytes.value <= 3 * 256 * 8
    assert lib.ps_colormap_workspace(0, 10, C.byref(nbytes)) == 0 and nbytes.value == 0
    assert lib.ps_colormap_workspace(-1, 10, C.byref(nbytes)) == 1
    assert lib.ps_colormap_workspace(1, 0, C.byref(nbytes)) == 1
    assert lib.ps_colormap_workspace(1, 10, None) == 1
    HW = 37 * 53
    stacked = torch.rand(3, HW, device=DEV)
    flat_acc = torch.rand(HW, device=DEV)
    assert lib.ps_colormap_workspace(3, HW, C.byref(nbytes)) == 0
    ws = torch.empty(nbytes.value, dtype=torch.uint8, device=DEV)
    out = torch.empty(4, HW, 3, device=DEV)
    good = dict(maps=stacked.data_ptr(), M=3, HW=HW, acc=flat_acc.data_ptr(), lut=lut.data_ptr(), ws=ws.data_ptr(),
                out=out.data_ptr())

    def run(**kw):
        x = dict(good, **kw)
        return lib.ps_colormap(x["maps"], x["M"], x["HW"], x["acc"], x["lut"], x["ws"], x["out"], _lib.stream())

    assert run() == 0
    assert run(maps=None, ws=None, M=0) == 0                   # no maps: the accumulation image only
    torch.cuda.synchronize()
    cases = [(dict(M=-1), b"M must be"), (dict(M=1025), b"M must be"), (dict(HW=0), b"HW must be"),
             (dict(HW=-5), b"HW must be"), (dict(maps=None), b"null"), (dict(ws=None), b"null"),
             (dict(acc=None), b"null"), (dict(lut=None), b"null"), (dict(out=None), b"null")]
    for kw, msg in cases:
        assert run(**kw) == 1, kw
        assert msg in lib.ps_last_error(), (kw, lib.ps_last_error())
    with pytest.raises(ValueError, match="256,3"):
        metrics.colormap_images(maps, acc, lut[:255])
    with pytest.raises(ValueError, match="differ in shape"):
        metrics.colormap_images([maps[0][:10]], acc, lut)
    with pytest.raises(ValueError, match=r"\[H,W,1\]"):
        metrics.colormap_images([], acc[..., 0], lut)


def ray_gen():
    from test_gpu_render import ray_generator
    return ray_generator()


def test_model_hook_on_a_rendered_image():
    model, cfg = c2_model()
    H, W = 48, 64
    out = model.get_outputs_for_camera_ray_bundle(ray_gen().image_rays(3, H, W))
    gt = torch.rand(H, W, 3, generator=torch.Generator().manual_seed(6)).to(DEV)
    keys = set(model.state_dict().keys())
    raw_m, raw = model.get_image_metrics_and_images(out, {"rgb": gt})
    lut = torch.from_numpy(seeded_lut(7)).to(DEV)
    model.colormap = lut
    try:
        assert set(model.state_dict().keys()) == keys
        m, imgs = model.get_image_metrics_and_images(out, {"rgb": gt})
    finally:
        model.colormap = None
    assert m == raw_m
    assert set(imgs) == {"img", "accumulation", "depth", "prop_depth_0", "prop_depth_1"}
    assert torch.equal(imgs["img"], raw["img"])
    acc = out["accumulation"]
    assert torch.equal(imgs["accumulation"], apply_colormap(acc, lut))
    for k in ("depth", "prop_depth_0", "prop_depth_1"):
        assert imgs[k].shape == (H, W, 3)
        assert torch.equal(imgs[k], apply_depth_colormap(out[k], acc, lut)), k
    assert set(model.get_image_metrics_and_images(out, {"rgb": gt})[1]) == {"img", "accumulation", "depth"}


def frames(n=3, H=40, W=48):
    g = torch.Generator().manual_seed(8)
    return [(2 * i + 1, torch.rand(H, W, 3, generator=g).to(DEV)) for i in range(n)]


@pytest.mark.parametrize("get_std", [False, True])
def test_average_eval_image_metrics(get_std):
    from presight_b200 import evaluate
    from presight_b200.metrics import LPIPS
    model, _ = c2_model()
    model.lpips = LPIPS.from_state_dicts(*torchvision_and_lin(3), device=DEV)
    gen = ray_gen()
    fr = frames()
    try:
        per = []
        for cam, img in fr:
            out = model.get_outputs_for_camera_ray_bundle(gen.image_rays(cam, *img.shape[:2]))
            per.append(model.get_image_metrics_and_images(out, {"rgb": img})[0])
        model.train()
        got = evaluate.average_eval_image_metrics(model, gen, iter(fr), get_std=get_std)
        assert model.training                                  # the previous mode is restored
        model.eval()
        evaluate.average_eval_image_metrics(model, gen, fr[:1])
        assert not model.training
    finally:
        model.lpips = None
    base = {"psnr", "ssim", "lpips", "num_rays_per_sec", "fps"}
    assert set(got) == (base | {f"{k}_std" for k in base} if get_std else base)
    for k in ("psnr", "ssim", "lpips"):
        vals = torch.tensor([p[k] for p in per])
        if get_std:
            std, mean = torch.std_mean(vals)
            assert got[k] == float(mean) and got[f"{k}_std"] == float(std), k
        else:
            assert got[k] == float(torch.mean(vals)), k
    assert got["num_rays_per_sec"] > 0 and 0 < got["fps"] < got["num_rays_per_sec"]


def test_average_eval_image_metrics_restores_the_mode_on_error():
    from presight_b200 import evaluate
    model, _ = c2_model()
    model.train()

    def broken():
        yield frames(1)[0]
        raise RuntimeError("frame source failed")

    with pytest.raises(RuntimeError, match="frame source failed"):
        evaluate.average_eval_image_metrics(model, ray_gen(), broken())
    assert model.training
    with pytest.raises(ValueError, match="no frames"):
        evaluate.average_eval_image_metrics(model, ray_gen(), [])
    assert model.training
