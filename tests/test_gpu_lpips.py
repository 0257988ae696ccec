"""LPIPS on the device: `ps_lpips` against the fp64 oracle (oracle/lpips_oracle.py) within the TF32 bound, its exact
properties (batch = pairs one at a time, repeatability, lpips(x, x) == 0, symmetry), the ABI's argument checks, and the
model's `lpips` hook."""
import ctypes as C

import pytest
import torch

from oracle import lpips_oracle as LO
from test_gpu_extract import c2_model
from test_lpips_host import alexnet_state_dict, lin_state_dict
from test_metrics_host import image_pair

pytestmark = pytest.mark.gpu
DEV = "cuda"

_NET = {}


def weights(seed=0):
    if seed not in _NET:
        _NET[seed] = (alexnet_state_dict(seed), lin_state_dict(seed))
    return _NET[seed]


def net(seed=0):
    from presight_b200.metrics import LPIPS
    return LPIPS.from_state_dicts(*weights(seed), device=DEV)


def on_dev(*arrays):
    return [torch.from_numpy(a).to(DEV) for a in arrays]


def close(got, want):
    return abs(got - want) <= 1e-3 * abs(want) + 1e-6


@pytest.mark.parametrize("kind", ["random", "smooth", "edge"])
@pytest.mark.parametrize("H,W", [(31, 31), (33, 47), (180, 320), (900, 1600)])
def test_lpips_matches_oracle(kind, H, W):
    pred, gt = image_pair(kind, H, W, seed=H + 3 * W)
    total, layers = net()(*on_dev(pred, gt), per_layer=True)
    assert total.dtype == layers.dtype == torch.float64 and total.dim() == 0 and layers.shape == (5,)
    want, want_layers = LO.lpips(pred, gt, *weights())
    got_layers = layers.tolist()
    assert close(float(total), want), (float(total), want)
    for k in range(5):
        assert close(got_layers[k], want_layers[k]), (k, got_layers[k], want_layers[k])


def test_batch_equals_single_pairs_bit_for_bit():
    n = net(1)
    pairs = [image_pair(k, 180, 320, seed=i) for i, k in enumerate(("random", "smooth", "edge"))]
    pred = torch.stack([torch.from_numpy(p) for p, _ in pairs]).to(DEV)
    gt = torch.stack([torch.from_numpy(g) for _, g in pairs]).to(DEV)
    total, layers = n(pred, gt, per_layer=True)
    assert total.shape == (3,) and layers.shape == (3, 5)
    for i in range(3):
        t, ly = n(pred[i], gt[i], per_layer=True)
        assert torch.equal(t, total[i]) and torch.equal(ly, layers[i])


def test_exact_properties():
    n = net(2)
    a, b = on_dev(*image_pair("random", 900, 1600, seed=11))
    x = n(a, b)
    assert torch.equal(x, n(a, b))                                  # repeated calls are bit-identical
    assert float(x) > 0
    assert torch.equal(n(b, a), x)                                  # symmetric bit for bit
    same, layers = n(a, a.clone(), per_layer=True)
    assert float(same) == 0.0 and torch.count_nonzero(layers) == 0


def test_abi_checks():
    from presight_b200 import _lib
    lib = _lib.load()
    n = net()
    nbytes = C.c_int64(0)
    assert lib.ps_lpips_workspace(2, 900, 1600, C.byref(nbytes)) == 0
    per_pair = nbytes.value
    assert lib.ps_lpips_workspace(1, 900, 1600, C.byref(nbytes)) == 0
    assert 100e6 < nbytes.value < 160e6 and per_pair > nbytes.value
    assert lib.ps_lpips_workspace(1, 30, 40, C.byref(nbytes)) == 1
    assert lib.ps_lpips_workspace(1, 40, 40, None) == 1

    a, b = on_dev(*image_pair("random", 40, 40, seed=0))
    assert lib.ps_lpips_workspace(1, 40, 40, C.byref(nbytes)) == 0
    ws = torch.empty(nbytes.value, dtype=torch.uint8, device=DEV)
    out = torch.empty(1, dtype=torch.float64, device=DEV)
    st = n._net()
    good = dict(pred=a.data_ptr(), gt=b.data_ptr(), B=1, H=40, W=40, net=C.byref(st), ws=ws.data_ptr(), out=out.data_ptr())

    def run(**kw):
        args = dict(good, **kw)
        return lib.ps_lpips(args["pred"], args["gt"], args["B"], args["H"], args["W"], args["net"], args["ws"], None,
                            args["out"], _lib.stream())

    assert run() == 0
    torch.cuda.synchronize()
    cases = [(dict(H=30), b"31 x 31"), (dict(W=12), b"31 x 31"), (dict(B=0), b"B must be"),
             (dict(pred=None), b"null"), (dict(gt=None), b"null"), (dict(net=None), b"null"), (dict(ws=None), b"null"),
             (dict(out=None), b"null"), (dict(H=1 << 20, W=1 << 20), b"overflow")]
    for kw, msg in cases:
        assert run(**kw) == 1, kw
        assert msg in lib.ps_last_error(), (kw, lib.ps_last_error())
    broken = n._net()
    broken.lin[3] = None
    assert run(net=C.byref(broken)) == 1 and b"layer 3" in lib.ps_last_error()

    with pytest.raises(ValueError, match="31 x 31"):
        n(a[:30], b[:30])
    with pytest.raises(ValueError):
        n(a, b[:39])


def test_model_hook_on_a_rendered_camera_image():
    from test_gpu_render import ray_generator
    model, _ = c2_model()
    keys = set(model.state_dict().keys())
    out = model.get_outputs_for_camera_ray_bundle(ray_generator().image_rays(1, 900, 1600))
    gt = torch.rand(900, 1600, 3, generator=torch.Generator().manual_seed(5)).to(DEV)
    plain, imgs = model.get_image_metrics_and_images(out, {"rgb": gt})
    assert set(plain) == {"psnr", "ssim"}
    n = net()
    model.lpips = n
    assert set(model.state_dict().keys()) == keys
    m, imgs2 = model.get_image_metrics_and_images(out, {"rgb": gt})
    assert set(m) == {"psnr", "ssim", "lpips"} and all(isinstance(v, float) for v in m.values())
    assert m["psnr"] == plain["psnr"] and m["ssim"] == plain["ssim"]
    assert m["lpips"] == float(n(out["rgb"], gt)) and m["lpips"] > 0
    assert torch.equal(imgs2["img"], imgs["img"])
    model.lpips = None
    assert set(model.get_image_metrics_and_images(out, {"rgb": gt})[0]) == {"psnr", "ssim"}
