"""CPU checks of the image metrics: the per-window core (presight_b200/csrc/metrics_core.h, the code the CUDA kernels run)
compiled for the host, against the numpy oracle's literal pad-convolve-crop SSIM and PSNR."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import metrics_oracle as MO

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def host_lib(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("metrics") / "libmetrics_host.so")
    src = os.path.join(HERE, "native", "metrics_host.cpp")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", src, "-o", out], check=True)
    lib = ctypes.CDLL(out)
    lib.image_metrics_host.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                       ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    return lib


def run(lib, pred, gt, data_range=1.0):
    pred, gt = (np.ascontiguousarray(a, dtype=np.float32) for a in (pred, gt))
    sse, psnr, ssim = np.zeros(1), np.zeros(1, np.float32), np.zeros(1)
    rc = lib.image_metrics_host(pred.ctypes.data, gt.ctypes.data, pred.shape[0], pred.shape[1], data_range,
                                sse.ctypes.data, psnr.ctypes.data, ssim.ctypes.data)
    return rc, float(sse[0]), float(psnr[0]), float(ssim[0])


def image_pair(kind, H, W, seed):
    """(pred, gt) float32 [H,W,3] in [0,1]."""
    rng = np.random.default_rng(seed)
    if kind == "random":
        gt = rng.random((H, W, 3))
        pred = np.clip(gt + 0.1 * rng.standard_normal((H, W, 3)), 0, 1)
    elif kind == "smooth":                                   # low-frequency content: small local variances
        yy, xx = np.meshgrid(np.linspace(0, 1, H), np.linspace(0, 1, W), indexing="ij")
        ph = rng.random(3) * 6.28
        gt = 0.5 + 0.4 * np.sin(3 * xx[..., None] + 2 * yy[..., None] + ph)
        pred = np.clip(gt + 0.02 * np.sin(7 * xx[..., None] - 5 * yy[..., None]) + 0.005 * rng.standard_normal(gt.shape),
                       0, 1)
    else:                                                    # "edge": saturated renders, values at 0 and 1
        gt = (rng.random((H, W, 3)) < 0.5).astype(np.float64)
        pred = np.where(rng.random((H, W, 3)) < 0.8, gt, rng.random((H, W, 3)))
        pred[: H // 2, : W // 3] = 1.0
    return pred.astype(np.float32), gt.astype(np.float32)


@pytest.mark.parametrize("kind", ["random", "smooth", "edge"])
@pytest.mark.parametrize("H,W", [(11, 11), (12, 37), (37, 12), (64, 50)])
def test_core_matches_oracle(host_lib, kind, H, W):
    pred, gt = image_pair(kind, H, W, seed=H * 100 + W)
    rc, sse, psnr, ssim = run(host_lib, pred, gt)
    assert rc == 0
    d = (pred - gt).astype(np.float64)                       # the fp32 difference, squared and summed in fp64
    assert sse == pytest.approx(float(np.sum(d * d)), rel=1e-12)
    assert abs(psnr - MO.psnr(pred, gt)) <= 1e-4
    assert abs(ssim - MO.ssim(pred, gt)) <= 1e-5, (ssim, MO.ssim(pred, gt))


@pytest.mark.parametrize("kind", ["random", "smooth"])
def test_core_matches_oracle_full_camera_image(host_lib, kind):
    pred, gt = image_pair(kind, 900, 1600, seed=7)
    rc, _, psnr, ssim = run(host_lib, pred, gt)
    assert rc == 0
    assert abs(psnr - MO.psnr(pred, gt)) <= 1e-4
    assert abs(ssim - MO.ssim(pred, gt)) <= 1e-5


@pytest.mark.parametrize("H,W", [(11, 11), (12, 37), (40, 29)])
def test_padded_form_keeps_only_windows_inside_the_image(H, W):
    """The oracle's literal reflect-pad / convolve / crop equals the valid-window form the kernels compute: the crop removes
    every output whose window reaches into the padding."""
    pred, gt = image_pair("random", H, W, seed=3)
    assert abs(MO.ssim(pred, gt) - MO.ssim_valid_windows(pred, gt)) <= 1e-13


def test_identical_images(host_lib):
    for kind in ("random", "smooth", "edge"):
        _, gt = image_pair(kind, 23, 31, seed=1)
        rc, sse, psnr, ssim = run(host_lib, gt, gt)
        assert rc == 0 and sse == 0.0
        assert psnr == np.inf
        assert ssim == 1.0
    assert MO.psnr(gt, gt) == np.inf


def test_constant_pair_is_nan(host_lib):
    for a, b in ((0.3, 0.7), (0.0, 0.0), (1.0, 0.25)):
        pred, gt = np.full((15, 20, 3), a, np.float32), np.full((15, 20, 3), b, np.float32)
        rc, _, _, ssim = run(host_lib, pred, gt)
        assert rc == 0 and np.isnan(ssim)
    assert np.isnan(MO.ssim(np.zeros((15, 20, 3)), np.zeros((15, 20, 3))))


def test_data_range_is_per_image_and_the_larger_of_the_two(host_lib):
    """Scaling only the prediction's spread changes c1 / c2 through the data range."""
    pred, gt = image_pair("random", 20, 24, seed=5)
    narrow = (0.25 + 0.5 * gt).astype(np.float32)
    _, _, _, s = run(host_lib, narrow, gt)
    assert abs(s - MO.ssim(narrow, gt)) <= 1e-5
    _, _, _, s2 = run(host_lib, gt, narrow)
    assert s == s2                                                     # symmetric, as the definition


def test_psnr_data_range(host_lib):
    pred, gt = image_pair("random", 16, 16, seed=2)
    _, _, p1, _ = run(host_lib, pred, gt, 1.0)
    _, _, p255, _ = run(host_lib, pred, gt, 255.0)
    assert abs(p255 - p1 - 20 * np.log10(255.0)) <= 1e-4
    assert abs(p255 - MO.psnr(pred, gt, 255.0)) <= 1e-4


@pytest.mark.parametrize("H,W", [(10, 11), (11, 10), (5, 40)])
def test_sizes_below_the_window_are_rejected(host_lib, H, W):
    pred, gt = image_pair("random", max(H, 1), max(W, 1), seed=0)
    assert run(host_lib, pred, gt)[0] == 1
    with pytest.raises(ValueError):
        MO.ssim(pred, gt)
