"""numpy fp64 restatement of the image metrics of nerfstudio's nerfacto — TEST INFRASTRUCTURE, NOT PRODUCT.

The reference model scores its evaluation images with torchmetrics (models/nerfacto.py `get_image_metrics_and_images`):
  PeakSignalNoiseRatio(data_range=1.0)     10 log10(data_range^2 / mean((pred - gt)^2)), the mean over all 3HW values
  structural_similarity_index_measure      with its defaults, on one image [1,3,H,W] at a time (torchmetrics 1.x
                                           `_ssim_update`): Gaussian window 11 x 11, sigma 1.5; data range
                                           max(max(pred) - min(pred), max(gt) - min(gt)); k1 = 0.01, k2 = 0.03;
                                           reflect pad 5, 2-D convolution of x, y, x^2, y^2, xy, variances E[x^2] - mu^2
                                           (not clamped), the SSIM map, crop 5 from every side, mean.
torchmetrics is not installed here, so `ssim` writes those steps out literally (pad, convolve, crop) rather than the
valid-window form the product computes; `ssim_valid_windows` is that second form, and the tests check that the two agree.
Images are [H,W,3] (channels-last, as the model renders them).
"""
from __future__ import annotations

import numpy as np

WIN, SIGMA, K1, K2 = 11, 1.5, 0.01, 0.03


def gaussian_window() -> np.ndarray:
    """[11,11]: the outer product of the normalised 1-D Gaussian (torchmetrics `_gaussian_kernel_2d`)."""
    d = np.arange(WIN, dtype=np.float64) - (WIN - 1) / 2
    g = np.exp(-((d / SIGMA) ** 2) / 2)
    g /= g.sum()
    return np.outer(g, g)


def psnr(pred, gt, data_range: float = 1.0) -> float:
    p, g = np.asarray(pred, np.float64), np.asarray(gt, np.float64)
    mse = np.sum((p - g) ** 2) / p.size
    with np.errstate(divide="ignore"):
        return float(10.0 * np.log10(data_range ** 2 / mse))


def _channels_first(a):
    return np.moveaxis(np.asarray(a, np.float64), -1, 0)          # [3,H,W]


def _data_range(x, y):
    return max(x.max() - x.min(), y.max() - y.min())


def _conv2d_valid(img, w):
    """[C,h,w] correlated with the [k,k] window, no padding -> [C,h-k+1,w-k+1]."""
    k = w.shape[0]
    H, W = img.shape[1] - k + 1, img.shape[2] - k + 1
    out = np.zeros((img.shape[0], H, W))
    for i in range(k):
        for j in range(k):
            out += w[i, j] * img[:, i:i + H, j:j + W]
    return out


def _ssim_map(moments, c1, c2):
    mu_x, mu_y, exx, eyy, exy = moments
    sxx, syy, sxy = exx - mu_x ** 2, eyy - mu_y ** 2, exy - mu_x * mu_y
    with np.errstate(divide="ignore", invalid="ignore"):
        return ((2 * mu_x * mu_y + c1) * (2 * sxy + c2)) / ((mu_x ** 2 + mu_y ** 2 + c1) * (sxx + syy + c2))


def ssim(pred, gt) -> float:
    """torchmetrics' SSIM of one [H,W,3] pair, step by step: reflect pad, convolve, SSIM map, crop, mean."""
    x, y = _channels_first(pred), _channels_first(gt)
    if x.shape[1] < WIN or x.shape[2] < WIN:
        raise ValueError("SSIM needs images of at least 11 x 11 pixels")
    dr = _data_range(x, y)
    c1, c2 = (K1 * dr) ** 2, (K2 * dr) ** 2
    p = (WIN - 1) // 2
    stack = np.concatenate([x, y, x * x, y * y, x * y])            # [15,H,W]
    padded = np.pad(stack, ((0, 0), (p, p), (p, p)), mode="reflect")
    conv = _conv2d_valid(padded, gaussian_window()).reshape(5, 3, x.shape[1], x.shape[2])
    full = _ssim_map(conv, c1, c2)
    return float(full[:, p:-p, p:-p].mean())


def ssim_valid_windows(pred, gt) -> float:
    """The same SSIM from the windows that lie wholly inside the image (no padding formed)."""
    x, y = _channels_first(pred), _channels_first(gt)
    dr = _data_range(x, y)
    c1, c2 = (K1 * dr) ** 2, (K2 * dr) ** 2
    stack = np.concatenate([x, y, x * x, y * y, x * y])
    conv = _conv2d_valid(stack, gaussian_window()).reshape(5, 3, x.shape[1] - WIN + 1, x.shape[2] - WIN + 1)
    return float(_ssim_map(conv, c1, c2).mean())
