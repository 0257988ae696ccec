"""Image metrics of rendered images on `ps_image_metrics` (reference: the torchmetrics calls of nerfstudio's
models/nerfacto.py `get_metrics_dict` / `get_image_metrics_and_images`, which PreSight's model inherits).

    psnr(pred, gt)           PeakSignalNoiseRatio(data_range=1.0): 10 log10(1 / mean((pred - gt)^2)), fp64 sum
    ssim(pred, gt)           structural_similarity_index_measure with its defaults, one image at a time
    image_metrics(pred, gt)  both for a batch of images in one call

Images are [H,W,3] or [B,H,W,3] fp32 channels-last, as `get_outputs_for_camera_ray_bundle` returns them.  Every result
stays on the device (no host read), and repeated calls give bit-identical results.  The exact definitions, and the
NaN SSIM of two constant images, are in csrc/metrics_core.h.  LPIPS, the reference's third evaluation metric, needs
pretrained AlexNet weights and is not provided.
"""
from __future__ import annotations

import ctypes as C
from typing import Tuple

import torch
from torch import Tensor

from ._lib import call, ptr, stream


def _images(pred: Tensor, gt: Tensor) -> Tuple[Tensor, Tensor]:
    if pred.shape != gt.shape:
        raise ValueError(f"pred {tuple(pred.shape)} and gt {tuple(gt.shape)} differ in shape")
    if pred.dim() not in (3, 4) or pred.shape[-1] != 3:
        raise ValueError(f"images must be [H,W,3] or [B,H,W,3], got {tuple(pred.shape)}")
    p, g = (t.detach().to(torch.float32).contiguous() for t in (pred, gt))
    return (p[None], g[None]) if p.dim() == 3 else (p, g)


def _run(pred: Tensor, gt: Tensor, B: int, H: int, W: int, data_range: float, with_ssim: bool):
    nbytes = C.c_int64(0)
    call("ps_image_metrics_workspace", B, H, W, C.byref(nbytes))
    ws = torch.empty(max(int(nbytes.value), 1), dtype=torch.uint8, device=pred.device)
    sse = torch.empty(B, dtype=torch.float64, device=pred.device)
    psnr = torch.empty(B, dtype=torch.float32, device=pred.device)
    ssim = torch.empty(B, dtype=torch.float64, device=pred.device) if with_ssim else None
    call("ps_image_metrics", ptr(pred), ptr(gt), B, H, W, float(data_range), ptr(ws), ptr(sse), ptr(psnr), ptr(ssim),
         stream())
    return sse, psnr, ssim


@torch.no_grad()
def image_metrics(pred: Tensor, gt: Tensor, data_range: float = 1.0) -> Tuple[Tensor, Tensor, Tensor]:
    """[B,H,W,3] (or [H,W,3]) pairs, H, W >= 11 -> (psnr [B] f32, ssim [B] f64, sse [B] f64), each image with its own
    SSIM data range; `data_range` is PSNR's."""
    p, g = _images(pred, gt)
    B, H, W, _ = p.shape
    sse, psnr, ssim = _run(p, g, B, H, W, data_range, True)
    return psnr, ssim, sse


@torch.no_grad()
def psnr(pred: Tensor, gt: Tensor, data_range: float = 1.0) -> Tensor:
    """PSNR over all values of `pred` / `gt` (any shape [..., 3], e.g. a ray batch [N,3]) -> device scalar f32."""
    if pred.shape != gt.shape or pred.shape[-1:] != (3,):
        raise ValueError(f"pred {tuple(pred.shape)} and gt {tuple(gt.shape)} must be one shape [..., 3]")
    p, g = (t.detach().to(torch.float32).contiguous() for t in (pred, gt))
    n = p.numel() // 3
    if n == 0:
        raise ValueError("psnr of an empty batch")
    if n > 2 ** 31 - 1:
        raise ValueError(f"psnr: {n} pixels exceed one call's 2^31 - 1")
    return _run(p, g, 1, 1, n, data_range, False)[1][0]


@torch.no_grad()
def ssim(pred: Tensor, gt: Tensor) -> Tensor:
    """SSIM of one [H,W,3] pair (a device scalar f64) or of each pair of [B,H,W,3] ([B] f64)."""
    out = image_metrics(pred, gt)[1]
    return out[0] if pred.dim() == 3 else out
