"""torch fp64 restatement of LPIPS as nerfstudio's nerfacto computes it — TEST INFRASTRUCTURE, NOT PRODUCT.

The reference model builds `LearnedPerceptualImagePatchSimilarity(normalize=True)` (torchmetrics
functional/image/lpips.py: AlexNet, LPIPS v0.1, mean reduction) and calls it on one [1,3,H,W] pair at a time:
  x = 2 x - 1; the scaling layer (x - shift) / scale, shift = (-0.030, -0.088, -0.188), scale = (0.458, 0.448, 0.450)
      (fp32 tensors in torchmetrics, used here at those fp32 values);
  AlexNet `features` cut after each ReLU (lpips 0.1 `pretrained_networks.alexnet`: slices [0:2], [2:5], [5:8],
      [8:10], [10:12] of torchvision's `features`);
  per layer: `normalize_tensor` f / (sqrt(sum_c f^2) + 1e-10), squared difference, the 1 x 1 no-bias `lin` convolution,
      mean over the layer's pixels; LPIPS = the sum over the five layers.
Written out with F.conv2d / F.max_pool2d on CPU fp64.  Weights are the state dicts `presight_b200.metrics.LPIPS`
reads: torchvision keys `features.{0,3,6,8,10}.{weight,bias}` and `lin{k}.model.1.weight` [1,C,1,1].
"""
from __future__ import annotations

from typing import List, Mapping, Tuple

import torch
import torch.nn.functional as F

SHIFT = torch.tensor([-0.030, -0.088, -0.188], dtype=torch.float32).double()
SCALE = torch.tensor([0.458, 0.448, 0.450], dtype=torch.float32).double()
# (torchvision features index, stride, padding, max-pool before the conv)
LAYERS = ((0, 4, 2, False), (3, 1, 2, True), (6, 1, 1, True), (8, 1, 1, False), (10, 1, 1, False))


def _nchw(img) -> torch.Tensor:
    t = torch.as_tensor(img).to(torch.float64)
    return t.permute(2, 0, 1)[None] if t.dim() == 3 else t.permute(0, 3, 1, 2)


def scaled_input(img) -> torch.Tensor:
    """[H,W,3] (or [B,H,W,3]) in [0,1] -> the [B,3,H,W] fp64 tensor AlexNet sees."""
    x = 2 * _nchw(img) - 1
    return (x - SHIFT[None, :, None, None]) / SCALE[None, :, None, None]


def features(x: torch.Tensor, alexnet_sd: Mapping[str, torch.Tensor]) -> List[torch.Tensor]:
    """The five relu outputs of AlexNet on the scaled input x [B,3,H,W]."""
    out = []
    for i, stride, pad, pool in LAYERS:
        if pool:
            x = F.max_pool2d(x, kernel_size=3, stride=2)
        w, b = (alexnet_sd[f"features.{i}.{n}"].detach().to(torch.float64) for n in ("weight", "bias"))
        x = F.relu(F.conv2d(x, w, b, stride=stride, padding=pad))
        out.append(x)
    return out


def normalize_tensor(f: torch.Tensor, eps: float = 1e-10) -> torch.Tensor:
    return f / (torch.sqrt(torch.sum(f ** 2, dim=1, keepdim=True)) + eps)


def lpips(x0, x1, alexnet_sd, lin_sd) -> Tuple[float, List[float]]:
    """LPIPS of one [H,W,3] pair in [0,1] -> (total, the five per-layer means)."""
    f0 = features(scaled_input(x0), alexnet_sd)
    f1 = features(scaled_input(x1), alexnet_sd)
    per_layer = []
    for k, (a, b) in enumerate(zip(f0, f1)):
        d = (normalize_tensor(a) - normalize_tensor(b)) ** 2
        lin = lin_sd[f"lin{k}.model.1.weight"].detach().to(torch.float64)
        per_layer.append(float(F.conv2d(d, lin).mean()))
    total = 0.0
    for v in per_layer:
        total += v
    return total, per_layer
