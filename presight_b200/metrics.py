"""Image metrics of rendered images on `ps_image_metrics` (reference: the torchmetrics calls of nerfstudio's
models/nerfacto.py `get_metrics_dict` / `get_image_metrics_and_images`, which PreSight's model inherits).

    psnr(pred, gt)           PeakSignalNoiseRatio(data_range=1.0): 10 log10(1 / mean((pred - gt)^2)), fp64 sum
    ssim(pred, gt)           structural_similarity_index_measure with its defaults, one image at a time
    image_metrics(pred, gt)  both for a batch of images in one call
    LPIPS                    LearnedPerceptualImagePatchSimilarity(normalize=True) (AlexNet, LPIPS v0.1) on `ps_lpips`
    colormap_images          the colormapped accumulation and depth images of nerfacto (utils/colormaps.py) on
                             `ps_colormap`

Images are [H,W,3] or [B,H,W,3] fp32 channels-last, as `get_outputs_for_camera_ray_bundle` returns them.  Every result
stays on the device (no host read), and repeated calls give bit-identical results.  The exact definitions, and the
NaN SSIM of two constant images, are in csrc/metrics_core.h.  LPIPS needs pretrained weights, which this project does
not ship: the caller brings torchvision's AlexNet state dict and the LPIPS v0.1 linear layers, or a reference checkpoint
that holds them (see `LPIPS`).  Likewise the colormaps need the caller's [256,3] table (e.g. matplotlib's turbo).
"""
from __future__ import annotations

import ctypes as C
import re
from typing import Dict, List, Mapping, Sequence, Tuple

import torch
from torch import Tensor

from ._lib import LpipsNet, call, ptr, stream


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


@torch.no_grad()
def colormap_images(depth_maps: Sequence[Tensor], accumulation: Tensor, lut: Tensor) -> Tuple[Tensor, List[Tensor]]:
    """nerfacto's evaluation images in one `ps_colormap` call: depth_maps [H,W,1] each (depth, prop_depth_0, ...),
    accumulation [H,W,1], lut [256,3] -> (apply_colormap(accumulation), [apply_depth_colormap(d, accumulation) for d]),
    each [H,W,3] fp32, bit-identical to nerfstudio's utils/colormaps.py run by torch on the device with default
    ColormapOptions and this table as the colormap.  No host read: the per-map min / max stay on the device."""
    if accumulation.dim() != 3 or accumulation.shape[-1] != 1:
        raise ValueError(f"accumulation must be [H,W,1], got {tuple(accumulation.shape)}")
    for d in depth_maps:
        if d.shape != accumulation.shape:
            raise ValueError(f"depth map {tuple(d.shape)} and accumulation {tuple(accumulation.shape)} differ in shape")
    if tuple(lut.shape) != (256, 3):
        raise ValueError(f"lut must be [256,3], got {tuple(lut.shape)}")
    H, W, _ = accumulation.shape
    dev, M = accumulation.device, len(depth_maps)
    acc = accumulation.detach().to(torch.float32).contiguous()
    table = lut.detach().to(device=dev, dtype=torch.float32).contiguous()
    maps = torch.stack([d.detach().reshape(H * W) for d in depth_maps]).to(torch.float32) if M else None
    nbytes = C.c_int64(0)
    call("ps_colormap_workspace", M, H * W, C.byref(nbytes))
    ws = torch.empty(int(nbytes.value), dtype=torch.uint8, device=dev) if M else None
    out = torch.empty(M + 1, H, W, 3, dtype=torch.float32, device=dev)
    call("ps_colormap", ptr(maps), M, H * W, ptr(acc), ptr(table), ptr(ws), ptr(out), stream())
    return out[0], list(out[1:])


# ---- LPIPS ----------------------------------------------------------------------------------------------------------
LPIPS_CHANNELS = (64, 192, 384, 256, 256)
_LPIPS_CIN = (3, 64, 192, 384, 256)
_LPIPS_CONV = ((11, 4, 2), (5, 1, 2), (3, 1, 1), (3, 1, 1), (3, 1, 1))   # kernel, stride, padding
_ALEXNET_INDEX = (0, 3, 6, 8, 10)                                          # torchvision `features.{i}`
_LPIPS_GROUP_BYTES = 1 << 30                 # workspace bound of one ps_lpips call (about 7 pairs at 1600 x 900)


def lpips_layer_shapes(H: int, W: int) -> List[Tuple[int, int]]:
    """(h, w) of the five AlexNet feature maps LPIPS compares for an H x W image; ValueError below 31 x 31, where the
    second max-pool leaves nothing."""
    if H < 31 or W < 31:
        raise ValueError(f"LPIPS needs images of at least 31 x 31 pixels, got {H} x {W}")

    def conv(n, k, s, p):
        return (n + 2 * p - k) // s + 1

    def pool(n):
        return (n - 3) // 2 + 1

    h1, w1 = conv(H, 11, 4, 2), conv(W, 11, 4, 2)
    h2, w2 = pool(h1), pool(w1)
    h3, w3 = pool(h2), pool(w2)
    return [(h1, w1), (h2, w2), (h3, w3), (h3, w3), (h3, w3)]


def lpips_flops(H: int, W: int) -> int:
    """Multiply-adds x 2 of the five convolutions for one H x W image (a pair costs twice this)."""
    return sum(2 * h * w * c * cin * k * k
               for (h, w), c, cin, (k, _, _) in zip(lpips_layer_shapes(H, W), LPIPS_CHANNELS, _LPIPS_CIN, _LPIPS_CONV))


def tf32_round(x: Tensor) -> Tensor:
    """fp32 -> the nearest TF32 value (ties away from zero), as cvt.rna.tf32.f32 rounds finite values."""
    bits = x.detach().to(torch.float32).contiguous().view(torch.int32)
    return ((bits + 0x1000) & -0x2000).view(torch.float32)


def _expected_keys() -> Dict[str, Tuple[int, ...]]:
    exp = {}
    for i, c, cin, (k, _, _) in zip(_ALEXNET_INDEX, LPIPS_CHANNELS, _LPIPS_CIN, _LPIPS_CONV):
        exp[f"features.{i}.weight"] = (c, cin, k, k)
        exp[f"features.{i}.bias"] = (c,)
    for j, c in enumerate(LPIPS_CHANNELS):
        exp[f"lin{j}.model.1.weight"] = (1, c, 1, 1)
    return exp


# where a reference checkpoint keeps the weights: torchmetrics' `_LPIPS` under the model's `lpips.net.`, its AlexNet
# slices holding torchvision's `features.{i}` layers
_REFERENCE_SLICES = {0: "net.slice1.0", 3: "net.slice2.3", 6: "net.slice3.6", 8: "net.slice4.8", 10: "net.slice5.10"}
_REFERENCE_KEY = re.compile(r"^((?:[^.]*\.)*?)lpips\.net\.(.+)$")
# the scaling layer `ps_lpips` applies (csrc/lpips.cu c_shift / c_scale)
_SCALING_LAYER = {"scaling_layer.shift": (-0.030, -0.088, -0.188), "scaling_layer.scale": (0.458, 0.448, 0.450)}


def _reference_names() -> Dict[str, str]:
    """key after `lpips.net.` -> the key `from_state_dicts` reads"""
    names = {}
    for i, s in _REFERENCE_SLICES.items():
        names[f"{s}.weight"], names[f"{s}.bias"] = f"features.{i}.weight", f"features.{i}.bias"
    names.update({f"lin{j}.model.1.weight": f"lin{j}.model.1.weight" for j in range(len(LPIPS_CHANNELS))})
    return names


def _check_keys(got: Mapping[str, Tensor], exp: Mapping[str, Tuple[int, ...]], extra: Sequence[str] = ()) -> None:
    bad = list(extra) + [f"missing {k}" for k in exp if k not in got]
    bad += [f"{k} has shape {tuple(got[k].shape)}, expected {exp[k]}" for k in exp
            if k in got and tuple(got[k].shape) != exp[k]]
    if bad:
        want = ", ".join(f"{k} {list(v)}" for k, v in exp.items())
        raise ValueError(f"LPIPS weights: {'; '.join(bad)}.  Expected keys and shapes: {want}")


class LPIPS:
    """LPIPS as nerfacto computes it: torchmetrics `LearnedPerceptualImagePatchSimilarity(net_type="alex",
    normalize=True)`, LPIPS v0.1, mean over the batch's pairs in the reference (here one value per pair).  Definition in
    include/presight_b200.h (`ps_lpips`); the convolutions run in TF32, as cuDNN runs torchmetrics' under PyTorch's
    default `allow_tf32`.

    A plain class, not an nn.Module: attached to a model it adds nothing to the model's state_dict.  The weights are the
    caller's: `LPIPS.from_state_dicts(torchvision_alexnet.state_dict(), lpips_alex_lin_state_dict)`.

        net = LPIPS.from_state_dicts(alexnet_sd, lin_sd)
        value = net(pred, gt)                    # [H,W,3] -> device f64 scalar, [B,H,W,3] -> [B]
    """

    def __init__(self, conv_w: List[Tensor], conv_b: List[Tensor], lin: List[Tensor]):
        """Packed tensors (see `from_state_dicts`): conv_w[k] [C_out][K_pad] TF32-rounded in (ky, kx, ci) order,
        conv_b[k] [C_out], lin[k] [C_k], all fp32 on one device."""
        self.conv_w, self.conv_b, self.lin = list(conv_w), list(conv_b), list(lin)
        self.device = self.conv_w[0].device

    @classmethod
    def from_state_dicts(cls, alexnet_sd: Mapping[str, Tensor], lin_sd: Mapping[str, Tensor],
                         device="cuda") -> "LPIPS":
        """alexnet_sd: torchvision's AlexNet keys `features.{0,3,6,8,10}.{weight,bias}` (what
        `torchvision.models.alexnet(...).state_dict()` and the `alexnet-owt-*.pth` file hold; `classifier.*` is
        ignored).  lin_sd: the LPIPS v0.1 `alex.pth` keys `lin{k}.model.1.weight`, each [1,C_k,1,1].  A missing key or a
        wrong shape raises a ValueError naming every expected key and shape.  Packing runs on CPU tensors as well."""
        got = {**{k: v for k, v in alexnet_sd.items() if k.startswith("features.")},
               **{k: v for k, v in lin_sd.items()}}
        _check_keys(got, _expected_keys())
        conv_w, conv_b, lin = [], [], []
        for i, c in zip(_ALEXNET_INDEX, LPIPS_CHANNELS):
            w = got[f"features.{i}.weight"].detach().to(torch.float32)
            k = w.shape[1] * w.shape[2] * w.shape[3]
            w = w.permute(0, 2, 3, 1).reshape(c, k)                       # (ky, kx, ci), the kernel's K order
            w = torch.nn.functional.pad(w, (0, -k % 32))
            conv_w.append(tf32_round(w).to(device).contiguous())
            conv_b.append(got[f"features.{i}.bias"].detach().to(torch.float32).to(device).contiguous())
        for j, c in enumerate(LPIPS_CHANNELS):
            lin.append(got[f"lin{j}.model.1.weight"].detach().to(torch.float32).reshape(c).to(device).contiguous())
        return cls(conv_w, conv_b, lin)

    @classmethod
    def from_reference_state_dict(cls, sd: Mapping[str, Tensor], device="cuda") -> "LPIPS":
        """The weights a reference checkpoint already holds: a model or pipeline state dict (the keys under any one
        prefix, e.g. `_model.` or `_model.module.`) whose `lpips.net.*` entries are torchmetrics' `_LPIPS`:
        `net.slice{1..5}.{0,3,6,8,10}.{weight,bias}` (torchvision's `features.{0,3,6,8,10}`) and
        `lin{k}.model.1.weight`.  A missing key, a wrong shape or keys under two different prefixes raise a ValueError
        naming every expected key and shape; so does a `scaling_layer.shift` / `scale`, when present, that differs from
        the constants `ps_lpips` applies."""
        found = {}
        for k, v in sd.items():
            m = _REFERENCE_KEY.match(k)
            if m:
                found.setdefault(m.group(1), {})[m.group(2)] = v
        names = _reference_names()
        shapes = _expected_keys()
        prefix = next(iter(found), "")
        exp = {f"{prefix}lpips.net.{k}": shapes[v] for k, v in names.items()}
        extra = []
        if len(found) > 1:
            extra.append("keys under more than one prefix: " + ", ".join(repr(p + "lpips.net.") for p in found))
        sub = found.get(prefix, {})
        _check_keys({f"{prefix}lpips.net.{k}": v for k, v in sub.items()}, exp, extra)
        for k, want in _SCALING_LAYER.items():
            if k in sub:
                v = sub[k].detach().to(device="cpu", dtype=torch.float32).reshape(-1)
                if not torch.equal(v, torch.tensor(want, dtype=torch.float32)):
                    raise ValueError(f"LPIPS weights: {prefix}lpips.net.{k} is {v.tolist()}, but ps_lpips applies "
                                     f"{list(want)}")
        got = {theirs: sub[k] for k, theirs in names.items()}
        return cls.from_state_dicts({k: v for k, v in got.items() if k.startswith("features.")},
                                    {k: v for k, v in got.items() if k.startswith("lin")}, device=device)

    def unpack(self) -> Tuple[Dict[str, Tensor], Dict[str, Tensor]]:
        """The packed weights back in the layouts `from_state_dicts` reads (convolution weights TF32-rounded)."""
        alex, lin = {}, {}
        for i, w, b, c, cin, (k, _, _) in zip(_ALEXNET_INDEX, self.conv_w, self.conv_b, LPIPS_CHANNELS, _LPIPS_CIN,
                                              _LPIPS_CONV):
            alex[f"features.{i}.weight"] = w[:, :k * k * cin].reshape(c, k, k, cin).permute(0, 3, 1, 2).contiguous()
            alex[f"features.{i}.bias"] = b.clone()
        for j, (v, c) in enumerate(zip(self.lin, LPIPS_CHANNELS)):
            lin[f"lin{j}.model.1.weight"] = v.reshape(1, c, 1, 1).clone()
        return alex, lin

    def _net(self) -> LpipsNet:
        net = LpipsNet()
        for k in range(5):
            net.conv_w[k], net.conv_b[k], net.lin[k] = ptr(self.conv_w[k]), ptr(self.conv_b[k]), ptr(self.lin[k])
        return net

    @torch.no_grad()
    def __call__(self, pred: Tensor, gt: Tensor, per_layer: bool = False):
        """pred, gt [H,W,3] or [B,H,W,3] fp32 in [0,1], H, W >= 31 -> LPIPS as a device f64 scalar (or [B]), plus the
        five per-layer means [5] (or [B,5]) when `per_layer`.  No host read.  Values outside [0,1] are not checked
        (that would need one); torchmetrics rejects them.  Large batches run in groups of bounded workspace; every pair
        is computed alone, so the grouping does not change any value."""
        p, g = _images(pred, gt)
        if p.device != self.device:
            raise ValueError(f"images on {p.device}, LPIPS weights on {self.device}")
        B, H, W, _ = p.shape
        lpips_layer_shapes(H, W)
        out = torch.empty(B, dtype=torch.float64, device=p.device)
        layers = torch.empty(B, 5, dtype=torch.float64, device=p.device)
        net = self._net()
        nbytes = C.c_int64(0)
        call("ps_lpips_workspace", 1, H, W, C.byref(nbytes))
        group = max(1, min(B, _LPIPS_GROUP_BYTES // int(nbytes.value)))
        call("ps_lpips_workspace", group, H, W, C.byref(nbytes))
        ws = torch.empty(int(nbytes.value), dtype=torch.uint8, device=p.device)
        for i in range(0, B, group):
            n = min(group, B - i)
            call("ps_lpips", ptr(p[i:i + n]), ptr(g[i:i + n]), n, H, W, C.byref(net), ptr(ws), ptr(layers[i:i + n]),
                 ptr(out[i:i + n]), stream())
        if pred.dim() == 3:
            out, layers = out[0], layers[0]
        return (out, layers) if per_layer else out
