"""Prior extraction from camera rays (reference: scripts/extract_priors.py:100-208).

For every training camera the reference casts rays through the valid pixels, finds each ray's threshold depth
(`get_depth_for_camera_ray_bundle`, chunks of 2^17 rays), places the hit at o + d * depth, keeps the hits inside a range
and height window, queries density and semantics there, drops hits with mean density <= 1 and voxelises the rest.
`PriorExtractor` does the same on the device:

    add(rays)   get_surface_hits (fused final level) -> ps_surface_hits -> query_priors -> density filter; only the
                kept hits' scene-unit points and colours (24 B per hit) are stored, and their metric minimum is folded
                into the voxel lattice's anchor
    finalize()  query_priors again on the stored points (the kernels are deterministic: the same density filter, and
                one point per kept hit against ~256 samples per ray for the depth pass) -> PriorVoxelizer -> the dict
                `priors.save_priors` writes.  The 64-d features (128 B per hit) are never stored.

Pixel selection (image decoding, seg-mask filtering) stays with the caller, who hands rays built by
`cameras.RayGenerator` from (camera, row, col) indices.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import torch
from torch import Tensor

from ._lib import call, ptr, stream
from .cameras.rays import RayBundle
from .priors import PriorVoxelizer


def _bound(v: Optional[float]) -> float:
    return float("nan") if v is None else float(v)


@torch.no_grad()
def surface_hits(origins: Tensor, directions: Tensor, depth: Tensor, pose_scale_factor: float,
                 max_range_m: Optional[float] = None, z_range_m: Optional[Tuple[Optional[float], Optional[float]]] = None):
    """ps_surface_hits -> (points_scaled [N,3] f32 = o + d * depth, points_m [N,3] f32 = points_scaled / pose_scale_factor,
    keep [N] bool = range <= max_range_m and z_min <= z <= z_max in metres).  A bound given as None is not applied."""
    o = origins.detach().to(torch.float32).contiguous()
    d = directions.detach().to(torch.float32).contiguous()
    t = depth.detach().to(torch.float32).contiguous().view(-1)
    N = o.shape[0]
    assert d.shape == (N, 3) and t.numel() == N, "origins / directions [N,3], depth [N] or [N,1]"
    z_lo, z_hi = z_range_m if z_range_m is not None else (None, None)
    ps = torch.empty(N, 3, device=o.device, dtype=torch.float32)
    pm = torch.empty(N, 3, device=o.device, dtype=torch.float32)
    keep = torch.empty(N, device=o.device, dtype=torch.uint8)
    call("ps_surface_hits", ptr(o), ptr(d), ptr(t), N, float(pose_scale_factor), _bound(max_range_m), _bound(z_lo),
         _bound(z_hi), ptr(ps), ptr(pm), ptr(keep), stream())
    return ps, pm, keep.bool()


class PriorExtractor:
    """Streams camera rays into `extracted_priors.pkl` content for one tile.

    model: NerfactoNuscMSModel in eval mode.  pose_scale_factor: scene units per metre.  voxel_size (m) and hit_thr_ratio
    as in `priors.postprocess_priors`.  max_range_m / z_range_m = (z_min, z_max): the reference's range and height
    selector (extract_priors.py:114-126); its constants are not part of this project, so there are no defaults — None
    means no bound (either end of z_range_m may be None too).  chunk_rays: rays per depth pass (the reference's 2^17)."""

    def __init__(self, model, pose_scale_factor: float, voxel_size: float = 0.4, hit_thr_ratio: float = 0.2,
                 max_range_m: Optional[float] = None, z_range_m: Optional[Tuple[Optional[float], Optional[float]]] = None,
                 chunk_rays: int = 1 << 17) -> None:
        assert not model.training, "PriorExtractor needs the model in eval mode (call model.eval())"
        assert pose_scale_factor > 0 and chunk_rays > 0
        self.model = model
        self.pose_scale = float(pose_scale_factor)
        self.voxel_size, self.hit_thr_ratio = float(voxel_size), float(hit_thr_ratio)
        self.max_range_m, self.z_range_m = max_range_m, z_range_m
        self.chunk_rays = int(chunk_rays)
        self._points: List[Tensor] = []          # kept hits, scene units [k,3] f32
        self._colors: List[Tensor] = []          # their colours [k,3] f32
        self._min: Optional[Tensor] = None       # running per-axis minimum of the kept hits in metres

    @property
    def n_hits(self) -> int:
        return sum(p.shape[0] for p in self._points)

    @torch.no_grad()
    def add(self, ray_bundle: RayBundle, colors: Optional[Tensor] = None) -> None:
        """Surface hits of `ray_bundle` (any number of rays, evaluated `chunk_rays` at a time) that pass the range / height
        selector and the mean-density filter.  colors: per-ray [N,3] values averaged into the voxels (zeros if None)."""
        n = len(ray_bundle)
        if colors is not None:
            assert colors.shape == (n, 3), "colors: one RGB triple per ray"
        for i in range(0, n, self.chunk_rays):
            j = min(i + self.chunk_rays, n)
            o, d = ray_bundle.origins[i:j], ray_bundle.directions[i:j]
            rb = RayBundle(origins=o, directions=d, camera_indices=None if ray_bundle.camera_indices is None
                           else ray_bundle.camera_indices[i:j])
            depth = self.model.get_surface_hits(rb)["depth"]
            ps, pm, keep = surface_hits(o, d, depth, self.pose_scale, self.max_range_m, self.z_range_m)
            dens, _ = self.model.query_priors(ps)
            idx = torch.nonzero(keep & (dens > 1)).view(-1)          # extract_priors.py:157
            self._points.append(ps[idx])
            c = torch.zeros(idx.numel(), 3, device=ps.device) if colors is None else colors[i:j].to(ps.device)[idx]
            self._colors.append(c.to(torch.float32).contiguous())
            self._min = PriorVoxelizer.min_bound(pm[idx], None, self._min)

    @torch.no_grad()
    def finalize(self) -> Dict[str, Tensor]:
        """Voxelise the stored hits -> the result dict of `PriorVoxelizer.finalize` (pass it to `priors.save_priors`)."""
        if self._min is None or self.n_hits == 0:
            raise RuntimeError("PriorExtractor: no surface hit passed the selector and the density filter")
        pts = torch.cat(self._points)
        cols = torch.cat(self._colors)
        n = pts.shape[0]
        vox = PriorVoxelizer(self._min, self.voxel_size, self.model.config.semantic_dim, capacity=2 * max(n, 1024))
        # metres exactly as ps_surface_hits computes them: an element-wise IEEE division (torch turns a division by a
        # Python scalar into a multiplication by its reciprocal, which can differ in the last bit)
        scale = torch.full((1, 3), self.pose_scale, device=pts.device, dtype=torch.float32)
        for i in range(0, n, self.chunk_rays):
            p = pts[i:i + self.chunk_rays]
            _, feats = self.model.query_priors(p)
            vox.add(p / scale, feats, cols[i:i + self.chunk_rays])
        return vox.finalize(self.hit_thr_ratio)
