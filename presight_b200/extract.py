"""Prior extraction from camera rays (reference: scripts/extract_priors.py:100-208).

For every training camera the reference casts rays through the valid pixels, finds each ray's threshold depth
(`get_depth_for_camera_ray_bundle`, chunks of 2^17 rays), places the hit at o + d * depth, keeps the hits inside a range
and height window, queries density and semantics there, drops hits with mean density <= 1 and voxelises the rest.
`PriorExtractor` does the same on the device:

    add(rays)   get_surface_hits (fused final level) -> ps_surface_hits -> query_priors -> ps_hits_append: the kept hits'
                scene-unit points and colours (24 B per hit) are appended, in ray order, to fixed-size store blocks,
                and their metric minimum is folded into the voxel lattice's anchor.  The host reads the store cursor
                only when the current block might not hold another chunk.
    finalize()  TileVoxelizer over the stored hits, block by block: the voxel keys first, then query_priors again on
                the stored points (the kernels are deterministic: the same density filter, and one point per kept hit
                against ~256 samples per ray for the depth pass) and the per-voxel sums -> the dict `priors.save_priors`
                writes.  The 64-d features (128 B per hit) are never stored, and nothing grows with the number of hits
                but the store itself.

Pixel selection (image decoding, seg-mask filtering) stays with the caller, who hands rays built by
`cameras.RayGenerator` from (camera, row, col) indices.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Tuple

import torch
from torch import Tensor

from ._lib import call, check, load, ptr, stream
from .cameras.rays import RayBundle
from .priors import TileVoxelizer


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
    means no bound (either end of z_range_m may be None too).  chunk_rays: rays per depth pass (the reference's 2^17).
    block_hits: kept hits per store block (24 B each; the default 2^24 is 384 MB), at least chunk_rays.  insert_slice:
    stored hits per slice of finalize()'s first pass (keys only)."""

    HIT_BYTES = 24                               # scene-unit point and colour, f32 each

    def __init__(self, model, pose_scale_factor: float, voxel_size: float = 0.4, hit_thr_ratio: float = 0.2,
                 max_range_m: Optional[float] = None, z_range_m: Optional[Tuple[Optional[float], Optional[float]]] = None,
                 chunk_rays: int = 1 << 17, block_hits: int = 1 << 24, insert_slice: int = 1 << 24) -> None:
        assert not model.training, "PriorExtractor needs the model in eval mode (call model.eval())"
        assert pose_scale_factor > 0 and chunk_rays > 0 and insert_slice > 0
        assert block_hits >= chunk_rays, "a store block must hold one chunk's hits"
        self.model = model
        self.pose_scale = float(pose_scale_factor)
        self.voxel_size, self.hit_thr_ratio = float(voxel_size), float(hit_thr_ratio)
        self.max_range_m, self.z_range_m = max_range_m, z_range_m
        self.chunk_rays, self.block_hits, self.insert_slice = int(chunk_rays), int(block_hits), int(insert_slice)
        self._blocks: List[Tuple[Tensor, Tensor]] = []   # store blocks: points [block_hits,3] (scene units), colours
        self._sealed: List[int] = []                     # hits in each full block
        self._cursor: Optional[Tensor] = None            # hits in the current (last) block, on the device
        self._cursor_hi = 0                              # host upper bound on the cursor: last read + rays since
        self._min: Optional[Tensor] = None               # running per-axis minimum of the kept hits in metres
        self._status: Optional[Tensor] = None
        self._ws: Optional[Tensor] = None

    def _filled(self) -> List[int]:
        if not self._blocks:
            return []
        return self._sealed + [int(self._cursor.item())]

    @property
    def _points(self) -> List[Tensor]:
        """The stored hits, scene units: one view per store block."""
        return [b[0][:n] for b, n in zip(self._blocks, self._filled())]

    @property
    def n_hits(self) -> int:
        return sum(self._filled())

    def _new_block(self, dev) -> None:
        try:
            blk = (torch.empty(self.block_hits, 3, device=dev), torch.empty(self.block_hits, 3, device=dev))
        except torch.cuda.OutOfMemoryError as e:
            raise RuntimeError(f"PriorExtractor: no device memory for another store block of {self.block_hits} hits "
                               f"after {sum(self._sealed)} hits stored ({self.HIT_BYTES} B per hit)") from e
        self._blocks.append(blk)
        self._cursor.zero_()
        self._cursor_hi = 0

    def _append(self, ps: Tensor, pm: Tensor, keep: Tensor, dens: Tensor, colors: Optional[Tensor]) -> None:
        n = ps.shape[0]
        dev = ps.device
        if self._cursor is None:
            self._cursor = torch.zeros(1, device=dev, dtype=torch.int64)
            self._status = torch.zeros(1, device=dev, dtype=torch.int32)
            self._min = torch.full((3,), float("inf"), device=dev)
            nbytes = C.c_int64()
            check(load().ps_hits_append_workspace(self.chunk_rays, C.byref(nbytes)), "ps_hits_append_workspace")
            self._ws = torch.empty(nbytes.value, device=dev, dtype=torch.uint8)
        if not self._blocks:
            self._new_block(dev)
        elif self._cursor_hi + n > self.block_hits:    # the block might not have room: read the cursor
            self._cursor_hi = int(self._cursor.item())
            if self._cursor_hi + n > self.block_hits:
                self._sealed.append(self._cursor_hi)
                self._new_block(dev)
        pts, cols = self._blocks[-1]
        call("ps_hits_append", ptr(ps), ptr(pm), ptr(keep), ptr(dens), ptr(colors), n, ptr(pts), ptr(cols),
             self.block_hits, ptr(self._cursor), ptr(self._min), ptr(self._status), ptr(self._ws), stream())
        self._cursor_hi += n

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
            dens = dens.detach().to(torch.float32).contiguous().view(-1)
            assert dens.numel() == j - i
            c = None if colors is None else colors[i:j].to(device=ps.device, dtype=torch.float32).contiguous()
            self._append(ps, pm, keep, dens, c)                   # extract_priors.py:157

    @torch.no_grad()
    def finalize(self) -> Dict[str, Tensor]:
        """Voxelise the stored hits -> the result dict of `PriorVoxelizer.finalize` (pass it to `priors.save_priors`)."""
        if self._min is None or self.n_hits == 0:
            raise RuntimeError("PriorExtractor: no surface hit passed the selector and the density filter")
        if int(self._status.item()) & 1:
            raise RuntimeError("PriorExtractor: a chunk's hits did not fit their store block")
        filled = self._filled()
        blocks = [(p[:k], c[:k]) for (p, c), k in zip(self._blocks, filled)]
        vox = TileVoxelizer(self._min, self.voxel_size, self.model.config.semantic_dim,
                            capacity=2 * min(self.insert_slice, sum(filled)))
        # metres exactly as ps_surface_hits computes them: an element-wise IEEE division (torch turns a division by a
        # Python scalar into a multiplication by its reciprocal, which can differ in the last bit)
        scale = torch.full((1, 3), self.pose_scale, device=self._min.device, dtype=torch.float32)
        for pts, _ in blocks:
            for i in range(0, pts.shape[0], self.insert_slice):
                vox.insert(pts[i:i + self.insert_slice] / scale)
        vox.seal()
        for pts, cols in blocks:
            for i in range(0, pts.shape[0], self.chunk_rays):
                p = pts[i:i + self.chunk_rays]
                _, feats = self.model.query_priors(p)
                vox.accumulate(p / scale, feats, cols[i:i + self.chunk_rays])
        return vox.finalize(self.hit_thr_ratio)
