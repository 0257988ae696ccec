"""Prior post-processing and wire format (reference: nerfstudio/scripts/extract_priors.py:156-208, 216-245; reader:
online-mapping/plugin/datasets/prior_utils/city_prior.py:59-73).

The reference concatenates every hit point of a tile on the HOST (~300 GB of RAM, docs/building_priors.md:65), filters
by density, voxel-down-samples with open3d and traces features per voxel in a Python loop.  Here the hit points stay in
HBM and go through a GPU hash-voxelizer (csrc/voxelize.cu): per-voxel centre of mass, colour mean, fp64 feature mean
rounded to fp16, hit count, then the hit-quantile filter — and the result is written as the same pickled dict
`{points f32, features f16, colors f32, hits, origin f32}` the occupancy / online-mapping plugins read.

`PriorVoxelizer` is the streaming form (one `add()` per camera / chunk once the bound is known); `postprocess_priors`
is the one-shot form over resident arrays.  Both size their table by the number of points.  `TileVoxelizer` gives the
same result in two passes with a table sized by the number of voxels, for a whole tile's hits (`extract.PriorExtractor`;
`finalize_rows` gives its rows before the filter, which `extract.ShardedPriorExtractor` applies across GPUs).
CUDA tensors only — no CPU fallback (the CPU restatement is oracle/).
"""
from __future__ import annotations

import pickle
from typing import Dict, Optional

import numpy as np
import torch
from torch import Tensor

from ._lib import call, ptr, stream


def _next_pow2(n: int) -> int:
    return 1 << max(1, (int(n) - 1).bit_length())


class PriorVoxelizer:
    """Accumulates hit points into voxels of `voxel_size` metres.  The voxel lattice is anchored, as open3d anchors it, at
    (min over all density-filtered points) - 1 - voxel_size / 2, so the bound must be known before the first `add`:
    pass `min_point` (e.g. from a first pass with `min_bound`) or use `postprocess_priors` on resident arrays."""

    def __init__(self, min_point: Tensor, voxel_size: float = 0.4, feature_dim: int = 64, capacity: int = 1 << 22,
                 with_colors: bool = True) -> None:
        assert min_point.is_cuda and min_point.numel() == 3, "min_point: 3 floats on the GPU"
        dev = min_point.device
        self.dev, self.voxel_size, self.C = dev, float(voxel_size), int(feature_dim)
        self.min_point = min_point.detach().to(torch.float32).contiguous()
        self.capacity = _next_pow2(capacity)
        self.keys = torch.full((self.capacity,), -1, device=dev, dtype=torch.int64)
        self.counts = torch.zeros(self.capacity, device=dev, dtype=torch.int32)        # u32 on the device
        self.sum_xyz = torch.zeros(self.capacity, 3, device=dev, dtype=torch.float64)
        self.sum_col = torch.zeros(self.capacity, 3, device=dev, dtype=torch.float64) if with_colors else None
        self.sum_feat = torch.zeros(self.capacity, self.C, device=dev, dtype=torch.float64) if self.C else None
        self.status = torch.zeros(1, device=dev, dtype=torch.int32)

    @staticmethod
    def min_bound(points: Tensor, densities: Optional[Tensor] = None, running: Optional[Tensor] = None) -> Tensor:
        """Per-axis min over the points with density > 1 (extract_priors.py:157, 236), folded into `running` if given."""
        out = running if running is not None else torch.full((3,), float("inf"), device=points.device)
        p = points.detach().to(torch.float32).contiguous()
        d = None if densities is None else densities.detach().to(torch.float32).contiguous()
        call("ps_voxel_min_bound", ptr(p), ptr(d), p.shape[0], ptr(out), stream())
        return out

    def add(self, points: Tensor, features: Optional[Tensor], colors: Optional[Tensor],
            densities: Optional[Tensor] = None) -> None:
        """points [n,3] f32 metres, features [n,C] f16, colors [n,3] f32, densities [n] (None = keep all)."""
        p = points.detach().to(torch.float32).contiguous()
        f = None if self.sum_feat is None else features.detach().to(torch.float16).contiguous()
        c = None if self.sum_col is None else colors.detach().to(torch.float32).contiguous()
        d = None if densities is None else densities.detach().to(torch.float32).contiguous()
        assert f is None or f.shape == (p.shape[0], self.C)
        call("ps_voxel_accumulate", ptr(p), ptr(f), ptr(c), ptr(d), p.shape[0], self.C, ptr(self.min_point),
             self.voxel_size, ptr(self.keys), self.capacity, ptr(self.counts), ptr(self.sum_xyz), ptr(self.sum_col),
             ptr(self.sum_feat), ptr(self.status), stream())

    def finalize(self, hit_thr_ratio: float = 0.2) -> Dict[str, Tensor]:
        """-> {"points" [M,3] f32, "features" [M,C] f16, "colors" [M,3] f32, "hits" [M] i64, "hit_thr" f64 scalar,
        "n_voxels" int} on the device, voxels in ascending (ix, iy, iz) order, after the `hits > quantile` filter
        (extract_priors.py:188-196)."""
        st = int(self.status.item())
        if st & 1:
            raise RuntimeError(f"PriorVoxelizer: hash table of {self.capacity} slots is full — construct it with a larger capacity")
        if st & 2:
            raise RuntimeError("PriorVoxelizer: a voxel index exceeds 21 bits per axis (tile larger than 2^21 voxels across)")
        dev = self.dev
        n_out = torch.zeros(1, device=dev, dtype=torch.int64)
        cap = self.capacity
        okeys = torch.empty(cap, device=dev, dtype=torch.int64)
        oxyz = torch.empty(cap, 3, device=dev, dtype=torch.float32)
        ocol = torch.empty(cap, 3, device=dev, dtype=torch.float32) if self.sum_col is not None else None
        ofeat = torch.empty(cap, self.C, device=dev, dtype=torch.float16) if self.sum_feat is not None else None
        ohits = torch.empty(cap, device=dev, dtype=torch.int64)
        call("ps_voxel_finalize", ptr(self.keys), cap, ptr(self.counts), ptr(self.sum_xyz), ptr(self.sum_col),
             ptr(self.sum_feat), self.C, ptr(n_out), ptr(okeys), ptr(oxyz), ptr(ocol), ptr(ofeat), ptr(ohits), stream())
        m = int(n_out.item())
        if m == 0:
            raise RuntimeError("PriorVoxelizer: no points passed the density filter")
        order = torch.argsort(okeys[:m])                    # canonical voxel order (open3d's is a hash map's; see oracle/)
        hits = ohits[:m][order]
        bins = int(hits.max().item()) + 1
        hist = torch.zeros(bins, device=dev, dtype=torch.int32)
        thr = torch.zeros(1, device=dev, dtype=torch.float64)
        status = torch.zeros(1, device=dev, dtype=torch.int32)
        call("ps_hits_quantile", ptr(hits), m, float(hit_thr_ratio), ptr(hist), bins, ptr(thr), ptr(status), stream())
        keep = hits.to(torch.float64) > thr                 # extract_priors.py:191
        sel = order[keep]
        return {"points": oxyz[:m][sel], "features": None if ofeat is None else ofeat[:m][sel],
                "colors": None if ocol is None else ocol[:m][sel], "hits": hits[keep], "hit_thr": thr[0], "n_voxels": m}


_TABLE_STATUS = {1: "the voxel key table is full", 2: "a voxel index exceeds 21 bits per axis (tile larger than 2^21 "
                 "voxels across)", 4: "a point reached pass 2 whose voxel was not inserted in pass 1"}


class TileVoxelizer:
    """`PriorVoxelizer`'s result for a whole tile in memory that follows the number of voxels V, not of points.

    Two passes over the same points (metres, f32), the lattice anchored at `min_point` as in `PriorVoxelizer`:
        insert(points)                       pass 1, keys only (12 B per table slot, load factor <= 1/2): before each slice
                                             of P points the table grows to >= 2 (V + P) slots (one host read per slice)
        seal()                               sorts the V keys; row r of the accumulators is the r-th smallest key
        accumulate(points, feats, colors)    pass 2: each point is added to its voxel's dense fp64 row (572 B per row)
        finalize(hit_thr_ratio)              -> the dict of `PriorVoxelizer.finalize`, rows already in ascending key order
    Peak device memory: the table, V accumulator rows and V output rows (168 B each), and the caller's slice."""

    def __init__(self, min_point: Tensor, voxel_size: float = 0.4, feature_dim: int = 64, with_colors: bool = True,
                 capacity: int = 1 << 16) -> None:
        assert min_point.is_cuda and min_point.numel() == 3, "min_point: 3 floats on the GPU"
        self.dev, self.voxel_size, self.C, self.with_colors = min_point.device, float(voxel_size), int(feature_dim), with_colors
        self.min_point = min_point.detach().to(torch.float32).contiguous()
        self.capacity = _next_pow2(capacity)
        self.keys = torch.full((self.capacity,), -1, device=self.dev, dtype=torch.int64)
        self._n_voxels = torch.zeros(1, device=self.dev, dtype=torch.int64)
        self.status = torch.zeros(1, device=self.dev, dtype=torch.int32)
        self.rows: Optional[Tensor] = None              # slot -> row, after seal()
        self.row_keys: Optional[Tensor] = None          # the V keys in ascending order, after seal()
        self.counts = self.sum_xyz = self.sum_col = self.sum_feat = None

    def _check(self, what: str) -> None:
        st = int(self.status.item())
        for bit, msg in _TABLE_STATUS.items():
            if st & bit:
                raise RuntimeError(f"TileVoxelizer.{what}: {msg}")

    def insert(self, points_m: Tensor) -> None:
        """Pass 1: the voxel keys of points [P,3] f32 metres."""
        assert self.rows is None, "TileVoxelizer.insert after seal()"
        p = points_m.detach().to(torch.float32).contiguous()
        P = p.shape[0]
        if P == 0:
            return
        need = 2 * (int(self._n_voxels.item()) + P)
        if self.capacity < need:
            cap = _next_pow2(need)
            keys = torch.full((cap,), -1, device=self.dev, dtype=torch.int64)
            call("ps_voxel_rehash", ptr(self.keys), self.capacity, ptr(keys), cap, ptr(self.status), stream())
            self.keys, self.capacity = keys, cap
        call("ps_voxel_insert", ptr(p), P, ptr(self.min_point), self.voxel_size, ptr(self.keys), self.capacity,
             ptr(self._n_voxels), ptr(self.status), stream())

    @property
    def n_voxels(self) -> int:
        return int(self._n_voxels.item())

    def seal(self) -> None:
        """Ends pass 1: ranks the keys and allocates the V accumulator rows."""
        assert self.rows is None, "TileVoxelizer.seal twice"
        self._check("seal")
        V = self.n_voxels
        if V == 0:
            raise RuntimeError("TileVoxelizer: no point was inserted")
        self.row_keys = torch.sort(self.keys[self.keys >= 0]).values
        assert self.row_keys.numel() == V
        self.rows = torch.empty(self.capacity, device=self.dev, dtype=torch.int32)
        call("ps_voxel_assign_rows", ptr(self.row_keys), V, ptr(self.keys), self.capacity, ptr(self.rows),
             ptr(self.status), stream())
        z = lambda *s: torch.zeros(*s, device=self.dev, dtype=torch.float64)
        self.counts = torch.zeros(V, device=self.dev, dtype=torch.int32)          # u32 on the device
        self.sum_xyz = z(V, 3)
        self.sum_col = z(V, 3) if self.with_colors else None
        self.sum_feat = z(V, self.C) if self.C else None

    def accumulate(self, points_m: Tensor, features: Optional[Tensor], colors: Optional[Tensor]) -> None:
        """Pass 2: points [P,3] f32 metres (each inserted in pass 1), features [P,C] f16, colors [P,3] f32."""
        assert self.rows is not None, "TileVoxelizer.accumulate before seal()"
        p = points_m.detach().to(torch.float32).contiguous()
        f = None if self.sum_feat is None else features.detach().to(torch.float16).contiguous()
        c = None if self.sum_col is None else colors.detach().to(torch.float32).contiguous()
        assert f is None or f.shape == (p.shape[0], self.C)
        assert c is None or c.shape == (p.shape[0], 3)
        call("ps_voxel_accumulate_rows", ptr(p), ptr(f), ptr(c), p.shape[0], self.C, ptr(self.min_point),
             self.voxel_size, ptr(self.keys), ptr(self.rows), self.capacity, ptr(self.counts), ptr(self.sum_xyz),
             ptr(self.sum_col), ptr(self.sum_feat), ptr(self.status), stream())

    def finalize_rows(self) -> Dict[str, Tensor]:
        """-> every voxel's row before the hit-quantile filter, in ascending key order: {"keys" [V] i64 (packed
        ix<<42 | iy<<21 | iz), "points", "features", "colors", "hits"} as `finalize` gives them.  Frees the table and
        the accumulators as it goes: the voxelizer is spent afterwards."""
        assert self.rows is not None, "TileVoxelizer.finalize before seal()"
        self._check("finalize")
        self.keys = self.rows = None
        dev, V, C = self.dev, self.row_keys.numel(), self.C
        oxyz = torch.empty(V, 3, device=dev, dtype=torch.float32)
        ocol = torch.empty(V, 3, device=dev, dtype=torch.float32) if self.sum_col is not None else None
        ofeat = torch.empty(V, C, device=dev, dtype=torch.float16) if self.sum_feat is not None else None
        hits = torch.empty(V, device=dev, dtype=torch.int64)
        call("ps_voxel_finalize_rows", ptr(self.counts), ptr(self.sum_xyz), ptr(self.sum_col), ptr(self.sum_feat), V, C,
             ptr(oxyz), ptr(ocol), ptr(ofeat), ptr(hits), stream())
        self.counts = self.sum_xyz = self.sum_col = self.sum_feat = None
        return {"keys": self.row_keys, "points": oxyz, "features": ofeat, "colors": ocol, "hits": hits}

    def finalize(self, hit_thr_ratio: float = 0.2) -> Dict[str, Tensor]:
        """-> the dict of `PriorVoxelizer.finalize` (voxels in ascending (ix, iy, iz) order, hit-quantile filtered).
        Frees the table and the accumulators as it goes: the voxelizer is spent afterwards."""
        r = self.finalize_rows()
        dev, hits, oxyz, ocol, ofeat = self.dev, r["hits"], r["points"], r["colors"], r["features"]
        V = hits.numel()
        lo, hi = (int(v) for v in torch.stack(torch.aminmax(hits)).tolist())
        if lo == 0:
            raise RuntimeError("TileVoxelizer: a voxel of pass 1 received no point in pass 2")
        bins = hi + 1
        hist = torch.zeros(bins, device=dev, dtype=torch.int32)
        thr = torch.zeros(1, device=dev, dtype=torch.float64)
        status = torch.zeros(1, device=dev, dtype=torch.int32)
        call("ps_hits_quantile", ptr(hits), V, float(hit_thr_ratio), ptr(hist), bins, ptr(thr), ptr(status), stream())
        keep = hits.to(torch.float64) > thr                 # extract_priors.py:191
        return {"points": oxyz[keep], "features": None if ofeat is None else ofeat[keep],
                "colors": None if ocol is None else ocol[keep], "hits": hits[keep], "hit_thr": thr[0], "n_voxels": V}


def postprocess_priors(points: Tensor, features: Tensor, colors: Tensor, densities: Optional[Tensor],
                       voxel_size: float = 0.4, hit_thr_ratio: float = 0.2, capacity: Optional[int] = None) -> Dict[str, Tensor]:
    """extract_priors.py:156-196 on resident arrays (one tile): density filter, voxel down-sampling, per-voxel means,
    hit-quantile filter.  `capacity`: hash-table slots (default: 2 x the number of points, rounded up to a power of 2)."""
    mn = PriorVoxelizer.min_bound(points, densities)
    vox = PriorVoxelizer(mn, voxel_size, features.shape[1], capacity or 2 * max(points.shape[0], 1024))
    vox.add(points, features, colors, densities)
    return vox.finalize(hit_thr_ratio)


def priors_to_dict(result: Dict[str, Tensor], origin) -> Dict[str, np.ndarray]:
    """The dict extract_priors.py:199-208 pickles (host arrays, reference dtypes)."""
    return {"points": result["points"].cpu().numpy().astype(np.float32),
            "features": result["features"].cpu().numpy().astype(np.float16),
            "colors": result["colors"].cpu().numpy().astype(np.float32),
            "hits": result["hits"].cpu().numpy(),
            "origin": np.asarray(origin.cpu() if torch.is_tensor(origin) else origin).astype(np.float32)}


def save_priors(path: str, result: Dict[str, Tensor], origin) -> None:
    """Write `extracted_priors.pkl` (extract_priors.py:197-208)."""
    with open(path, "wb") as f:
        pickle.dump(priors_to_dict(result, origin), f)
