"""Geometry metrics on the device: how far the model's surfaces are from the LiDAR.

    depth_metrics(pred_maps, target_m, pose_scale_factor)   depth errors of rendered depth maps against a LiDAR depth
                                                            image (`ps_depth_metrics`, csrc/depth_metrics.cu)
    NNGrid(ref_points_m, r_m).query(points_m, taus_m)       distance of every point to its nearest reference point
                                                            within r (`ps_nn_grid_*`, csrc/nn_grid.cu)
    prior_geometry_metrics(prior_points_m, ref_points_m, r_m, taus_m)
                                                            accuracy / completeness / precision / recall / F-score of
                                                            extracted priors against a reference cloud

Every result stays on the device until the caller reads it; no floating-point atomics are used, so repeated calls give
bit-identical results.  Reading LiDAR files, projecting sweeps into depth images and cropping reference clouds to a
tile are the caller's (INTEGRATION.md section H).
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Optional, Sequence, Tuple, Union

import torch
from torch import Tensor

from ._lib import NN_BLOCK_QUERIES, NN_MAX_TAUS, NNGrid as _NNGridStruct, call, ptr, stream

DEPTH_METRICS = ("abs_rel", "sq_rel", "rmse", "rmse_log", "a1", "a2", "a3", "n_valid")
_MAX_DEPTH_MAPS = 4


@torch.no_grad()
def depth_metrics(pred_maps: Union[Tensor, Sequence[Tensor]], target_m: Tensor, pose_scale_factor,
                  min_m: float = 1.0, max_m: float = 75.0) -> Tensor:
    """Depth errors of M in [1, 4] rendered depth maps of one image (e.g. the "depth" and "expected_depth" outputs of
    `get_outputs_for_camera_ray_bundle`, [H,W] or [H,W,1] in scene units; one tensor is one map) against a LiDAR depth
    image `target_m` (the same number of pixels, metres, 0 = no LiDAR return) -> [M, 8] f64 on the device, columns
    `DEPTH_METRICS`: abs_rel, sq_rel, rmse, rmse_log, a1, a2, a3, n_valid.

    This is the Eigen et al. / Monodepth evaluation convention: the prediction is brought to metres (divided by
    `pose_scale_factor`, depth along the ray), pixels with min_m < target < max_m count, and the prediction is clamped
    to [min_m, max_m] before the errors are taken.  An image without a valid pixel gives NaN metrics and n_valid 0.
    `pose_scale_factor` is a number or a CUDA tensor whose first element is read on the device (no host read).  The
    exact arithmetic is in csrc/depth_metrics_core.h."""
    maps = [pred_maps] if torch.is_tensor(pred_maps) else list(pred_maps)
    if not 1 <= len(maps) <= _MAX_DEPTH_MAPS:
        raise ValueError(f"depth_metrics takes 1 to {_MAX_DEPTH_MAPS} depth maps, got {len(maps)}")
    HW = target_m.numel()
    if HW == 0:
        raise ValueError("depth_metrics: empty target image")
    for m in maps:
        if m.numel() != HW:
            raise ValueError(f"depth map {tuple(m.shape)} and target {tuple(target_m.shape)} differ in pixel count")
    if not 0.0 < min_m < max_m < math.inf:
        raise ValueError(f"depth_metrics: need 0 < min_m < max_m < inf, got {min_m}, {max_m}")
    dev = maps[0].device
    pred = torch.stack([m.detach().reshape(HW).to(device=dev, dtype=torch.float32) for m in maps]).contiguous()
    tgt = target_m.detach().reshape(HW).to(device=dev, dtype=torch.float32).contiguous()
    if torch.is_tensor(pose_scale_factor) and pose_scale_factor.is_cuda:
        scale_dev, scale = pose_scale_factor.detach().reshape(-1)[:1].to(torch.float32).contiguous(), 1.0
    else:
        v = pose_scale_factor
        scale_dev, scale = None, float(v.reshape(-1)[0] if torch.is_tensor(v) else v)
        if not scale > 0.0:
            raise ValueError(f"depth_metrics: pose_scale_factor must be positive, got {scale}")
    M = len(maps)
    nbytes = C.c_int64(0)
    call("ps_depth_metrics_workspace", M, HW, C.byref(nbytes))
    ws = torch.empty(int(nbytes.value), dtype=torch.uint8, device=dev)
    out = torch.empty(M, len(DEPTH_METRICS), dtype=torch.float64, device=dev)
    call("ps_depth_metrics", ptr(pred), M, HW, ptr(tgt), scale, ptr(scale_dev), float(min_m), float(max_m), ptr(ws),
         ptr(out), stream())
    return out


def _points(p: Tensor, what: str) -> Tensor:
    if p.dim() != 2 or p.shape[1] != 3:
        raise ValueError(f"{what} must be [N,3], got {tuple(p.shape)}")
    if p.shape[0] == 0:
        raise ValueError(f"{what} is empty")
    return p.detach().to(torch.float32).contiguous()


def _taus(taus_m: Sequence[float], r_m: float) -> Tuple[float, ...]:
    taus = tuple(float(t) for t in taus_m)
    if len(taus) > NN_MAX_TAUS:
        raise ValueError(f"at most {NN_MAX_TAUS} thresholds, got {len(taus)}")
    for t in taus:
        if not 0.0 < t <= r_m:
            raise ValueError(f"threshold {t} outside (0, r = {r_m}]")
    return taus


class NNGrid:
    """A reference point cloud [M,3] (f32, metres) on a grid of cells of side `r_m`, for nearest-neighbour distances
    within r.  Building it reads two small values back (the bounds, to check that every axis fits 2^21 cells, and the
    number of occupied cells, to size the cell table); queries make no host read.  The table holds about 2 slots per
    occupied cell (16 B each) and the points are kept once more in cell order."""

    def __init__(self, ref_points_m: Tensor, r_m: float):
        pts = _points(ref_points_m, "reference points")
        if not pts.is_cuda:
            raise RuntimeError("presight_b200 kernels need CUDA tensors (no CPU fallback exists)")
        r = float(r_m)
        dev, M = pts.device, int(pts.shape[0])
        bounds = torch.tensor([math.inf] * 3 + [-math.inf] * 3, dtype=torch.float32).to(dev)
        call("ps_nn_grid_bounds", ptr(pts), M, ptr(bounds), stream())
        b = (C.c_float * 6)(*bounds.tolist())
        keys = torch.empty(M, dtype=torch.int64, device=dev)
        call("ps_nn_grid_keys", ptr(pts), M, b, r, ptr(keys), stream())
        sorted_keys, perm = torch.sort(keys, stable=True)
        n_cells = torch.zeros(1, dtype=torch.int64, device=dev)
        call("ps_nn_grid_count_cells", ptr(sorted_keys), M, ptr(n_cells), stream())
        self.n_cells = int(n_cells)
        self.capacity = max(2, 1 << (2 * self.n_cells - 1).bit_length())
        self.cell_keys = torch.full((self.capacity,), -1, dtype=torch.int64, device=dev)
        self.cell_ranges = torch.zeros(self.capacity, 2, dtype=torch.int32, device=dev)
        self.points = torch.empty_like(pts)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        call("ps_nn_grid_cells", ptr(pts), ptr(perm), ptr(sorted_keys), M, ptr(self.cell_keys), ptr(self.cell_ranges),
             self.capacity, ptr(self.points), ptr(status), stream())
        if int(status) != 0:
            raise RuntimeError(f"NNGrid: building the cell table failed (status {int(status)})")
        self.origin = tuple(b[:3])
        self.r = r
        self.num_points = M

    def _struct(self) -> _NNGridStruct:
        g = _NNGridStruct()
        g.points, g.cell_keys, g.cell_ranges = ptr(self.points), ptr(self.cell_keys), ptr(self.cell_ranges)
        g.capacity, g.cell = self.capacity, self.r
        for a in range(3):
            g.origin[a] = self.origin[a]
        return g

    @torch.no_grad()
    def query(self, points_m: Tensor, taus_m: Sequence[float] = (), chunk: int = 1 << 22,
              return_distances: bool = False) -> Tuple[Tensor, Tensor, Optional[Tensor]]:
        """points_m [N,3] -> (mean distance, a device f64 scalar; counts [K] i64 of distances < taus_m[k]; the distances
        [N] f64 when `return_distances`, else None).  A distance is that to the nearest reference point when it is < r,
        else r; it is computed in fp64 from the fp32 coordinates.  The points run in chunks of `chunk` (rounded down to
        a multiple of PS_NN_BLOCK_QUERIES), so N is not bounded by memory; the results do not depend on the chunk."""
        q = _points(points_m, "query points")
        if q.device != self.points.device:
            raise ValueError(f"query points on {q.device}, grid on {self.points.device}")
        taus = _taus(taus_m, self.r)
        K, N, dev = len(taus), int(q.shape[0]), q.device
        chunk = max(NN_BLOCK_QUERIES, int(chunk) // NN_BLOCK_QUERIES * NN_BLOCK_QUERIES)
        nblocks = -(-N // NN_BLOCK_QUERIES)
        block_sums = torch.empty(nblocks, dtype=torch.float64, device=dev)
        block_counts = torch.empty(nblocks * K, dtype=torch.int64, device=dev) if K else None
        dist = torch.empty(N, dtype=torch.float64, device=dev) if return_distances else None
        taus_host = (C.c_double * max(K, 1))(*taus)
        grid = self._struct()
        for s in range(0, N, chunk):
            n = min(chunk, N - s)
            call("ps_nn_grid_query", C.byref(grid), ptr(q[s:s + n]), n, s // NN_BLOCK_QUERIES, taus_host, K,
                 ptr(None if dist is None else dist[s:s + n]), ptr(block_sums), ptr(block_counts), stream())
        mean = torch.empty(1, dtype=torch.float64, device=dev)
        counts = torch.empty(K, dtype=torch.int64, device=dev)
        call("ps_nn_grid_reduce", ptr(block_sums), ptr(block_counts), nblocks, K, N, ptr(mean),
             ptr(counts) if K else None, stream())
        return mean[0], counts, dist


@torch.no_grad()
def prior_geometry_metrics(prior_points_m: Tensor, ref_points_m: Tensor, r_m: float, taus_m: Sequence[float],
                           chunk: int = 1 << 22, return_distances: bool = False) -> Dict[str, Tensor]:
    """Accuracy and completeness of extracted priors against a reference cloud in the same frame, both [.,3] f32 metres
    (the priors as `PriorExtractor.finalize()["points"]` holds them, without the pkl's `origin`; the reference e.g. the
    tile's LiDAR sweeps, cropped and down-sampled by the caller).  Every distance is the nearest-neighbour distance
    within `r_m`, or r_m when there is none (`NNGrid`).  Returns device tensors:
        accuracy      mean distance from the priors to the reference (f64 scalar)
        completeness  mean distance from the reference to the priors (f64 scalar)
        precision     [K] fraction of priors closer than taus_m[k] to the reference (each tau <= r_m)
        recall        [K] fraction of reference points closer than taus_m[k] to the priors
        fscore        [K] 2 P R / (P + R), 0 where P + R == 0
    and with `return_distances` the per-point distances `prior_to_ref` [N] and `ref_to_prior` [M] (f64).  Empty inputs
    raise a ValueError."""
    prior = _points(prior_points_m, "prior points")
    ref = _points(ref_points_m, "reference points")
    r = float(r_m)
    taus = _taus(taus_m, r)
    acc, prec_n, d_pr = NNGrid(ref, r).query(prior, taus, chunk, return_distances)
    comp, rec_n, d_rp = NNGrid(prior, r).query(ref, taus, chunk, return_distances)
    precision = prec_n.double() / prior.shape[0]
    recall = rec_n.double() / ref.shape[0]
    total = precision + recall
    fscore = torch.where(total > 0, 2.0 * precision * recall / torch.where(total > 0, total, 1.0),
                         torch.zeros_like(total))
    out = {"accuracy": acc, "completeness": comp, "precision": precision, "recall": recall, "fscore": fscore}
    if return_distances:
        out["prior_to_ref"], out["ref_to_prior"] = d_pr, d_rp
    return out
