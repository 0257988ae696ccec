"""fp64 restatement of the geometry metrics (presight_b200/geometry.py): depth errors of rendered depth maps against
LiDAR depth (csrc/depth_metrics_core.h), and nearest-neighbour distances within a radius between two clouds
(csrc/nn_grid.cu) through scipy's cKDTree, with the cell keys of the grid."""
from __future__ import annotations

import numpy as np
from scipy.spatial import cKDTree

DEPTH_METRICS = ("abs_rel", "sq_rel", "rmse", "rmse_log", "a1", "a2", "a3", "n_valid")
CELL_BITS = 21


def depth_metrics(pred_maps, target_m, pose_scale, min_m=1.0, max_m=75.0):
    """[M, 8]: abs_rel, sq_rel, rmse, rmse_log, a1, a2, a3, n_valid of each map (scene units) against target_m (metres,
    0 = no LiDAR).  pred / pose_scale in fp32, valid = min_m < t < max_m, prediction clamped to [min_m, max_m], every
    per-pixel term in fp64 from the fp32 values."""
    t = np.asarray(target_m, np.float32).reshape(-1)
    lo, hi = np.float32(min_m), np.float32(max_m)
    valid = (t > lo) & (t < hi)
    n = int(valid.sum())
    out = np.full((len(pred_maps), 8), np.nan)
    for m, pred in enumerate(pred_maps):
        p = np.asarray(pred, np.float32).reshape(-1) / np.float32(pose_scale)
        p = np.where(p < lo, lo, np.where(p > hi, hi, p)).astype(np.float32)
        out[m, 7] = n
        if n == 0:
            continue
        pd, td = p[valid].astype(np.float64), t[valid].astype(np.float64)
        d = pd - td
        ratio = np.maximum(pd / td, td / pd)
        out[m, :7] = (np.mean(np.abs(d) / td), np.mean(d * d / td), np.sqrt(np.mean(d * d)),
                      np.sqrt(np.mean((np.log(pd) - np.log(td)) ** 2)),
                      np.mean(ratio < 1.25), np.mean(ratio < 1.25 ** 2), np.mean(ratio < 1.25 ** 3))
    return out


def exact_distances(q, p):
    """sqrt(((qx - px)^2 + (qy - py)^2) + (qz - pz)^2) row by row, fp64 from the fp32 coordinates."""
    e = np.asarray(q, np.float32).astype(np.float64) - np.asarray(p, np.float32).astype(np.float64)
    return np.sqrt((e[:, 0] * e[:, 0] + e[:, 1] * e[:, 1]) + e[:, 2] * e[:, 2])


def nn_distances(queries, ref, r):
    """Distance of every query point to its nearest reference point if < r, else r.  cKDTree finds the neighbour on the
    points cast to fp64, searching a little past r; the distance to it is then recomputed in the grid's order of
    operations and compared with r exactly."""
    q = np.asarray(queries, np.float32)
    p = np.asarray(ref, np.float32)
    _, idx = cKDTree(p.astype(np.float64)).query(q.astype(np.float64), k=1, distance_upper_bound=r * (1 + 1e-9),
                                                  workers=-1)
    out = np.full(len(q), float(r))
    found = idx < len(p)
    d = exact_distances(q[found], p[idx[found]])
    out[found] = np.where(d < r, d, r)
    return out


def nn_distances_brute(queries, ref, r):
    """The same by exhaustive search (small sets)."""
    q = np.asarray(queries, np.float32).astype(np.float64)
    p = np.asarray(ref, np.float32).astype(np.float64)
    e = q[:, None, :] - p[None, :, :]
    d = np.sqrt((e[..., 0] * e[..., 0] + e[..., 1] * e[..., 1]) + e[..., 2] * e[..., 2]).min(axis=1)
    return np.where(d < r, d, float(r))


def prior_geometry_metrics(prior, ref, r, taus):
    """accuracy, completeness, precision [K], recall [K], fscore [K] (see presight_b200.geometry)."""
    d_pr, d_rp = nn_distances(prior, ref, r), nn_distances(ref, prior, r)
    prec = np.array([np.mean(d_pr < t) for t in taus])
    rec = np.array([np.mean(d_rp < t) for t in taus])
    tot = prec + rec
    f = np.where(tot > 0, 2 * prec * rec / np.where(tot > 0, tot, 1.0), 0.0)
    return {"accuracy": d_pr.mean(), "completeness": d_rp.mean(), "precision": prec, "recall": rec, "fscore": f,
            "prior_to_ref": d_pr, "ref_to_prior": d_rp}


def cell_coords(points, origin, r):
    """floor(((double)p - (double)origin) / r) per axis, int64."""
    p = np.asarray(points, np.float32).astype(np.float64)
    o = np.asarray(origin, np.float32).astype(np.float64)
    return np.floor((p - o) / r).astype(np.int64)


def cell_keys(points, origin, r):
    c = cell_coords(points, origin, r)
    return (c[:, 0] << (2 * CELL_BITS)) | (c[:, 1] << CELL_BITS) | c[:, 2]


def unpack_cell_keys(keys):
    m = (1 << CELL_BITS) - 1
    keys = np.asarray(keys, np.int64)
    return np.stack([(keys >> (2 * CELL_BITS)) & m, (keys >> CELL_BITS) & m, keys & m], axis=1)


def cells_per_axis(points, r):
    """floor((max - min) / r) + 1 per axis; ValueError when an axis needs more than 2^21 cells."""
    p = np.asarray(points, np.float32)
    lo, hi = p.min(axis=0).astype(np.float64), p.max(axis=0).astype(np.float64)
    cells = np.floor((hi - lo) / r).astype(np.int64) + 1
    if (cells > (1 << CELL_BITS)).any():
        raise ValueError(f"{cells.tolist()} cells per axis exceed 2^21")
    return cells
