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

`ShardedPriorExtractor` spreads one tile's extraction over the GPUs of a process group: each rank adds its share of the
rays, and finalize() moves every stored hit to the rank that owns its voxel (ps_voxel_partition + all_to_all_single),
voxelises there, applies the hit threshold of all ranks' voxels and gathers the kept voxels on one rank.

Pixel selection (image decoding, seg-mask filtering) stays with the caller, who hands rays built by
`cameras.RayGenerator` from (camera, row, col) indices.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Tuple

import torch
import torch.distributed as dist
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
        blocks = [(p[:k], c[:k]) for (p, c), k in zip(self._blocks, self._filled())]
        return self._voxelize(blocks, self._min).finalize(self.hit_thr_ratio)

    def _voxelize(self, blocks: List[Tuple[Tensor, Tensor]], anchor: Tensor) -> TileVoxelizer:
        """TileVoxelizer over stored hits (scene-unit points, colours), both passes done: ready to finalize."""
        vox = TileVoxelizer(anchor, self.voxel_size, self.model.config.semantic_dim,
                            capacity=2 * min(self.insert_slice, sum(p.shape[0] for p, _ in blocks)))
        # metres exactly as ps_surface_hits computes them: an element-wise IEEE division (torch turns a division by a
        # Python scalar into a multiplication by its reciprocal, which can differ in the last bit)
        scale = torch.full((1, 3), self.pose_scale, device=anchor.device, dtype=torch.float32)
        for pts, _ in blocks:
            for i in range(0, pts.shape[0], self.insert_slice):
                vox.insert(pts[i:i + self.insert_slice] / scale)
        vox.seal()
        for pts, cols in blocks:
            for i in range(0, pts.shape[0], self.chunk_rays):
                p = pts[i:i + self.chunk_rays]
                _, feats = self.model.query_priors(p)
                vox.accumulate(p / scale, feats, cols[i:i + self.chunk_rays])
        return vox


class ShardedPriorExtractor(PriorExtractor):
    """`PriorExtractor` for one tile over the GPUs of a `torch.distributed` group (NCCL, one GPU per rank).

    Each rank `add()`s its own share of the tile's rays, in any split (`parallel.shard_range`, round-robin, or none at
    all on some ranks).  `finalize(dst)` then returns, on rank `dst`, what `PriorExtractor.finalize` returns for all the
    ranks' rays on one GPU -- the same voxels, hit counts, threshold and features; centres and colours up to the
    rounding of their fp64 sums -- and None on the other ranks:
        anchor      all-reduce MIN of the ranks' running minima (the lattice anchor is a per-axis minimum)
        exchange    per store block: ps_voxel_partition packs the hits by the rank that owns their voxel (a hash of the
                    voxel key), the counts are swapped (one host read) and the hits move with all_to_all_single; the
                    block is freed.  `max over ranks` rounds of one block each, so a rank holds its store, one block's
                    send buffer and the hits it owns
        voxelize    TileVoxelizer over the owned hits: the ranks' voxel sets are disjoint, and each voxel gets all its
                    hits on its owner
        threshold   the hit quantile over the sum of the ranks' histograms of per-voxel hit counts
        gather      the kept rows of every rank to `dst`, ordered by voxel key
    group: the process group (None: the default one; world 1 when no process group is initialised).  The store is
    released as it is exchanged: the extractor is spent after finalize()."""

    def __init__(self, model, pose_scale_factor: float, voxel_size: float = 0.4, hit_thr_ratio: float = 0.2,
                 max_range_m: Optional[float] = None, z_range_m: Optional[Tuple[Optional[float], Optional[float]]] = None,
                 chunk_rays: int = 1 << 17, block_hits: int = 1 << 24, insert_slice: int = 1 << 24, group=None) -> None:
        super().__init__(model, pose_scale_factor, voxel_size, hit_thr_ratio, max_range_m, z_range_m, chunk_rays,
                         block_hits, insert_slice)
        on = dist.is_available() and dist.is_initialized()
        self.group = group
        self.world = dist.get_world_size(group) if on else 1
        self.rank = dist.get_rank(group) if on else 0
        self.exchanged_bytes = 0                         # hits this rank sent to other ranks in finalize(), 24 B each

    def _all_reduce(self, t: Tensor, op) -> Tensor:
        if self.world > 1:
            dist.all_reduce(t, op=op, group=self.group)
        return t

    def _all_gather(self, t: Tensor) -> List[int]:
        """The ranks' int64 vectors `t`, concatenated in rank order, on the host."""
        if self.world == 1:
            return t.tolist()
        out = torch.empty(self.world * t.numel(), device=t.device, dtype=t.dtype)
        dist.all_gather_into_tensor(out, t, group=self.group)
        return out.tolist()

    def _peer(self, r: int) -> int:
        return r if self.group is None else dist.get_global_rank(self.group, r)

    @torch.no_grad()
    def finalize(self, dst: int = 0) -> Optional[Dict[str, Tensor]]:
        """-> on rank `dst`, the result dict of `PriorExtractor.finalize` for the rays of every rank; None elsewhere.
        Every rank of the group calls it."""
        assert 0 <= dst < self.world, f"dst {dst} is not a rank of a group of {self.world}"
        anchor, rounds = self._anchor()
        owned = self._exchange(anchor, rounds)
        kept, n_voxels, thr = self._voxelize_owned(owned, anchor)
        return self._gather(kept, n_voxels, thr, dst)

    def _anchor(self) -> Tuple[Tensor, int]:
        """The global lattice anchor and the number of exchange rounds; the same error on every rank when there is
        nothing to voxelise or a store overflowed."""
        dev = self._min.device if self._min is not None else torch.device("cuda", torch.cuda.current_device())
        anchor = self._min.clone() if self._min is not None else torch.full((3,), float("inf"), device=dev)
        self._all_reduce(anchor, dist.ReduceOp.MIN)
        flags = torch.zeros(2, device=dev, dtype=torch.int64)          # store blocks, store status
        flags[0] = len(self._blocks)
        if self._status is not None:
            flags[1] = self._status[0]
        self._all_reduce(flags, dist.ReduceOp.MAX)
        rounds, st = flags.tolist()
        if bool(torch.isinf(anchor).any()):
            raise RuntimeError("PriorExtractor: no surface hit passed the selector and the density filter")
        if st & 1:
            raise RuntimeError("PriorExtractor: a chunk's hits did not fit their store block")
        return anchor, rounds

    def _exchange(self, anchor: Tensor, rounds: int) -> List[Tuple[Tensor, Tensor]]:
        """Moves every stored hit to the rank that owns its voxel -> the hits this rank owns (points, colours)."""
        dev, W = anchor.device, self.world
        filled = self._filled()
        nbytes = C.c_int64()
        check(load().ps_voxel_partition_workspace(self.block_hits, W, C.byref(nbytes)), "ps_voxel_partition_workspace")
        ws = torch.empty(nbytes.value, device=dev, dtype=torch.uint8)
        counts = torch.empty(W, device=dev, dtype=torch.int64)
        recv_counts = torch.empty(W, device=dev, dtype=torch.int64)
        status = torch.zeros(1, device=dev, dtype=torch.int32)
        owned: List[Tuple[Tensor, Tensor]] = []
        self.exchanged_bytes = 0
        for i in range(rounds):
            if i < len(self._blocks):                   # ranks with fewer blocks send empty rounds
                n = filled[i]
                pts, cols = (t[:n] for t in self._blocks[i])
                self._blocks[i] = None
            else:
                n = 0
                pts = cols = torch.empty(0, 3, device=dev)
            send_p = torch.empty(n, 3, device=dev)
            send_c = torch.empty(n, 3, device=dev)
            call("ps_voxel_partition", ptr(pts), ptr(cols), n, self.pose_scale, ptr(anchor), self.voxel_size, W,
                 ptr(send_p), ptr(send_c), ptr(counts), ptr(status), ptr(ws), stream())
            del pts, cols                               # the store block goes back to the allocator
            if W == 1:
                owned.append((send_p, send_c))
                continue
            dist.all_to_all_single(recv_counts, counts, group=self.group)
            split = torch.cat([counts, recv_counts]).tolist()
            sent, recv = split[:W], split[W:]
            recv_p = torch.empty(sum(recv), 3, device=dev)
            recv_c = torch.empty(sum(recv), 3, device=dev)
            dist.all_to_all_single(recv_p, send_p, recv, sent, group=self.group)
            dist.all_to_all_single(recv_c, send_c, recv, sent, group=self.group)
            self.exchanged_bytes += (sum(sent) - sent[self.rank]) * self.HIT_BYTES
            owned.append((recv_p, recv_c))
            del send_p, send_c
        self._blocks, self._sealed = [], []
        if int(self._all_reduce(status, dist.ReduceOp.MAX).item()) & 2:
            raise RuntimeError("PriorExtractor: a voxel index exceeds 21 bits per axis (tile larger than 2^21 voxels "
                               "across)")
        return owned

    def _voxelize_owned(self, owned: List[Tuple[Tensor, Tensor]], anchor: Tensor):
        """TileVoxelizer over this rank's hits, filtered by the hit threshold of all ranks' voxels -> (kept rows,
        voxels of all ranks, threshold [1] f64)."""
        dev = anchor.device
        if sum(p.shape[0] for p, _ in owned):
            rows = self._voxelize(owned, anchor).finalize_rows()
        else:                                           # this rank owns no voxel
            C_ = self.model.config.semantic_dim
            rows = {"keys": torch.empty(0, device=dev, dtype=torch.int64), "points": torch.empty(0, 3, device=dev),
                    "features": torch.empty(0, C_, device=dev, dtype=torch.float16),
                    "colors": torch.empty(0, 3, device=dev), "hits": torch.empty(0, device=dev, dtype=torch.int64)}
        del owned
        hits = rows["hits"]
        V = hits.numel()
        lo, hi = (int(v) for v in torch.stack(torch.aminmax(hits)).tolist()) if V else (1, 0)
        if lo == 0:
            raise RuntimeError("TileVoxelizer: a voxel of pass 1 received no point in pass 2")
        per_rank = self._all_gather(torch.tensor([V, hi], device=dev, dtype=torch.int64))
        n_voxels, bins = sum(per_rank[0::2]), max(per_rank[1::2]) + 1
        hist = torch.zeros(bins, device=dev, dtype=torch.int32)        # u32 on the device
        status = torch.zeros(1, device=dev, dtype=torch.int32)
        call("ps_hits_histogram", ptr(hits), V, ptr(hist), bins, ptr(status), stream())
        self._all_reduce(hist, dist.ReduceOp.SUM)
        thr = torch.zeros(1, device=dev, dtype=torch.float64)
        call("ps_hits_quantile_from_histogram", ptr(hist), bins, n_voxels, float(self.hit_thr_ratio), ptr(thr),
             stream())
        keep = hits.to(torch.float64) > thr             # extract_priors.py:191
        return {k: v[keep] for k, v in rows.items()}, n_voxels, thr

    def _gather(self, kept: Dict[str, Tensor], n_voxels: int, thr: Tensor, dst: int) -> Optional[Dict[str, Tensor]]:
        """The kept rows of every rank -> rank `dst`, in ascending key order (None on the other ranks)."""
        if self.world > 1:
            K = self._all_gather(torch.tensor([kept["keys"].numel()], device=thr.device, dtype=torch.int64))
            ops, parts = [], {}
            for name, t in kept.items():
                if self.rank == dst:
                    parts[name] = [t if r == dst else torch.empty((K[r],) + tuple(t.shape[1:]), device=t.device,
                                                                  dtype=t.dtype) for r in range(self.world)]
                    ops += [dist.P2POp(dist.irecv, parts[name][r], self._peer(r), self.group)
                            for r in range(self.world) if r != dst and K[r]]
                elif K[self.rank]:
                    ops.append(dist.P2POp(dist.isend, t, self._peer(dst), self.group))
            if ops:
                for req in dist.batch_isend_irecv(ops):
                    req.wait()
            if self.rank != dst:
                return None
            kept = {name: torch.cat(p) for name, p in parts.items()}
            order = torch.argsort(kept["keys"])         # owners hold disjoint keys: a total order
            kept = {name: t[order] for name, t in kept.items()}
        return {"points": kept["points"], "features": kept["features"], "colors": kept["colors"],
                "hits": kept["hits"], "hit_thr": thr[0], "n_voxels": n_voxels}
