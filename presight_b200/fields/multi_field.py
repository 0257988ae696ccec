"""Nearest-centroid routers over sub-fields (reference: fields/PreSight/ingp_field_ms.py,
prop_density_field_ms.py, sky_field_ms.py).

Routing runs in `ps_nearest_centroid`; points are then bucketed per sub-field with one device-side sort
(no per-field `torch.any` host sync as in ingp_field_ms.py:103) and a single bincount read-back.
State-dict layout (`centroids`, `fields.{i}.*`) matches the reference.
"""
from __future__ import annotations

from copy import deepcopy
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import torch
from torch import Tensor, nn

from .. import ops
from ..cameras.rays import RaySamples
from .ingp_field import FieldHeadNames, iNGPField
from .prop_density_field import PropNetDensityField
from .sky_field import SkyField


def _route(points: Tensor, centroids: Tensor, n_fields: int):
    """-> (order [P] permutation grouping points by field, counts list[int])."""
    assign = ops.nearest_centroid(points, centroids).long()
    order = torch.argsort(assign, stable=True)
    counts = torch.bincount(assign, minlength=n_fields).tolist()   # one host sync for all fields
    return order, counts


def _dispatch(points: Tensor, centroids: Tensor, n_fields: int, per_field: Callable, extras: Sequence[Optional[Tensor]] = ()):
    """Run `per_field(i, pts_i, *extras_i) -> dict` on every non-empty bucket and scatter the results back."""
    if n_fields == 1:
        return per_field(0, points, *extras)
    order, counts = _route(points, centroids, n_fields)
    sorted_pts = points[order]
    sorted_extras = [None if e is None else e[order] for e in extras]
    pieces: Dict[str, List[Tensor]] = {}
    start = 0
    for i, c in enumerate(counts):
        if c == 0:
            continue
        sub = per_field(i, sorted_pts[start:start + c], *[None if e is None else e[start:start + c] for e in sorted_extras])
        for k, v in sub.items():
            pieces.setdefault(k, []).append(v)
        start += c
    inv = torch.empty_like(order)
    inv[order] = torch.arange(order.numel(), device=order.device)
    return {k: torch.cat(v, dim=0)[inv] for k, v in pieces.items()}


class iNGPFieldMS(nn.Module):
    def __init__(self, fields: List[iNGPField], centroids: Tensor) -> None:
        super().__init__()
        self.register_buffer("centroids", deepcopy(centroids))
        self.fields = nn.ModuleList(fields)

    def forward(self, ray_samples: RaySamples, appearance_embedding: Optional[Tensor]) -> Dict[str, Tensor]:
        """ingp_field_ms.py:80-126."""
        positions = ray_samples.frustums.get_positions()
        output_shape = positions.shape[:-1]
        positions = positions.reshape(-1, 3)
        directions = ray_samples.frustums.directions.expand(*output_shape, 3).reshape(-1, 3)
        app = None if appearance_embedding is None else appearance_embedding.flatten(0, -2)

        def run(i, p, d, a):
            f: iNGPField = self.fields[i]
            density, emb = f.density_fn(p)
            out = f.get_outputs(d, density_embedding=emb, appearance_embedding=a)
            out[FieldHeadNames.DENSITY] = density
            return out
        res = _dispatch(positions, self.centroids, len(self.fields), run, (directions, app))
        return {k: v.reshape(*output_shape, -1) for k, v in res.items()}

    def supports_fused(self) -> bool:
        """One sub-field: the ray-tile fused kernels.  Several: the sub-field mode of the same kernels (routing on the
        device, presight_b200/fused.py) when every sub-field has the reference field's architecture."""
        if len(self.fields) == 1:
            return True
        return self._ms_meta() is not None

    def _ms_meta(self):
        from .. import fused
        f0 = self.fields[0]
        if not f0.use_semantics:
            return None
        enc = f0.mlp_base_grid
        grid = fused.GridMeta(enc._scalings_host, enc.log2_hashmap_size, enc.features_per_level)

        def dims(mlp):
            ls = list(mlp.layers)
            return (ls[0].weight.shape[1],) + tuple(l.weight.shape[0] for l in ls)
        A = f0.appearance_embedding_dim
        base = fused.MlpMeta(dims(f0.mlp_base_mlp), f0.mlp_base_mlp._out_act)
        sem = fused.MlpMeta(dims(f0.semantic_head), f0.semantic_head._out_act)
        rgb = fused.MlpMeta(dims(f0.rgb_head), f0.rgb_head._out_act)
        if not fused.tc5_field_supported(grid, base, sem, rgb, f0.geo_feat_dim, f0.mlp_base_mlp.precision, 64, A):
            return None
        for f in self.fields[1:]:
            e = f.mlp_base_grid
            if (tuple(e._scalings_host) != tuple(enc._scalings_host) or e.log2_hashmap_size != enc.log2_hashmap_size
                    or e.features_per_level != enc.features_per_level or dims(f.mlp_base_mlp) != base.dims
                    or dims(f.semantic_head) != sem.dims or dims(f.rgb_head) != rgb.dims
                    or (f.spatial_distortion is None) != (f0.spatial_distortion is None)):
                return None
        return grid

    def fused_level(self, origins: Tensor, directions: Tensor, eu_bins: Tensor, appearance: Optional[Tensor],
                    threshold: float = 0.5):
        """Fast path of forward() + compositing: see iNGPField.fused_level (one sub-field) / fused.field_level_ms."""
        if len(self.fields) == 1:
            return self.fields[0].fused_level(origins, directions, eu_bins, appearance, threshold)
        from .. import fused
        grid = self._ms_meta()
        params = []
        for f in self.fields:
            layers = [*f.mlp_base_mlp.layers, *f.semantic_head.layers, *f.rgb_head.layers]
            params.append((f.mlp_base_grid.hash_table, [l.weight for l in layers], [l.bias for l in layers]))
        return fused.field_level_ms(origins, directions, eu_bins, appearance, self.centroids,
                                    self._aabbs_host(), self.fields[0].spatial_distortion is not None, grid, threshold,
                                    params)

    def supports_level_depth(self, S: int) -> bool:
        """`level_depth` serves these sub-fields: the first one fits the fused density kernels and all share its grid,
        base-MLP shapes and contraction (the semantic and colour heads play no part in the depth)."""
        f0 = self.fields[0]
        if not f0.supports_level_depth(S):
            return False
        g0 = f0._grid_meta()
        shapes = [l.weight.shape for l in f0.mlp_base_mlp.layers]
        return all(f._grid_meta() == g0 and [l.weight.shape for l in f.mlp_base_mlp.layers] == shapes
                   and all(l.bias is not None for l in f.mlp_base_mlp.layers)
                   and (f.spatial_distortion is None) == (f0.spatial_distortion is None) for f in self.fields[1:])

    def level_depth(self, origins: Tensor, directions: Tensor, eu_bins: Tensor, threshold: float = 0.5) -> Tensor:
        """Threshold depth [N,1] of the final level: iNGPField.level_depth for one sub-field, the routed mode of the fused
        density kernels + one compositing pass for several.  Callers check `supports_level_depth` first."""
        if len(self.fields) == 1:
            return self.fields[0].level_depth(origins, directions, eu_bins, threshold)
        from .. import fused
        params = []
        for f in self.fields:
            l0, l1 = list(f.mlp_base_mlp.layers)
            params.append((f.mlp_base_grid.hash_table, l0.weight, l0.bias, l1.weight, l1.bias))
        return fused.density_level_depth_ms(origins, directions, eu_bins, self.centroids, self._aabbs_host(),
                                            self.fields[0].spatial_distortion is not None, self.fields[0]._grid_meta(),
                                            params, threshold)

    def _aabbs_host(self):
        key = tuple(f.aabb.data_ptr() for f in self.fields) + tuple(f.aabb._version for f in self.fields)
        if getattr(self, "_aabbs_cache", None) is None or self._aabbs_cache[0] != key:
            self._aabbs_cache = (key, [list(f.aabb_host()) for f in self.fields])
        return self._aabbs_cache[1]

    def density_fn(self, positions: Tensor) -> Tuple[Tensor, Tensor]:
        """ingp_field_ms.py:128-153."""
        output_shape = positions.shape[:-1]
        flat = positions.reshape(-1, 3)

        def run(i, p):
            density, emb = self.fields[i].density_fn(p)
            return {"density": density, "embedding": emb}
        res = _dispatch(flat, self.centroids, len(self.fields), run)
        return res["density"].reshape(*output_shape, 1), res["embedding"].reshape(*output_shape, -1)

    def get_density(self, ray_samples: RaySamples):
        return self.density_fn(ray_samples.frustums.get_positions())

    def semantic_fn(self, positions: Tensor) -> Tensor:
        """ingp_field_ms.py:161-185."""
        output_shape = positions.shape[:-1]
        res = _dispatch(positions.reshape(-1, 3), self.centroids, len(self.fields),
                        lambda i, p: {"semantics": self.fields[i].semantic_fn(p)})
        return res["semantics"].reshape(*output_shape, -1)


class PropNetDensityFieldMS(nn.Module):
    def __init__(self, fields: List[PropNetDensityField], centroids: Tensor) -> None:
        super().__init__()
        self.register_buffer("centroids", deepcopy(centroids))
        self.fields = nn.ModuleList(fields)

    def get_density(self, ray_samples: RaySamples) -> Tuple[Tensor, None]:
        return self.density_fn(ray_samples.frustums.get_positions()), None

    def supports_fused(self) -> bool:
        if len(self.fields) == 1:
            return True
        return self._ms_meta() is not None

    def _ms_meta(self):
        from .. import fused
        f0 = self.fields[0]
        if f0.use_linear:
            return None
        enc = f0.encoding
        grid = fused.GridMeta(enc._scalings_host, enc.log2_hashmap_size, enc.features_per_level)
        layers = list(f0.mlp_base[1].layers)
        if not (len(layers) == 2 and layers[1].weight.shape[0] == 1
                and all(l.bias is not None for l in layers)
                and fused.tc5_ms_prop_supported(grid, layers[0].weight.shape[0], f0._precision)):
            return None
        for f in self.fields[1:]:
            e = f.encoding
            ls = None if f.use_linear else list(f.mlp_base[1].layers)
            if (ls is None or tuple(e._scalings_host) != tuple(enc._scalings_host) or e.log2_hashmap_size != enc.log2_hashmap_size
                    or e.features_per_level != enc.features_per_level or len(ls) != 2
                    or ls[0].weight.shape != layers[0].weight.shape
                    or (f.spatial_distortion is None) != (f0.spatial_distortion is None)):
                return None
        return grid

    def level_weights(self, origins: Tensor, directions: Tensor, eu_bins: Tensor) -> Tensor:
        """Fast path of `get_weights(density_fn(positions))`: PropNetDensityField.level_weights for one sub-field, the
        sub-field mode of the fused proposal kernels (routing on the device) for several."""
        if len(self.fields) == 1:
            return self.fields[0].level_weights(origins, directions, eu_bins)
        from .. import fused
        grid = self._ms_meta()
        params = []
        for f in self.fields:
            l0, l1 = list(f.mlp_base[1].layers)
            params.append((f.encoding.hash_table, l0.weight, l0.bias, l1.weight, l1.bias))
        key = tuple(f.aabb.data_ptr() for f in self.fields) + tuple(f.aabb._version for f in self.fields)
        if getattr(self, "_aabbs_cache", None) is None or self._aabbs_cache[0] != key:
            self._aabbs_cache = (key, [list(f.aabb_host()) for f in self.fields])
        return fused.prop_level_weights_ms(origins, directions, eu_bins, self.centroids, self._aabbs_cache[1],
                                           self.fields[0].spatial_distortion is not None, grid, params)

    def density_fn(self, positions: Tensor) -> Tensor:
        """prop_density_field_ms.py:86-105."""
        output_shape = positions.shape[:-1]
        res = _dispatch(positions.reshape(-1, 3), self.centroids, len(self.fields),
                        lambda i, p: {"density": self.fields[i].density_fn(p)})
        return res["density"].reshape(*output_shape, 1)


class SkyFieldMS(nn.Module):
    def __init__(self, fields: List[SkyField], centroids: Tensor) -> None:
        super().__init__()
        self.register_buffer("centroids", deepcopy(centroids))
        self.fields = nn.ModuleList(fields)
        self.batched = True      # several sub-fields: one batched evaluation + selection instead of the routed loop

    def forward(self, ray_samples: RaySamples, appearance_embedding: Optional[Tensor]) -> Dict[str, Tensor]:
        """sky_field_ms.py:81-117 (routed by ray origin)."""
        origins = ray_samples.frustums.origins[:, 0, :]
        directions = ray_samples.frustums.directions[:, 0, :]
        # reference layout [N,S,A] (sample 0 is used) or per-ray [N,A]
        app = None if appearance_embedding is None else (
            appearance_embedding if appearance_embedding.dim() == 2 else appearance_embedding[:, 0, :])
        if len(self.fields) > 1 and self.batched and origins.is_cuda:
            return self._forward_batched(origins.contiguous(), directions.contiguous(), app)
        res = _dispatch(origins.contiguous(), self.centroids, len(self.fields),
                        lambda i, o, d, a: self.fields[i].get_outputs(d, a), (directions, app))
        return {k: v.contiguous() for k, v in res.items()}

    def _forward_batched(self, origins: Tensor, directions: Tensor, app: Optional[Tensor]) -> Dict[str, Tensor]:
        """Several sub-fields, no host synchronisation: the sky networks are per-RAY and tiny (32-wide, 3 layers), so every
        sub-field's two heads run on all rays (the same fused MLP kernels, 2 launches per sub-field and direction) and each
        ray keeps the output of the sub-field nearest to its origin — the values the routed loop of the reference
        computes and, through the selection's gradient (zero rows for the rays of other sub-fields), the same parameter
        gradients.  Costs nf x the sky arithmetic (about 2 ms at 65 536 rays and 16 sub-fields) and buys a step without
        any device->host read; the routed loop (`batched = False`) needs one read of the bucket sizes per call.
        One autograd node per head (ops.mlp_select): the first version's nf nodes and 4 nf element-wise launches per head
        were 5 ms of host time per step at 16 sub-fields (tools/host_profile.py)."""
        sf = ops.nearest_centroid(origins, self.centroids).long()                     # [N]
        d = self.fields[0].direction_encoding.forward_raw(directions)                 # [N,16], no gradient
        x = d if app is None else torch.cat([d, app], dim=-1)

        def head(name, inp):      # one autograd node for the nf networks of this head (ops._MlpSelect)
            mods = [getattr(f, name) for f in self.fields]
            nets = [([l.weight for l in m.layers], [l.bias for l in m.layers]) for m in mods]
            return ops.mlp_select(inp, sf, nets, mods[0]._out_act, mods[0].precision)

        out = {FieldHeadNames.RGB: head("rgb_head", x)}
        if all(f.use_semantics for f in self.fields):
            out[FieldHeadNames.SEMANTICS] = head("semantic_head", d)
        return out
