"""iNGPField (reference: nerfstudio/fields/PreSight/ingp_field.py) on the b200 kernels.

Module nesting and parameter names follow the reference so its checkpoints load unchanged:
`mlp_base_grid.hash_table`, `mlp_base_mlp.layers.{i}`, `mlp_base.{0,1}.*` (the Sequential alias),
`semantic_head.layers.{i}`, `rgb_head.layers.{i}`, buffers `aabb`, `max_res`, `num_levels`, `log2_hashmap_size`.
"""
from __future__ import annotations

from copy import deepcopy
from typing import Dict, Literal, Optional, Tuple

import torch
from torch import Tensor, nn

from .. import ops
from ..cameras.rays import RaySamples
from ..field_components.encodings import HashEncoding, SHEncoding
from ..field_components.mlp import MLP
from ..field_components.spatial_distortions import SpatialDistortion
from .base_field import Field


class FieldHeadNames:
    """Subset of nerfstudio/field_components/field_heads.py:28-43 used by PreSight."""
    RGB = "rgb"
    DENSITY = "density"
    SEMANTICS = "semantics"


class iNGPField(Field):
    def __init__(
        self,
        aabb: Tensor,
        num_layers: int = 2,
        hidden_dim: int = 64,
        geo_feat_dim: int = 15,
        num_levels: int = 16,
        base_res: int = 16,
        max_res: int = 2048,
        log2_hashmap_size: int = 19,
        num_layers_color: int = 3,
        features_per_level: int = 2,
        hidden_dim_color: int = 64,
        appearance_embedding_dim: int = 32,
        use_semantics: bool = False,
        hidden_dim_semantic_head: int = 64,
        semantic_dim: int = 64,
        spatial_distortion: Optional[SpatialDistortion] = None,
        implementation: Literal["b200", "b200+fp32"] = "b200",
        field_type: Literal["iNGP", "TriPlane"] = "iNGP",
        **kwargs,
    ) -> None:
        super().__init__()
        self.register_buffer("aabb", deepcopy(aabb))
        self.geo_feat_dim = geo_feat_dim
        self.register_buffer("max_res", torch.tensor(max_res))
        self.register_buffer("num_levels", torch.tensor(num_levels))
        self.register_buffer("log2_hashmap_size", torch.tensor(log2_hashmap_size))
        self.spatial_distortion = spatial_distortion
        self.appearance_embedding_dim = appearance_embedding_dim
        self.use_semantics = use_semantics
        self.semantic_dim = semantic_dim if use_semantics else 0
        self.base_res = base_res
        self.direction_encoding = SHEncoding(levels=4, implementation=implementation)
        if field_type != "iNGP":
            raise ValueError(f"Unknown `field_type`: {field_type}")
        self.mlp_base_grid = HashEncoding(num_levels=num_levels, min_res=base_res, max_res=max_res,
                                          log2_hashmap_size=log2_hashmap_size, features_per_level=features_per_level,
                                          implementation=implementation)
        self.mlp_base_mlp = MLP(in_dim=self.mlp_base_grid.get_out_dim(), num_layers=num_layers, layer_width=hidden_dim,
                                out_dim=1 + self.geo_feat_dim + self.semantic_dim, activation=nn.ReLU(),
                                out_activation=None, implementation=implementation)
        self.mlp_base = torch.nn.Sequential(self.mlp_base_grid, self.mlp_base_mlp)
        if self.use_semantics:
            self.semantic_head = MLP(in_dim=self.semantic_dim, num_layers=3, layer_width=hidden_dim_semantic_head,
                                     out_dim=semantic_dim, activation=nn.ReLU(), out_activation=None,
                                     implementation=implementation)
        self.rgb_head = MLP(in_dim=self.direction_encoding.get_out_dim() + self.geo_feat_dim + self.appearance_embedding_dim,
                            num_layers=num_layers_color, layer_width=hidden_dim_color, out_dim=3, activation=nn.ReLU(),
                            out_activation=nn.Sigmoid(), implementation=implementation)

    def get_density(self, ray_samples: RaySamples) -> Tuple[Tensor, Tensor]:
        return self.density_fn(ray_samples.frustums.get_positions())

    def density_fn(self, positions: Tensor, times=None) -> Tuple[Tensor, Tensor]:
        """ingp_field.py:168-191: prologue kernel -> hash kernel -> fused MLP kernel -> trunc_exp kernel."""
        x01, selector = ops.normalize_positions(positions, self.aabb_host(), self.spatial_distortion is not None)
        h = self.mlp_base(x01.view(-1, 3)).view(*positions.shape[:-1], -1)
        raw, emb = torch.split(h, [1, self.geo_feat_dim + self.semantic_dim], dim=-1)
        density = ops.trunc_exp(raw.contiguous(), selector.reshape(-1)).view(*positions.shape[:-1], 1)
        return density, emb

    def get_outputs(self, directions: Tensor, density_embedding: Tensor,
                    appearance_embedding: Optional[Tensor]) -> Dict[str, Tensor]:
        """ingp_field.py:193-237."""
        assert density_embedding is not None
        outputs = {}
        outputs_shape = directions.shape[:-1]
        if self.use_semantics:
            density_embedding, semantic_embedding = torch.split(density_embedding, [self.geo_feat_dim, self.semantic_dim],
                                                                dim=-1)
            semantics_input = semantic_embedding.reshape(-1, self.semantic_dim)
            outputs[FieldHeadNames.SEMANTICS] = self.semantic_head(semantics_input).view(*outputs_shape, -1)
        d = self.direction_encoding.forward_raw(directions.reshape(-1, 3))
        parts = [d, density_embedding.reshape(-1, self.geo_feat_dim)]
        if appearance_embedding is not None:
            parts.append(appearance_embedding.reshape(-1, self.appearance_embedding_dim))
        h = torch.cat(parts, dim=-1)
        outputs[FieldHeadNames.RGB] = self.rgb_head(h).view(*outputs_shape, 3)
        return outputs

    def forward(self, ray_samples: RaySamples, appearance_embedding=None) -> Dict[str, Tensor]:
        density, density_embedding = self.get_density(ray_samples)
        dirs = ray_samples.frustums.directions.expand(*density.shape[:-1], 3)
        field_outputs = self.get_outputs(dirs, density_embedding=density_embedding,
                                         appearance_embedding=appearance_embedding)
        field_outputs[FieldHeadNames.DENSITY] = density
        return field_outputs

    def fused_level(self, origins: Tensor, directions: Tensor, eu_bins: Tensor, appearance: Optional[Tensor],
                    threshold: float = 0.5):
        """Fast path of forward() + compositing for contiguous bins (see presight_b200/fused.py).
        appearance: per-ray [N, A] or None.  Returns (weights [N,S,1], rgb, acc, depth_expected_unclipped,
        depth_threshold, semantics, tminmax)."""
        from .. import fused
        enc = self.mlp_base_grid

        def meta(mlp):
            ls = list(mlp.layers)
            return (fused.MlpMeta((ls[0].weight.shape[1],) + tuple(l.weight.shape[0] for l in ls), mlp._out_act),
                    ([l.weight for l in ls], [l.bias for l in ls]))
        base_m, base_p = meta(self.mlp_base_mlp)
        rgb_m, rgb_p = meta(self.rgb_head)
        sem_m, sem_p = meta(self.semantic_head) if self.use_semantics else (None, None)
        return fused.field_level(
            origins, directions, eu_bins, appearance, enc.hash_table, self.aabb_host(),
            self.spatial_distortion is not None,
            fused.GridMeta(enc._scalings_host, enc.log2_hashmap_size, enc.features_per_level), base_m, sem_m, rgb_m,
            self.geo_feat_dim, self.mlp_base_mlp.precision, threshold, base_p, sem_p, rgb_p)

    def _grid_meta(self):
        from .. import fused
        enc = self.mlp_base_grid
        return fused.GridMeta(enc._scalings_host, enc.log2_hashmap_size, enc.features_per_level)

    def supports_level_depth(self, S: int) -> bool:
        """True when `level_depth` serves this field with S samples per ray: a 2-layer base MLP with biases whose density
        head fits the fused density kernels (fused.tc5_density_supported: bf16 class, hidden 64, L*F <= 48)."""
        from .. import fused
        ls = list(self.mlp_base_mlp.layers)
        return (len(ls) == 2 and all(l.bias is not None for l in ls)
                and fused.tc5_density_supported(self._grid_meta(), ls[0].weight.shape[0], self.mlp_base_mlp.precision, S))

    def level_depth(self, origins: Tensor, directions: Tensor, eu_bins: Tensor, threshold: float = 0.5) -> Tensor:
        """Threshold depth [N,1] of the final level from its bins (the depth of `get_depth`), forward only, on the fused
        density kernels: hash gather, base0 + ReLU and the density column of base1 only (no features or 80-wide output
        written to memory).  Callers check `supports_level_depth` first."""
        from .. import fused
        l0, l1 = list(self.mlp_base_mlp.layers)
        return fused.density_level_depth(origins, directions, eu_bins, self.mlp_base_grid.hash_table, self.aabb_host(),
                                         self.spatial_distortion is not None, self._grid_meta(), l0.weight, l0.bias,
                                         l1.weight, l1.bias, threshold)

    def semantic_fn(self, positions: Tensor) -> Tensor:
        """ingp_field.py:253-267."""
        assert self.use_semantics, "Cannot query semantics when `self.use_semantics` is set to False"
        _, density_embedding = self.density_fn(positions)
        _, semantic_embedding = torch.split(density_embedding, [self.geo_feat_dim, self.semantic_dim], dim=-1)
        semantics_input = semantic_embedding.reshape(-1, self.semantic_dim)
        return self.semantic_head(semantics_input).view(*positions.shape[:-1], -1)
