"""Synthetic nuScenes-shaped workloads (SURVEY §8d): 6-camera ray batches and random-init city-NeRF configs.

There is no dataset on the bench box, so rays are drawn the way the reference's data pipeline would produce them
(data/PreSight/mynuscenes_ms_dataparser.py:81,284-300; cameras/cameras.py:851-858): 6 pinhole cameras 1600x900,
fx = fy = 1266, yaw offsets {0, +-55, +-110, 180} deg, ego poses on a random walk inside a 400 m x 400 m tile,
world scaled by pose_scale_factor = 0.05 and mean-centred, pixels uniform over the image.
"""
from __future__ import annotations

import math
from typing import Dict, Tuple

import torch

from .model import NerfactoNuscMSModelConfig

POSE_SCALE = 0.05
CAM_YAWS_DEG = (0.0, 55.0, -55.0, 110.0, -110.0, 180.0)
W, H, FX, FY, CX, CY = 1600, 900, 1266.0, 1266.0, 800.0, 450.0


def _trajectory(g: torch.Generator, n_frames: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Ego trajectory: 2-D random walk, 2 m steps, wrapped into the 400 m tile -> (xy [F,2] metres, yaw [F])."""
    steps = torch.randn(n_frames, 2, generator=g) * 2.0
    xy = torch.cumsum(steps, dim=0)
    xy = (xy + 200.0) % 400.0 - 200.0
    ego_yaw = torch.cumsum(torch.randn(n_frames, generator=g) * 0.05, dim=0)
    return xy, ego_yaw


def make_rays(n_rays: int, seed: int = 42, n_frames: int = 200, n_videos: int = 10) -> Dict[str, torch.Tensor]:
    """Host-side (CPU) batch: origins/directions [N,3], camera / video indices [N,1], and loss targets."""
    g = torch.Generator().manual_seed(seed)
    xy, ego_yaw = _trajectory(g, n_frames)                # cameras at z = 1.5 m
    frame = torch.randint(0, n_frames, (n_rays,), generator=g)
    cam = torch.randint(0, 6, (n_rays,), generator=g)
    u = torch.rand(n_rays, generator=g) * W
    v = torch.rand(n_rays, generator=g) * H
    yaw = ego_yaw[frame] + torch.tensor(CAM_YAWS_DEG)[cam] * (math.pi / 180.0)
    dc = torch.stack([(u - CX) / FX, (v - CY) / FY, torch.ones(n_rays)], dim=-1)
    dc = dc / dc.norm(dim=-1, keepdim=True)
    right = torch.stack([torch.sin(yaw), -torch.cos(yaw), torch.zeros(n_rays)], dim=-1)
    down = torch.tensor([0.0, 0.0, -1.0]).expand(n_rays, 3)
    fwd = torch.stack([torch.cos(yaw), torch.sin(yaw), torch.zeros(n_rays)], dim=-1)
    dirs = dc[:, 0:1] * right + dc[:, 1:2] * down + dc[:, 2:3] * fwd
    dirs = dirs / dirs.norm(dim=-1, keepdim=True)
    origins = torch.cat([xy[frame], torch.full((n_rays, 1), 1.5)], dim=-1) * POSE_SCALE
    return {
        "origins": origins.contiguous(),
        "directions": dirs.contiguous(),
        "camera_indices": (frame * 6 + cam).view(-1, 1),
        "video_ids": (frame % n_videos).view(-1, 1),
        "rgb": torch.rand(n_rays, 3, generator=g),
        "features": torch.rand(n_rays, 64, generator=g),
        "sky": (torch.rand(n_rays, 1, generator=g) < 0.15).float(),
        "n_cameras": n_frames * 6,
        "n_videos": n_videos,
    }


def make_cameras(seed: int = 42, n_frames: int = 200) -> Dict[str, torch.Tensor]:
    """The cameras `make_rays(..., seed, n_frames)` draws its rays from, as a `RayGenerator` takes them (host tensors):
    camera_to_worlds [6F,3,4] (OpenGL axes: x right, y up, looking along -z; camera index frame * 6 + camera, as in
    make_rays), fx, fy, cx, cy [6F], and the image size H, W.  A pixel (row v, col u) of camera i gives the ray make_rays
    draws for that camera at the continuous pixel (u + 0.5, v + 0.5)."""
    g = torch.Generator().manual_seed(seed)
    xy, ego_yaw = _trajectory(g, n_frames)
    yaw = (ego_yaw[:, None] + torch.tensor(CAM_YAWS_DEG)[None, :] * (math.pi / 180.0)).reshape(-1)     # [6F]
    C = yaw.shape[0]
    right = torch.stack([torch.sin(yaw), -torch.cos(yaw), torch.zeros(C)], dim=-1)
    up = torch.tensor([0.0, 0.0, 1.0]).expand(C, 3)
    back = -torch.stack([torch.cos(yaw), torch.sin(yaw), torch.zeros(C)], dim=-1)
    origin = torch.cat([xy, torch.full((n_frames, 1), 1.5)], dim=-1).repeat_interleave(6, dim=0) * POSE_SCALE
    c2w = torch.stack([right, up, back, origin], dim=-1)                                             # [C,3,4]
    full = lambda v: torch.full((C,), v)                                                             # noqa: E731
    return {"camera_to_worlds": c2w.contiguous(), "fx": full(FX), "fy": full(FY), "cx": full(CX), "cy": full(CY),
            "H": H, "W": W}


def tile_aabb() -> torch.Tensor:
    """Tile box +-15 m in xy, -5..+15 m in z (dataparser :266-269), scaled by 0.05 -> [1,2,3]."""
    lo = torch.tensor([-215.0, -215.0, -5.0]) * POSE_SCALE
    hi = torch.tensor([215.0, 215.0, 15.0]) * POSE_SCALE
    return torch.stack([lo, hi])[None]


def _common(**kw) -> NerfactoNuscMSModelConfig:
    base = dict(near_plane=0.1 * POSE_SCALE, far_plane=1000.0 * POSE_SCALE,
                piecewise_sampler_threshold=100.0 * POSE_SCALE)
    base.update(kw)
    return NerfactoNuscMSModelConfig(**base)


def config_c1(implementation: str = "b200") -> NerfactoNuscMSModelConfig:
    """BASELINE config 1/3 — nerfacto-style: main L16 F2 T2^19 16->2048; props L5 F2 T2^17 hidden 16,
    16->128 / 16->256; samples 256/96/48; no semantics; 32-d appearance (SURVEY §8 C1)."""
    return _common(
        num_levels=16, base_res=16, max_res=2048, log2_hashmap_size=19, features_per_level=2,
        num_proposal_samples_per_ray=(256, 96), num_nerf_samples_per_ray=48,
        proposal_net_args_list=[
            {"hidden_dim": 16, "log2_hashmap_size": 17, "num_levels": 5, "max_res": 128, "features_per_level": 2},
            {"hidden_dim": 16, "log2_hashmap_size": 17, "num_levels": 5, "max_res": 256, "features_per_level": 2}],
        use_semantics=False, appearance_embed_dim=32, video_embed_dim=0, use_sky_model=False,
        implementation=implementation)


def config_c2(implementation: str = "b200") -> NerfactoNuscMSModelConfig:
    """BASELINE config 2/4 — PreSight city NeRF train step: main L16 F2 T2^22 16->2048; props L8 F1 T2^20
    hidden 64, 16->1024 / 16->4096; samples 128/64/64; 64-d semantics; 4+12-d appearance; sky model."""
    return _common(
        num_levels=16, base_res=16, max_res=2048, log2_hashmap_size=22, features_per_level=2,
        num_proposal_samples_per_ray=(128, 64), num_nerf_samples_per_ray=64,
        proposal_net_args_list=[
            {"hidden_dim": 64, "log2_hashmap_size": 20, "num_levels": 8, "max_res": 1024, "features_per_level": 1},
            {"hidden_dim": 64, "log2_hashmap_size": 20, "num_levels": 8, "max_res": 4096, "features_per_level": 1}],
        use_semantics=True, semantic_dim=64, appearance_embed_dim=4, video_embed_dim=12, use_sky_model=True,
        sky_mlp_dims=32, implementation=implementation)


def config_presight(implementation: str = "b200") -> NerfactoNuscMSModelConfig:
    """PreSight's shipped shape (configs/method_configs.py:87-141 = the model's defaults): main L10 F4 T2^20 16->16384 per
    sub-field, props L8 F1 T2^20 hidden 64 (16->1024 / 16->4096), samples 128/64/64, 64-d semantics, sky model; used with
    16 sub-fields (`num_aabbs=16`), see `sub_field_layout`."""
    return _common(implementation=implementation)


def sub_field_layout(n_fields: int = 16) -> Tuple[torch.Tensor, torch.Tensor]:
    """-> (centroids [nf,3], aabbs [nf,2,3]) in scene units: sub-fields on a sqrt(nf) x sqrt(nf) lattice over the 400 m
    tile — what the dataparser's k-means over camera positions gives for a uniformly driven tile
    (mynuscenes_ms_dataparser.py:230-271: a box around each cluster's cameras with a 15 m margin, -5..+15 m in z)."""
    k = int(round(math.sqrt(n_fields)))
    assert k * k == n_fields, "sub-field count must be a square"
    cell = 400.0 / k
    cx = (torch.arange(k, dtype=torch.float32) + 0.5) * cell - 200.0
    cen = torch.stack(torch.meshgrid(cx, cx, indexing="ij"), dim=-1).reshape(-1, 2)
    centroids = torch.cat([cen, torch.full((n_fields, 1), 1.5)], dim=-1)
    half = cell / 2 + 15.0
    lo = torch.cat([cen - half, torch.full((n_fields, 1), -5.0)], dim=-1)
    hi = torch.cat([cen + half, torch.full((n_fields, 1), 15.0)], dim=-1)
    return centroids * POSE_SCALE, torch.stack([lo, hi], dim=1) * POSE_SCALE


def prior_tile_grid(tile_index: int) -> torch.Tensor:
    """C5: 400 x 200 x 16 voxel centres = 100 m x 50 m x 8 m at 0.25 / 0.25 / 0.5 m around a tile-specific centre, world
    metres x pose scale (SURVEY §8d) -> [1 280 000, 3] on the host."""
    g = torch.Generator().manual_seed(tile_index)
    centre = (torch.rand(2, generator=g) - 0.5) * 300.0
    xs = torch.arange(400, dtype=torch.float32) * 0.25 - 50.0 + centre[0]
    ys = torch.arange(200, dtype=torch.float32) * 0.25 - 25.0 + centre[1]
    zs = torch.arange(16, dtype=torch.float32) * 0.5 - 2.0
    pts = torch.stack(torch.meshgrid(xs, ys, zs, indexing="ij"), dim=-1).reshape(-1, 3)
    return pts * POSE_SCALE


def prior_query_bytes_per_point(cfg: NerfactoNuscMSModelConfig) -> Tuple[int, int]:
    """(reference-faithful, duplicate-main-encode-elided) algorithmic bytes per queried point (SURVEY §8d C5)."""
    props = 0
    for i in range(cfg.num_proposal_iterations):
        a = cfg.proposal_net_args_list[min(i, len(cfg.proposal_net_args_list) - 1)]
        props += hash_bytes_fwd(a["num_levels"], a["features_per_level"])
    main = hash_bytes_fwd(cfg.num_levels, cfg.features_per_level)
    return 2 * main + props + 4 + 128, main + props + 4 + 128


# algorithmic bytes (SURVEY §8d): hash fwd = 12 + 8LF*4 + LF*4, bwd = 12 + LF*4 + 2*8LF*4 per point
def hash_bytes_fwd(L: int, F: int) -> int:
    return 12 + 8 * L * F * 4 + L * F * 4


def hash_bytes_bwd(L: int, F: int) -> int:
    return 12 + L * F * 4 + 2 * 8 * L * F * 4


def step_bytes_per_ray(cfg: NerfactoNuscMSModelConfig, update_step: bool = True) -> int:
    """Algorithmic bytes of one train step per ray: sum over sampling levels of S_k x (hash fwd + hash bwd for the
    nets trained this step) (SURVEY §8d / BASELINE.md §2: C2 = 378 880, C1 = 535 424)."""
    total = 0
    for i, S in enumerate(cfg.num_proposal_samples_per_ray):
        a = cfg.proposal_net_args_list[min(i, len(cfg.proposal_net_args_list) - 1)]
        L, F = a["num_levels"], a["features_per_level"]
        total += S * (hash_bytes_fwd(L, F) + (hash_bytes_bwd(L, F) if update_step else 0))
    total += cfg.num_nerf_samples_per_ray * (hash_bytes_fwd(cfg.num_levels, cfg.features_per_level)
                                             + hash_bytes_bwd(cfg.num_levels, cfg.features_per_level))
    return total


def depth_pass_bytes_per_ray(cfg: NerfactoNuscMSModelConfig) -> int:
    """Algorithmic bytes of the eval depth pass per ray (get_depth / get_surface_hits): sum over the sampling levels of
    S_k x hash fwd bytes (C2 = 132 096, PreSight's shipped shape = 150 528)."""
    total = 0
    for i, S in enumerate(cfg.num_proposal_samples_per_ray):
        a = cfg.proposal_net_args_list[min(i, len(cfg.proposal_net_args_list) - 1)]
        total += S * hash_bytes_fwd(a["num_levels"], a["features_per_level"])
    return total + cfg.num_nerf_samples_per_ray * hash_bytes_fwd(cfg.num_levels, cfg.features_per_level)
