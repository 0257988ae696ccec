"""City-NeRF model driver (reference: nerfstudio/models/PreSight/nerfacto_nusc_ms.py).

`NerfactoNuscMSModel` wires the b200 fields, the proposal sampler and the compositing kernels exactly like the
reference's `populate_modules` (:203-383), `get_outputs` (:452-546), `get_depth` (:688-708) and the prior query of
scripts/extract_priors.py:130-138.  Module names (`field`, `proposal_networks`, `sky_model`,
`appearance_embedding`, `video_embedding`) match the reference so state dicts are interchangeable.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import TYPE_CHECKING, Dict, List, Literal, Optional, Tuple

import numpy as np
import torch
from torch import Tensor, nn

from . import ops
from .cameras.rays import RayBundle, RaySamples
from .field_components.spatial_distortions import SceneContraction
from .fields.ingp_field import FieldHeadNames, iNGPField
from .fields.multi_field import PropNetDensityFieldMS, SkyFieldMS, iNGPFieldMS
from .fields.prop_density_field import PropNetDensityField
from .fields.sky_field import SkyField
from .model_components.ray_samplers import ProposalNetworkSampler, SpacedSampler
from .model_components.renderers import AccumulationRenderer, DepthRenderer, RGBRenderer

if TYPE_CHECKING:
    from .metrics import LPIPS

VIDEO_ID = "video_id"


@dataclass
class NerfactoNuscMSModelConfig:
    """Hot-path subset of the reference's config (nerfacto_nusc_ms.py:76-200), same names and defaults."""
    near_plane: float = 0.1
    far_plane: float = 1000.0
    background_color: Literal["random", "last_sample", "black", "white"] = "black"
    hidden_dim: int = 64
    hidden_dim_color: int = 64
    num_levels: int = 10
    base_res: int = 16
    max_res: int = 16384
    log2_hashmap_size: int = 20
    features_per_level: int = 4
    num_proposal_samples_per_ray: Tuple[int, ...] = (128, 64)
    num_nerf_samples_per_ray: int = 64
    proposal_update_every: int = 5
    proposal_warmup: int = 1000
    use_proposal_weight_anneal: bool = True
    proposal_weights_anneal_slope: float = 10.0
    proposal_weights_anneal_max_num_iters: int = 1000
    num_proposal_iterations: int = 2
    use_same_proposal_network: bool = False
    proposal_net_args_list: List[Dict] = field(
        default_factory=lambda: [
            {"features_per_level": 1, "log2_hashmap_size": 20, "num_levels": 8, "base_res": 16, "max_res": 1024,
             "use_linear": False},
            {"features_per_level": 1, "log2_hashmap_size": 20, "num_levels": 8, "base_res": 16, "max_res": 4096,
             "use_linear": False},
        ])
    piecewise_sampler_threshold: float = 1.0
    use_single_jitter: bool = True
    disable_scene_contraction: bool = False
    implementation: Literal["b200", "b200+fp32"] = "b200"
    appearance_embed_dim: int = 4
    video_embed_dim: int = 12
    use_sky_model: bool = True
    num_sky_mlp_layers: int = 3
    sky_mlp_dims: int = 32
    use_semantics: bool = True
    semantic_dim: int = 64
    use_average_appearance_embedding: bool = True
    eval_num_rays_per_chunk: int = 1 << 15
    # loss dict (nerfacto_nusc_ms.py:127-133,167,192)
    interlevel_loss_mult: float = 1.0
    enable_z_anti_aliasing: bool = True
    pulse_width: Tuple[float, ...] = (0.03, 0.003)
    distortion_loss_mult: float = 0.002
    sky_loss_mult: float = 0.001
    semantic_loss_mult: float = 0.5
    # depth supervision (:169-199); needs batch["depth"] (metres) and batch["pose_scale_factor"]
    use_lidar_loss: bool = False
    use_monodepth_loss: bool = False
    expected_depth_loss_mult: float = 1.0
    lidar_depth_upperbound: float = 75.0
    monodepth_depth_upperbound: float = 40.0
    monodepth_loss_inverse: bool = False
    line_of_sight_mult: float = 0.1
    line_of_sight_decay_steps: int = 5000
    line_of_sight_start_step: int = 1000
    line_of_sight_end_step: int = 30000
    line_of_sight_max_sigma: float = 5.0
    line_of_sight_min_sigma: float = 2.0


class TrainingCallbackLocation:
    """engine/callbacks.py:48-53."""
    BEFORE_TRAIN_ITERATION = "BEFORE_TRAIN_ITERATION"
    AFTER_TRAIN_ITERATION = "AFTER_TRAIN_ITERATION"


class TrainingCallback:
    """The subset of engine/callbacks.py:56-117 the model's callbacks use: `func(step=...)` every
    `update_every_num_iters` iterations at the listed locations."""

    def __init__(self, where_to_run, func, update_every_num_iters: Optional[int] = 1) -> None:
        self.where_to_run, self.func, self.update_every_num_iters = list(where_to_run), func, update_every_num_iters

    def run_callback(self, step: int) -> None:
        if self.update_every_num_iters is None or step % self.update_every_num_iters == 0:
            self.func(step=step)

    def run_callback_at_location(self, step: int, location) -> None:
        if location in self.where_to_run:
            self.run_callback(step=step)


class _EmbeddingLookup(torch.autograd.Function):
    """weight[idx] whose backward is one index_add_ (atomics) instead of torch's sort + segmented reduction — the tables
    here have a handful of rows (cameras, videos) and tens of thousands of lookups per step."""

    @staticmethod
    def forward(ctx, weight, idx):
        ctx.save_for_backward(idx)
        ctx.shape = weight.shape
        return weight.index_select(0, idx.reshape(-1)).view(*idx.shape, weight.shape[1])

    @staticmethod
    def backward(ctx, g):
        (idx,) = ctx.saved_tensors
        gw = torch.zeros(ctx.shape, device=g.device, dtype=g.dtype)
        gw.index_add_(0, idx.reshape(-1), g.reshape(-1, ctx.shape[1]))
        return gw, None


class Embedding(nn.Module):
    """nerfstudio/field_components/embedding.py:24-55."""

    def __init__(self, in_dim: int, out_dim: int) -> None:
        super().__init__()
        self.in_dim, self.out_dim = in_dim, out_dim
        self.embedding = nn.Embedding(in_dim, out_dim)

    def mean(self, dim=0):
        return self.embedding.weight.mean(dim)

    def forward(self, in_tensor: Tensor) -> Tensor:
        if in_tensor.is_cuda and self.embedding.weight.requires_grad and torch.is_grad_enabled():
            return _EmbeddingLookup.apply(self.embedding.weight, in_tensor)
        return self.embedding(in_tensor)


class NearFarCollider:
    """nerfstudio/model_components/scene_colliders.py:169-187."""

    def __init__(self, near_plane: float, far_plane: float) -> None:
        self.near_plane, self.far_plane = near_plane, far_plane
        self.training = True

    def __call__(self, ray_bundle: RayBundle) -> RayBundle:
        ones = torch.ones_like(ray_bundle.origins[..., 0:1])
        near_plane = self.near_plane if self.training else 0
        ray_bundle.nears = ones * near_plane
        ray_bundle.fars = ones * self.far_plane
        return ray_bundle


class NerfactoNuscMSModel(nn.Module):
    # LPIPS of the evaluation images (`metrics.LPIPS`, built from the caller's pretrained weights); None leaves it out.
    # A plain attribute, not a submodule, so state_dict() keeps the reference's keys.
    lpips: Optional[LPIPS] = None
    # [256,3] colormap table (e.g. matplotlib's turbo colours) for the evaluation images; None returns them raw.  A plain
    # attribute as well, for the same reason.
    colormap: Optional[Tensor] = None

    def __init__(self, config: NerfactoNuscMSModelConfig, centroids: Tensor, aabbs: Tensor, num_train_cameras: int = 1,
                 num_train_videos: int = 1) -> None:
        super().__init__()
        self.config = config
        self.use_fused = True      # level-fused fast paths for single-sub-field models (presight_b200/fused.py)
        self.centroids = centroids
        self.aabbs = aabbs
        c = config
        contraction = None if c.disable_scene_contraction else SceneContraction(order=float("inf"))
        app_dim = c.appearance_embed_dim + c.video_embed_dim
        fields = [iNGPField(aabb, hidden_dim=c.hidden_dim, num_levels=c.num_levels, max_res=c.max_res,
                            base_res=c.base_res, features_per_level=c.features_per_level,
                            log2_hashmap_size=c.log2_hashmap_size, hidden_dim_color=c.hidden_dim_color,
                            spatial_distortion=contraction, use_semantics=c.use_semantics, semantic_dim=c.semantic_dim,
                            appearance_embedding_dim=app_dim, implementation=c.implementation) for aabb in aabbs]
        self.field = iNGPFieldMS(fields, centroids)
        if c.appearance_embed_dim > 0:
            self.appearance_embedding = Embedding(num_train_cameras, c.appearance_embed_dim)
        if c.video_embed_dim > 0:
            self.video_embedding = Embedding(num_train_videos, c.video_embed_dim)
        self.density_fns = []
        self.proposal_networks = nn.ModuleList()
        n_props = c.num_proposal_iterations
        if c.use_same_proposal_network:
            assert len(c.proposal_net_args_list) == 1, "Only one proposal network is allowed."
            net = PropNetDensityFieldMS([PropNetDensityField(aabb, spatial_distortion=contraction,
                                                             **c.proposal_net_args_list[0],
                                                             implementation=c.implementation) for aabb in aabbs],
                                        centroids)
            self.proposal_networks.append(net)
            self.density_fns.extend([net.density_fn for _ in range(n_props)])
        else:
            for i in range(n_props):
                args = c.proposal_net_args_list[min(i, len(c.proposal_net_args_list) - 1)]
                net = PropNetDensityFieldMS([PropNetDensityField(aabb, spatial_distortion=contraction, **args,
                                                                 implementation=c.implementation) for aabb in aabbs],
                                            centroids)
                self.proposal_networks.append(net)
            self.density_fns.extend([net.density_fn for net in self.proposal_networks])

        def update_schedule(step):
            return np.clip(np.interp(step, [0, c.proposal_warmup], [0, c.proposal_update_every]), 1,
                           c.proposal_update_every)
        initial_sampler = SpacedSampler(piecewise_threshold=c.piecewise_sampler_threshold,
                                        single_jitter=c.use_single_jitter)
        self.proposal_sampler = ProposalNetworkSampler(
            num_nerf_samples_per_ray=c.num_nerf_samples_per_ray,
            num_proposal_samples_per_ray=c.num_proposal_samples_per_ray,
            num_proposal_network_iterations=c.num_proposal_iterations, single_jitter=c.use_single_jitter,
            update_sched=update_schedule, initial_sampler=initial_sampler)
        self.collider = NearFarCollider(near_plane=c.near_plane, far_plane=c.far_plane)
        if c.background_color not in ("black", "last_sample"):
            # the fused final level composites onto black and `get_loss_dict` does not blend a background into the
            # targets (renderers.py:174-197); PreSight's configs all use black.  ("last_sample" equals black for the loss.)
            raise NotImplementedError(f"background_color={c.background_color!r}: the model driver renders onto black only "
                                      "(use RGBRenderer directly for white / random backgrounds)")
        self.renderer_rgb = RGBRenderer(background_color=c.background_color)
        self.renderer_accumulation = AccumulationRenderer()
        self.renderer_depth = DepthRenderer(method="threshold")
        self.renderer_expected_depth = DepthRenderer(method="expected")
        if c.use_sky_model:
            self.sky_model = SkyFieldMS([SkyField(mlp_num_layers=c.num_sky_mlp_layers, mlp_layer_width=c.sky_mlp_dims,
                                                  appearance_embedding_dim=app_dim, use_semantics=c.use_semantics,
                                                  semantic_dim=c.semantic_dim, implementation=c.implementation)
                                         for _ in aabbs], centroids)

    def train(self, mode: bool = True):
        super().train(mode)
        self.collider.training = mode
        return self

    def get_param_groups(self) -> Dict[str, List[nn.Parameter]]:
        """nerfacto_nusc_ms.py:385-398."""
        groups = {"proposal_networks": list(self.proposal_networks.parameters()), "fields": list(self.field.parameters())}
        for name in ("appearance_embedding", "video_embedding", "sky_model"):
            if hasattr(self, name):
                groups["fields"] += list(getattr(self, name).parameters())
        return groups

    def set_step(self, step: int) -> None:
        """What the reference's BEFORE_TRAIN_ITERATION callback does (nerfacto_nusc_ms.py:425-434): remember the step (it
        drives the line-of-sight schedules) and anneal the proposal weights (mip-NeRF 360 eq. 18)."""
        c = self.config
        self.step = int(step)
        if c.use_proposal_weight_anneal:
            train_frac = float(np.clip(step / c.proposal_weights_anneal_max_num_iters, 0, 1))
            b = c.proposal_weights_anneal_slope
            self.proposal_sampler.set_anneal(b * train_frac / ((b - 1) * train_frac + 1))

    def get_training_callbacks(self, training_callback_attributes=None) -> List[TrainingCallback]:
        """nerfacto_nusc_ms.py:405-450: with proposal-weight annealing on (the default) the trainer must run `set_step`
        before and `proposal_sampler.step_cb` after every iteration — the latter drives the proposal networks' update
        schedule; without these calls every step is an "update" step with anneal 1 and frozen line-of-sight schedules."""
        callbacks: List[TrainingCallback] = []
        if self.config.use_proposal_weight_anneal:
            callbacks.append(TrainingCallback([TrainingCallbackLocation.BEFORE_TRAIN_ITERATION],
                                              lambda step: self.set_step(step), 1))
            callbacks.append(TrainingCallback([TrainingCallbackLocation.AFTER_TRAIN_ITERATION],
                                              lambda step: self.proposal_sampler.step_cb(step), 1))
        return callbacks

    # ------------------------------------------------------------------------------------------
    def _appearance(self, ray_samples: RaySamples) -> Optional[Tensor]:
        """nerfacto_nusc_ms.py:456-490 -> per-ray embeddings [N,A] or None.  (The reference expands them to [N,S,A];
        here only the un-fused field path does, so that autograd never materialises an [N,S,A] gradient — selecting
        sample 0 of an expanded view costs a 268 MB zero-fill, an add and a reduction per step at C2 sizes.)"""
        c = self.config
        cam = ray_samples.camera_indices.squeeze(dim=-1)          # [N,1]
        N, S = ray_samples.shape
        if self.training:
            parts = []
            if c.appearance_embed_dim > 0:
                parts.append(self.appearance_embedding(cam))
            if c.video_embed_dim > 0:
                parts.append(self.video_embedding(ray_samples.metadata[VIDEO_ID].squeeze(dim=-1)))
            emb = torch.cat(parts, dim=-1)[:, 0, :] if parts else None
        else:
            dim = c.appearance_embed_dim + c.video_embed_dim
            if dim == 0:
                emb = None
            elif c.use_average_appearance_embedding:
                parts = []
                if c.appearance_embed_dim > 0:
                    parts.append(self.appearance_embedding.mean(dim=0))
                if c.video_embed_dim > 0:
                    parts.append(self.video_embedding.mean(dim=0))
                emb = torch.cat(parts, dim=-1)[None, :].expand(N, dim)
            else:
                emb = torch.zeros((N, dim), device=cam.device)
        return emb

    def forward(self, ray_bundle: RayBundle, jitters: Optional[List[Tensor]] = None,
                appearance: Optional[Tensor] = None) -> Dict[str, object]:
        """Model.forward (models/base_model.py:131-142): collider, then get_outputs."""
        return self.get_outputs(self.collider(ray_bundle), jitters, appearance)

    def get_outputs(self, ray_bundle: RayBundle, jitters: Optional[List[Tensor]] = None,
                    appearance: Optional[Tensor] = None) -> Dict[str, object]:
        """nerfacto_nusc_ms.py:452-546.  `jitters` (per-level [N,1] uniforms) and `appearance` ([N,A], already
        looked-up embeddings) are optional injection points so parity runs can share randomness and inputs."""
        ops.clear_grad_events()          # cross-stream gradient hand-offs never outlive the step that published them
        ray_samples, weights_list, ray_samples_list = self.proposal_sampler(ray_bundle, density_fns=self.density_fns,
                                                                            jitters=jitters)
        N, S = ray_samples.shape
        app = self._appearance(ray_samples) if appearance is None else appearance          # [N,A] per ray
        eu = ray_samples.frustums.eu_bins
        if self.use_fused and self.field.supports_fused():
            # level-fused fast path (presight_b200/fused.py): field + compositing as one autograd node
            weights, rgb, acc_raw, dexp_raw, depth, sem_out, tmm = self.field.fused_level(
                ray_bundle.origins, ray_bundle.directions, eu, app, 0.5)
        else:
            fo = self.field.forward(ray_samples, appearance_embedding=None if app is None
                                    else app[:, None, :].expand(N, S, -1))
            sem = fo.get(FieldHeadNames.SEMANTICS)
            # one-pass compositing kernel: weights + rgb + accumulation + both depths + semantics (:503-511, :530)
            w, rgb, acc_raw, dexp_raw, depth, sem_out, tmm = ops.composite(
                eu, fo[FieldHeadNames.DENSITY].reshape(N, S), fo[FieldHeadNames.RGB], sem, 0.5)
            weights = w.view(N, S, 1)
        weights_list.append(weights)
        ray_samples_list.append(ray_samples)
        expected_depth = torch.clip(dexp_raw, tmm[0], tmm[1])            # renderers.py:379 (batch-global clip)
        sky_outputs = {}
        if self.config.use_sky_model:
            sky_outputs = self.sky_model(ray_samples, appearance_embedding=app)
        # epilogue (:512-532) as one kernel: accumulation clamp, sky colour / sky semantics behind the scene
        rgb, accumulation, semantics = ops.sky_blend(
            rgb, acc_raw, sem_out if self.config.use_semantics else None, sky_outputs.get(FieldHeadNames.RGB),
            sky_outputs.get(FieldHeadNames.SEMANTICS), clamp_rgb=not self.training)
        outputs: Dict[str, object] = {"rgb": rgb, "accumulation": accumulation, "depth": depth,
                                      "expected_depth": expected_depth}
        if self.config.use_semantics:
            outputs["semantics"] = semantics
        if self.training:
            outputs["weights_list"] = weights_list
            outputs["ray_samples_list"] = ray_samples_list
        for i in range(self.config.num_proposal_iterations):
            outputs[f"prop_depth_{i}"] = self.renderer_depth(weights=weights_list[i], ray_samples=ray_samples_list[i])
        return outputs

    step: int = 0      # training step, set by the trainer's callback (drives the line-of-sight schedules)

    def get_line_of_sight_sigma(self, step: int) -> float:
        """nerfacto_nusc_ms.py:387-396."""
        c = self.config
        frac = float(np.clip((step - c.line_of_sight_start_step) / (c.line_of_sight_end_step - c.line_of_sight_start_step),
                             0.0, 1.0))
        return c.line_of_sight_max_sigma - frac * (c.line_of_sight_max_sigma - c.line_of_sight_min_sigma)

    def get_line_of_sight_mult(self, step: int) -> float:
        """nerfacto_nusc_ms.py:398-403."""
        c = self.config
        if step <= c.line_of_sight_start_step:
            return 0.0
        return c.line_of_sight_mult / (2.0 ** (step // c.line_of_sight_decay_steps))

    @staticmethod
    def _pose_scale_factor(ray_samples: RaySamples, batch: Dict[str, Tensor]):
        """nerfacto_nusc_ms.py:584: the reference reads `ray_samples.metadata["pose_scale_factor"][0, 0, 0]`; a batch entry
        of the same name is accepted too.  Missing from both is an error (depth units would silently be wrong).  A CUDA
        tensor is handed to the kernel as it is and read on the device."""
        md = getattr(ray_samples, "metadata", None) or {}
        v = md.get("pose_scale_factor", batch.get("pose_scale_factor"))
        if v is None:
            raise KeyError("depth supervision needs `pose_scale_factor` in ray_samples.metadata (as the reference's "
                           "datamanager provides) or in the batch")
        return v if (torch.is_tensor(v) and v.is_cuda) else float(v.reshape(-1)[0] if torch.is_tensor(v) else v)

    def get_loss_dict(self, outputs: Dict[str, object], batch: Dict[str, Tensor]) -> Dict[str, Tensor]:
        """nerfacto_nusc_ms.py:558-645, every term on a kernel: `ps_render_losses` for the three rendered-output terms
        (rgb, sky, semantic), `ps_depth_losses` for the depth supervision (expected depth + line of sight),
        `ps_zaa_interlevel_loss` / `ps_interlevel_loss` per proposal level, `ps_distortion_loss`.
        batch: "rgb" [N,3], "sky" [N,1] (1 = sky), "features" [N,C], "depth" [N] (metres)."""
        from . import losses
        c = self.config
        use_sky = c.use_sky_model and "sky" in batch
        use_sem = c.use_semantics and "features" in batch
        terms = losses.render_losses(outputs, batch, use_sky, use_sem)
        loss_dict = {"rgb_loss": terms[0]}
        if use_sky:
            loss_dict["sky_loss"] = c.sky_loss_mult * terms[1]
        if use_sem:
            loss_dict["semantic_loss"] = c.semantic_loss_mult * terms[2]
        if (c.use_monodepth_loss or c.use_lidar_loss) and "depth" in batch:
            # :577-629 — both terms and both gradients in ONE kernel (ps_depth_losses).  Branch order as in the reference:
            # the mono-depth branch runs first and the LiDAR branch, when both are enabled, overwrites its entries.
            last = outputs["ray_samples_list"][-1]
            scale = self._pose_scale_factor(last, batch)
            sigma, mult = self.get_line_of_sight_sigma(self.step), self.get_line_of_sight_mult(self.step)
            lidar = c.use_lidar_loss
            terms_d = losses.depth_supervision_losses(
                outputs["weights_list"][-1], outputs["expected_depth"], batch["depth"].view(-1, 1),
                None if lidar else batch["sky"].view(-1, 1), scale, sigma,
                c.lidar_depth_upperbound if lidar else c.monodepth_depth_upperbound,
                inverse=(not lidar) and c.monodepth_loss_inverse, eu_bins=last.frustums.eu_bins)
            loss_dict["expected_depth_loss"] = c.expected_depth_loss_mult * terms_d[0]
            loss_dict["line_of_sight_loss"] = mult * terms_d[1]
        if self.training:
            wl = outputs["weights_list"]
            sp = [rs.sp_bins for rs in outputs["ray_samples_list"]]
            if c.enable_z_anti_aliasing:
                il = losses.z_anti_aliasing_interlevel_loss(wl, sp, c.pulse_width)
            else:
                il = losses.interlevel_loss(wl, sp)
            loss_dict["interlevel_loss"] = c.interlevel_loss_mult * il
            loss_dict["distortion_loss"] = c.distortion_loss_mult * losses.distortion_loss(wl, sp)
        return loss_dict

    def get_depth(self, ray_bundle: RayBundle, threshold: float = 0.5) -> Dict[str, object]:
        """nerfacto_nusc_ms.py:688-708."""
        ray_bundle = self.collider(ray_bundle)
        ray_samples, weights_list, ray_samples_list = self.proposal_sampler(ray_bundle, density_fns=self.density_fns)
        density, _ = self.field.get_density(ray_samples)
        N, S = ray_samples.shape
        w, _, _, dexp_raw, depth, _, tmm = ops.composite(ray_samples.frustums.eu_bins, density.reshape(N, S), None, None,
                                                         threshold)
        outputs: Dict[str, object] = {"depth": depth, "expected_depth": torch.clip(dexp_raw, tmm[0], tmm[1])}
        if self.training:
            outputs["weights_list"] = weights_list
            outputs["ray_samples_list"] = ray_samples_list
        return outputs

    @torch.no_grad()
    def get_surface_hits(self, ray_bundle: RayBundle, threshold: float = 0.5) -> Dict[str, Tensor]:
        """The threshold depth of `get_depth` for prior extraction (scripts/extract_priors.py:100-113) -> {"depth": [N,1]}.
        Same collider and proposal sampling as `get_depth`; the final level runs on the fused density kernels
        (iNGPFieldMS.level_depth) when the field fits them, else exactly `get_depth`'s computation."""
        ray_bundle = self.collider(ray_bundle)
        ray_samples, _, _ = self.proposal_sampler(ray_bundle, density_fns=self.density_fns)
        N, S = ray_samples.shape
        eu = ray_samples.frustums.eu_bins
        if self.use_fused and self.field.supports_level_depth(S):
            return {"depth": self.field.level_depth(ray_bundle.origins, ray_bundle.directions, eu, threshold)}
        density, _ = self.field.get_density(ray_samples)
        _, _, _, _, depth, _, _ = ops.composite(eu, density.reshape(N, S), None, None, threshold)
        return {"depth": depth}

    @torch.no_grad()
    def get_depth_for_camera_ray_bundle(self, camera_ray_bundle: RayBundle, threshold: float = 0.5) -> Dict[str, Tensor]:
        """nerfacto_nusc_ms.py:710-734: chunked evaluation."""
        chunk = self.config.eval_num_rays_per_chunk
        n = len(camera_ray_bundle)
        lists: Dict[str, List[Tensor]] = {}
        for i in range(0, n, chunk):
            rb = RayBundle(origins=camera_ray_bundle.origins[i:i + chunk], directions=camera_ray_bundle.directions[i:i + chunk],
                           camera_indices=None if camera_ray_bundle.camera_indices is None
                           else camera_ray_bundle.camera_indices[i:i + chunk])
            for k, v in self.get_depth(rb, threshold).items():
                if torch.is_tensor(v):
                    lists.setdefault(k, []).append(v)
        return {k: torch.cat(v) for k, v in lists.items()}

    @torch.no_grad()
    def get_outputs_for_camera_ray_bundle(self, camera_ray_bundle: RayBundle) -> Dict[str, Tensor]:
        """nerfstudio's Model.get_outputs_for_camera_ray_bundle (models/base_model.py): a bundle whose fields are
        [H,W,.] is flattened row-major and rendered by `forward` in consecutive slices of `eval_num_rays_per_chunk` rays;
        the tensor outputs are concatenated and viewed as [H,W,-1].  Per-chunk statistics stay per chunk as in the
        reference: `expected_depth` is clipped to its own chunk's min / max (renderers.py:379)."""
        H, W = camera_ray_bundle.origins.shape[:2]
        n = H * W
        names = ("origins", "directions", "pixel_area", "camera_indices", "nears", "fars", "times")
        flat = {k: getattr(camera_ray_bundle, k) for k in names}
        flat = {k: None if v is None else v.reshape(n, -1) for k, v in flat.items()}
        metadata = {k: v.reshape(n, -1) for k, v in camera_ray_bundle.metadata.items()}
        chunk = self.config.eval_num_rays_per_chunk
        lists: Dict[str, List[Tensor]] = {}
        for i in range(0, n, chunk):
            s = slice(i, i + chunk)
            chunk_rb = RayBundle(**{k: None if v is None else v[s] for k, v in flat.items()},
                                 metadata={k: v[s] for k, v in metadata.items()})
            for k, v in self.forward(chunk_rb).items():
                if torch.is_tensor(v):
                    lists.setdefault(k, []).append(v)
        return {k: torch.cat(v).view(H, W, -1) for k, v in lists.items()}

    def get_metrics_dict(self, outputs: Dict[str, object], batch: Dict[str, Tensor]) -> Dict[str, Tensor]:
        """nerfacto's get_metrics_dict: {"psnr": PSNR of the ray batch's rgb against batch["rgb"]}, a CUDA scalar (no host
        read, so the training step stays free of synchronisations)."""
        from . import metrics
        return {"psnr": metrics.psnr(outputs["rgb"], batch["rgb"])}

    def get_image_metrics_and_images(self, outputs: Dict[str, Tensor], batch: Dict[str, Tensor]
                                     ) -> Tuple[Dict[str, float], Dict[str, Tensor]]:
        """nerfacto's get_image_metrics_and_images for one rendered image: outputs of `get_outputs_for_camera_ray_bundle`,
        batch["rgb"] [H,W,3] in [0,1] -> ({"psnr", "ssim"} as floats, and "lpips" when `self.lpips` is set; {"img": gt and
        prediction side by side [H,2W,3], "accumulation", "depth"}).  One host read for the numbers.  LPIPS scores the
        render clamped to [0,1], as the reference does.  With `self.colormap` unset the images are raw [H,W,1]; with it
        set they are the reference's colormapped [H,W,3] images, `prop_depth_{i}` of every proposal iteration included,
        all from one `ps_colormap` call (`metrics.colormap_images`).
        When the batch holds a LiDAR depth image "depth" ([H,W] or [H,W,1], metres, 0 = no return), the numbers also
        hold `depth_{m}` and `expected_depth_{m}` for m in abs_rel, sq_rel, rmse, rmse_log, a1, a2, a3: the depth errors
        of the "depth" and "expected_depth" outputs (`geometry.depth_metrics` with 1 m < target <
        `lidar_depth_upperbound`, NaN without a valid pixel).  They need `pose_scale_factor` in the batch (KeyError
        otherwise)."""
        from . import metrics
        gt, pred = batch["rgb"].to(outputs["rgb"].device), outputs["rgb"]
        psnr, ssim, _ = metrics.image_metrics(pred, gt)
        vals = [psnr[0].double(), ssim[0]]
        if self.lpips is not None:
            vals.append(self.lpips(pred.clamp(0.0, 1.0), gt))
        depth_names = []
        if "depth" in batch:
            from . import geometry
            names = [n for n in geometry.DEPTH_METRICS if n != "n_valid"]
            dm = geometry.depth_metrics([outputs["depth"], outputs["expected_depth"]],
                                        batch["depth"].to(pred.device), self._pose_scale_factor(None, batch),
                                        1.0, self.config.lidar_depth_upperbound)
            depth_names = [f"{p}_{n}" for p in ("depth", "expected_depth") for n in names]
            vals.extend(dm[:, :len(names)].reshape(-1))
        images_dict = {"img": torch.cat([gt, pred], dim=1), "accumulation": outputs["accumulation"],
                       "depth": outputs["depth"]}
        if self.colormap is not None:
            props = [f"prop_depth_{i}" for i in range(self.config.num_proposal_iterations)]
            acc_img, depth_imgs = metrics.colormap_images([outputs["depth"]] + [outputs[k] for k in props],
                                                          outputs["accumulation"], self.colormap)
            images_dict.update({"accumulation": acc_img, "depth": depth_imgs[0]}, **dict(zip(props, depth_imgs[1:])))
        vals = torch.stack(vals).tolist()
        metrics_dict = {"psnr": float(vals[0]), "ssim": float(vals[1])}
        if self.lpips is not None:
            metrics_dict["lpips"] = float(vals[2])
        metrics_dict.update(zip(depth_names, (float(v) for v in vals[len(vals) - len(depth_names):])))
        return metrics_dict, images_dict

    @torch.no_grad()
    def query_priors(self, points_scaled: Tensor) -> Tuple[Tensor, Tensor]:
        """scripts/extract_priors.py:130-138: mean density over proposal nets + field, clipped fp16 semantics."""
        if self.use_fused and len(self.field.fields) == 1 and self.field.supports_fused() and self.config.use_semantics:
            from . import fused
            return fused.query_priors(points_scaled, [p.fields[0] for p in self.proposal_networks],
                                      self.field.fields[0])
        if (self.use_fused and len(self.field.fields) > 1 and self.config.use_semantics and self.field.supports_fused()
                and all(p.supports_fused() for p in self.proposal_networks)):
            from . import fused
            return fused.query_priors_ms(points_scaled, list(self.proposal_networks), self.field)
        dens = [p.density_fn(points_scaled).squeeze(-1) for p in self.proposal_networks]
        dens.append(self.field.density_fn(points_scaled)[0].squeeze(-1))
        densities_mean = torch.stack(dens, dim=0).mean(dim=0)
        feats = self.field.semantic_fn(points_scaled).clip(0.0, 1.0).to(torch.float16)
        return densities_mean, feats
