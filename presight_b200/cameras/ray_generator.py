"""RayGenerator (reference: nerfstudio/model_components/ray_generators.py:25-61 on top of
nerfstudio/cameras/cameras.py:497-880) for PreSight's cameras — PERSPECTIVE, no distortion parameters, camera optimizer
off — on `ps_generate_rays`: (camera, row, col) indices in, a RayBundle out, one kernel."""
from __future__ import annotations

from typing import Optional

import torch
from torch import Tensor, nn

from .._lib import call, ptr, stream
from .rays import RayBundle


class RayGenerator(nn.Module):
    def __init__(self, camera_to_worlds: Tensor, fx: Tensor, fy: Tensor, cx: Tensor, cy: Tensor,
                 pixel_offset: float = 0.5) -> None:
        """camera_to_worlds [C,3,4]; fx, fy, cx, cy [C] (or [C,1]) — the tensors a `Cameras` object holds."""
        super().__init__()
        C = camera_to_worlds.shape[0]
        if camera_to_worlds.shape != (C, 3, 4):
            raise ValueError(f"camera_to_worlds must be [C,3,4], got {tuple(camera_to_worlds.shape)}")
        self.register_buffer("camera_to_worlds", camera_to_worlds.detach().float().contiguous(), persistent=False)
        for name, t in (("fx", fx), ("fy", fy), ("cx", cx), ("cy", cy)):
            t = torch.as_tensor(t, dtype=torch.float32).reshape(-1)
            if t.numel() == 1:
                t = t.expand(C)
            if t.numel() != C:
                raise ValueError(f"{name} must have one entry per camera")
            self.register_buffer(name, t.contiguous().clone(), persistent=False)
        self.pixel_offset = float(pixel_offset)
        self.validate_indices = True

    def forward(self, ray_indices: Tensor, camera_opt_to_camera: Optional[Tensor] = None) -> RayBundle:
        """ray_indices [N,3] int64 = (camera, row, col) -> RayBundle (origins, unit directions, pixel_area [N,1],
        camera_indices [N,1], metadata["directions_norm"] [N,1])."""
        if camera_opt_to_camera is not None:
            raise NotImplementedError("pose optimisation is off in PreSight's configs; only the identity is supported")
        assert ray_indices.dim() == 2 and ray_indices.shape[1] == 3, "ray_indices must be [N,3]"
        idx = ray_indices.to(torch.int64).contiguous()
        N, dev = idx.shape[0], self.camera_to_worlds.device
        if self.validate_indices and N:
            # the reference's gather raises on a bad camera index; the kernel cannot, so check on the device (an
            # asynchronous assert: no host sync, the error surfaces at the next synchronisation)
            cam = idx[:, 0]
            torch._assert_async(((cam >= 0) & (cam < self.camera_to_worlds.shape[0])).all(),
                                "RayGenerator: camera index out of range")
        origins = torch.empty(N, 3, device=dev, dtype=torch.float32)
        directions = torch.empty(N, 3, device=dev, dtype=torch.float32)
        pixel_area = torch.empty(N, 1, device=dev, dtype=torch.float32)
        norm = torch.empty(N, 1, device=dev, dtype=torch.float32)
        call("ps_generate_rays", ptr(self.camera_to_worlds), ptr(self.fx), ptr(self.fy), ptr(self.cx), ptr(self.cy),
             self.camera_to_worlds.shape[0], ptr(idx), N, self.pixel_offset, ptr(origins), ptr(directions),
             ptr(pixel_area), ptr(norm), stream())
        return RayBundle(origins=origins, directions=directions, pixel_area=pixel_area, camera_indices=idx[:, :1],
                         metadata={"directions_norm": norm})

    def image_rays(self, camera_index: int, H: int, W: int) -> RayBundle:
        """Every pixel of one H x W camera image -> a RayBundle whose fields are [H,W,.] (camera_indices included), as
        `Cameras.generate_rays(camera_indices=i)` hands it to `get_outputs_for_camera_ray_bundle`.  The (camera, row, col)
        indices are built on the device in row-major order and go through `forward`."""
        dev = self.camera_to_worlds.device
        rows = torch.arange(H, device=dev, dtype=torch.int64)[:, None].expand(H, W)
        cols = torch.arange(W, device=dev, dtype=torch.int64)[None, :].expand(H, W)
        idx = torch.stack([torch.full((H, W), int(camera_index), device=dev, dtype=torch.int64), rows, cols], dim=-1)
        rb = self.forward(idx.view(H * W, 3))

        def img(t: Tensor) -> Tensor:
            return t.view(H, W, -1)
        return RayBundle(origins=img(rb.origins), directions=img(rb.directions), pixel_area=img(rb.pixel_area),
                         camera_indices=img(rb.camera_indices), metadata={k: img(v) for k, v in rb.metadata.items()})
