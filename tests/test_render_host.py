"""CPU checks of whole-image rendering: the row-major chunking of `get_outputs_for_camera_ray_bundle` (with `forward`
replaced by a recorder) and the synthetic cameras `make_cameras` against the rays `make_rays` draws from them."""
import dataclasses
import math

import torch

from presight_b200 import synthetic
from presight_b200.cameras.rays import RayBundle
from presight_b200.model import NerfactoNuscMSModel


def small_model(chunk):
    cfg = synthetic.config_c2()
    cfg = dataclasses.replace(cfg, log2_hashmap_size=12, eval_num_rays_per_chunk=chunk,
                              proposal_net_args_list=[dict(a, log2_hashmap_size=12) for a in cfg.proposal_net_args_list])
    return NerfactoNuscMSModel(cfg, torch.zeros(1, 3), synthetic.tile_aabb())


def test_camera_ray_bundle_chunks_are_consecutive_row_major_slices():
    model = small_model(100)
    calls = []

    def forward(rb):
        calls.append(rb)
        return {"rgb": rb.origins * 2, "cam": rb.camera_indices.float(), "not_a_tensor": 3}
    model.forward = forward
    H, W = 13, 17                                            # 221 rays: chunks of 100, 100, 21
    g = torch.Generator().manual_seed(0)
    o = torch.rand(H, W, 3, generator=g)
    cam = torch.arange(H * W).view(H, W, 1)
    norm = torch.rand(H, W, 1, generator=g)
    out = model.get_outputs_for_camera_ray_bundle(RayBundle(origins=o, directions=o, camera_indices=cam,
                                                            metadata={"directions_norm": norm}))
    assert [len(rb) for rb in calls] == [100, 100, 21]
    flat = cam.view(-1)
    for i, rb in enumerate(calls):
        assert torch.equal(rb.camera_indices.view(-1), flat[100 * i:100 * i + len(rb)])
        assert torch.equal(rb.metadata["directions_norm"].view(-1), norm.view(-1)[100 * i:100 * i + len(rb)])
        assert rb.pixel_area is None
    assert set(out) == {"rgb", "cam"}
    assert torch.equal(out["rgb"], o * 2) and torch.equal(out["cam"].long(), cam)


def test_make_cameras_reproduce_make_rays():
    n, seed, frames = 2000, 5, 30
    rays = synthetic.make_rays(n, seed=seed, n_frames=frames)
    cams = synthetic.make_cameras(seed=seed, n_frames=frames)
    assert cams["camera_to_worlds"].shape == (6 * frames, 3, 4) and (cams["H"], cams["W"]) == (900, 1600)
    # make_rays' continuous pixel of every ray, from the same generator draws
    g = torch.Generator().manual_seed(seed)
    torch.randn(frames, 2, generator=g), torch.randn(frames, generator=g)
    torch.randint(0, frames, (n,), generator=g), torch.randint(0, 6, (n,), generator=g)
    u = torch.rand(n, generator=g) * synthetic.W
    v = torch.rand(n, generator=g) * synthetic.H
    c2w = cams["camera_to_worlds"][rays["camera_indices"][:, 0]]
    i = rays["camera_indices"][:, 0]
    d_cam = torch.stack([(u - cams["cx"][i]) / cams["fx"][i], -(v - cams["cy"][i]) / cams["fy"][i], -torch.ones(n)], -1)
    d = (c2w[:, :, :3] @ d_cam[:, :, None])[..., 0]
    d = d / d.norm(dim=-1, keepdim=True)
    assert float((d - rays["directions"]).abs().max()) <= 1e-6
    assert torch.equal(c2w[:, :, 3], rays["origins"])
    r = cams["camera_to_worlds"][:, :, :3]
    assert float((r.transpose(1, 2) @ r - torch.eye(3)).abs().max()) <= 1e-6     # rotations
    assert math.isclose(float(torch.det(r[0])), 1.0, abs_tol=1e-6)
