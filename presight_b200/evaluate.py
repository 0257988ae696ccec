"""The evaluation-split loop of the reference pipeline: `VanillaPipeline.get_average_eval_image_metrics`
(nerfstudio pipelines/base_pipeline.py) for `NerfactoNuscMSModel`, with the camera rays built on the device by
`RayGenerator.image_rays` instead of the eval dataloader.  Writing the images to disk is not part of it."""
from __future__ import annotations

import time
from typing import Dict, Iterable, Tuple, Union

import torch
from torch import Tensor


def average_eval_image_metrics(model, ray_generator,
                               frames: Iterable[Union[Tuple[int, Tensor], Tuple[int, Tensor, Tensor]]],
                               get_std: bool = False, pose_scale_factor=None) -> Dict[str, float]:
    """frames: (camera_index, image [H,W,3] in [0,1]) per evaluation image, or (camera_index, image, depth_m) with a
    LiDAR depth image [H,W] or [H,W,1] in metres (0 = no return), which adds the depth keys of
    `get_image_metrics_and_images` (`depth_abs_rel` ... `expected_depth_a3`) to the averages; `pose_scale_factor`, when
    given, goes into every frame's batch (the depth keys need it).  Every frame must have the same form.  Each image is
    rendered (`ray_generator.image_rays` + `model.get_outputs_for_camera_ray_bundle`) and scored
    (`model.get_image_metrics_and_images`, "lpips" included when `model.lpips` is set); each frame's dict gains
    `num_rays_per_sec` = H W / wall time and `fps` = num_rays_per_sec / (H W).  The wall time is the host clock around
    ray generation, render and metrics, which the metrics' one host read closes.  Returns the mean of every key over the
    frames, as the reference computes it (a float32 tensor of the per-frame values), and with `get_std` also
    `{key}_std`, the unbiased standard deviation of `torch.std_mean`.  The model runs in eval mode; its previous mode
    is restored on return and on error."""
    was_training = model.training
    model.eval()
    try:
        per_frame = []
        for frame in frames:
            camera_index, image = frame[0], frame[1]
            batch = {"rgb": image}
            if len(frame) == 3:
                batch["depth"] = frame[2]
            elif len(frame) != 2:
                raise ValueError(f"average_eval_image_metrics: a frame is (camera_index, image[, depth_m]), got "
                                 f"{len(frame)} items")
            if pose_scale_factor is not None:
                batch["pose_scale_factor"] = pose_scale_factor
            H, W = int(image.shape[0]), int(image.shape[1])
            start = time.perf_counter()
            outputs = model.get_outputs_for_camera_ray_bundle(ray_generator.image_rays(camera_index, H, W))
            metrics_dict, _ = model.get_image_metrics_and_images(outputs, batch)
            metrics_dict["num_rays_per_sec"] = H * W / (time.perf_counter() - start)
            metrics_dict["fps"] = metrics_dict["num_rays_per_sec"] / (H * W)
            per_frame.append(metrics_dict)
    finally:
        model.train(was_training)
    if not per_frame:
        raise ValueError("average_eval_image_metrics: no frames")
    if any(m.keys() != per_frame[0].keys() for m in per_frame):
        raise ValueError("average_eval_image_metrics: frames with and without depth cannot be averaged together")
    out: Dict[str, float] = {}
    for key in per_frame[0]:
        vals = torch.tensor([m[key] for m in per_frame])
        if get_std:
            std, mean = torch.std_mean(vals)
            out[key], out[f"{key}_std"] = float(mean), float(std)
        else:
            out[key] = float(torch.mean(vals))
    return out
