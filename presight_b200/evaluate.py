"""The evaluation-split loop of the reference pipeline: `VanillaPipeline.get_average_eval_image_metrics`
(nerfstudio pipelines/base_pipeline.py) for `NerfactoNuscMSModel`, with the camera rays built on the device by
`RayGenerator.image_rays` instead of the eval dataloader.  Writing the images to disk is not part of it."""
from __future__ import annotations

import time
from typing import Dict, Iterable, Tuple

import torch
from torch import Tensor


def average_eval_image_metrics(model, ray_generator, frames: Iterable[Tuple[int, Tensor]],
                               get_std: bool = False) -> Dict[str, float]:
    """frames: (camera_index, image [H,W,3] in [0,1]) per evaluation image.  Each image is rendered
    (`ray_generator.image_rays` + `model.get_outputs_for_camera_ray_bundle`) and scored
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
        for camera_index, image in frames:
            H, W = int(image.shape[0]), int(image.shape[1])
            start = time.perf_counter()
            outputs = model.get_outputs_for_camera_ray_bundle(ray_generator.image_rays(camera_index, H, W))
            metrics_dict, _ = model.get_image_metrics_and_images(outputs, {"rgb": image})
            metrics_dict["num_rays_per_sec"] = H * W / (time.perf_counter() - start)
            metrics_dict["fps"] = metrics_dict["num_rays_per_sec"] / (H * W)
            per_frame.append(metrics_dict)
    finally:
        model.train(was_training)
    if not per_frame:
        raise ValueError("average_eval_image_metrics: no frames")
    out: Dict[str, float] = {}
    for key in per_frame[0]:
        vals = torch.tensor([m[key] for m in per_frame])
        if get_std:
            std, mean = torch.std_mean(vals)
            out[key], out[f"{key}_std"] = float(mean), float(std)
        else:
            out[key] = float(torch.mean(vals))
    return out
