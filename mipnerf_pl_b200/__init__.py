"""mipnerf_pl_b200 — B200-native (sm_100a) Mip-NeRF per-ray hot path behind the
reference's Python surface (hjxwhy/mipnerf_pl: models/mip_nerf.py, models/mip.py).

Importing the package never touches CUDA; the first op call loads
libmipnerf_b200.so and raises if it is missing (no CPU fallback).
"""
from .rays import (Rays, Rays_keys, namedtuple_map, rearrange_render_image, blender_rays, spheric_pose,
                   random_ray_batch, rays_to_torch, RayStaging)
from .mip_nerf import MLP, MipNerf
from .nerf_system import MipNeRFSystem, default_hparams, calc_psnr
from .ops import (sample_along_rays, resample_along_rays, cast_rays, integrated_pos_enc, pos_enc,
                  sorted_piecewise_constant_pdf, volumetric_rendering, distloss, philox_uniform, philox_normal)
from .weights import make_state_dict
from .train import FusedAdam, MipLRDecay, allreduce_grads, forward_backward, fused_loss, mip_lr
from .datasets import (Blender, Multicam, DeviceRayBank, Scene, dataset_dict, load_blender_scene, load_multicam_scene,
                       image_rays, convert_blender_to_multiscale, write_synthetic_blender_scene, philox_pixel_ids)
from .render import generate_rays, render_frame, render_sharded, shard_bounds, shard_rows, gather_rows
from .graph import GraphedForward, GraphedTrainStep
from .metrics import eval_errors, ssim, evaluate, render_path, spheric_path, save_images

__all__ = [
    "Rays", "Rays_keys", "namedtuple_map", "rearrange_render_image", "blender_rays", "spheric_pose",
    "random_ray_batch", "rays_to_torch", "RayStaging", "MLP", "MipNerf", "MipNeRFSystem", "default_hparams", "calc_psnr",
    "sample_along_rays", "resample_along_rays", "cast_rays", "integrated_pos_enc", "pos_enc",
    "sorted_piecewise_constant_pdf", "volumetric_rendering", "distloss", "make_state_dict", "generate_rays", "render_frame",
    "render_sharded", "shard_bounds", "shard_rows", "gather_rows", "FusedAdam", "MipLRDecay", "allreduce_grads",
    "forward_backward", "fused_loss", "mip_lr", "Blender", "Multicam", "DeviceRayBank", "Scene", "dataset_dict",
    "load_blender_scene", "load_multicam_scene", "image_rays", "convert_blender_to_multiscale",
    "write_synthetic_blender_scene", "GraphedForward", "GraphedTrainStep", "philox_pixel_ids", "philox_uniform", "philox_normal", "eval_errors", "ssim", "evaluate",
    "render_path", "spheric_path", "save_images",
]
