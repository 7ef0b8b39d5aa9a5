"""Config-override module in the reference's own "python globals" style (reference experiments/basic_conf.py and
train.py:97-107): pass it to `--conf-overwrites` to rebind the generator / critic / optimizer factories to the
B200-native implementations.  Values mirror basic_conf.py:22-68."""
from functools import partial

import numpy as np
import torch
from torch.optim.lr_scheduler import MultiStepLR

from ..data.augment import SpatialTransform2
from ..data.Scaler import FactorZeroCenterScaler
from ..model.discriminator import PatchGANDiscriminator
from ..model.generator import ResnetGenerator
from ..optim import FusedAdam

lr = 2e-4
betas = (5e-1, 0.999)
milestones = [6000, 8000]
lr_gamma = 0.1
weight_clip = 0.01
max_HU_delta = 600
desired_HU_bounds = (350, 450)
HU_norm_range = (-1024, 1500)
scaler = FactorZeroCenterScaler(*HU_norm_range, max_HU_delta)

compute_dtype = torch.bfloat16

generator_args = {"n_resnet_blocks": 4, "n_updownsample_blocks": 2, "init_channels_out": 16}
generator_class = partial(ResnetGenerator, **generator_args, compute_dtype=compute_dtype)
generator_optim_class = partial(FusedAdam, lr=lr, betas=betas)
generator_lr_scheduler_class = partial(MultiStepLR, milestones=milestones, gamma=lr_gamma)

critic_args = {"channels_in": 1, "init_channels_out": 8, "discriminator_depth": 3, "negative_slope": 0.2}
critic_class = partial(PatchGANDiscriminator, **critic_args, compute_dtype=compute_dtype)
critic_optim_class = partial(FusedAdam, lr=lr, betas=betas)
critic_lr_scheduler_class = partial(MultiStepLR, milestones=milestones, gamma=lr_gamma)

# Training augmentation: batchgenerators SpatialTransform_2 of basic_conf.py:88-106 on the device, with the values
# SURVEY §3.4 records (elastic p=0.1, scale 0.7-1.4 p=0.2, rotation ±30° p=0.2, taken here as all three axes).  The
# arguments it does not record (patch_center_dist_from_border, deformation_scale, border modes and orders, random_crop)
# stay at upstream's defaults.  Pass it as DevicePatchSampler(..., transform=train_transform); validation sampling stays
# untransformed.
patch_size = (128, 128, 128)
train_transform = SpatialTransform2(
    patch_size, do_elastic_deform=True, p_el_per_sample=0.1, do_scale=True, scale=(0.7, 1.4), p_scale_per_sample=0.2,
    do_rotation=True, angle_x=(-np.pi / 6, np.pi / 6), angle_y=(-np.pi / 6, np.pi / 6), angle_z=(-np.pi / 6, np.pi / 6),
    p_rot_per_sample=0.2)
