"""SR3 noise-prediction UNet -- drop-in for the reference's models/diffusion_models/sr3/unet.py:7-124 (SURVEY.md 8f N1).

The plain conditional UNet of the family: ``forward(x, time)`` with ``x = cat([condition, x_t], 1)`` goes straight into
the stem convolution; no FD splitter, no HF-guided cross attention, ONE mid block without attention (:77-81).  Same
constructor signature and state_dict keys (347 tensors for the canonical config); runs through ``UNetPlan`` (kind 'sr3').
"""
from torch import nn

from ..nn_modules.functional_layers import Swish
from ..resdiff.unet import PlannedUNet, build_unet_body, noise_level_mlp


class UNet(PlannedUNet):
    def __init__(self, in_channel=6, out_channel=3, inner_channel=32, norm_groups=32, channel_mults=(1, 2, 4, 8, 8),
                 attn_res=(8,), res_blocks=3, dropout=0, with_noise_level_emb=True, image_width=128, image_height=128,
                 image_channels=3, precision="bf16"):
        super().__init__()
        if not with_noise_level_emb:
            raise NotImplementedError("with_noise_level_emb=False is never used on the reference's path")
        if in_channel != 2 * image_channels:
            raise AssertionError("SR3 consumes cat([condition, x_t]): in_channel must be 2 * image_channels")
        self.noise_level_mlp = noise_level_mlp(inner_channel, Swish())
        self.image_channels = image_channels
        self.image_height, self.image_width = image_height, image_width
        self.inner_channel, self.norm_groups, self.dropout = inner_channel, norm_groups, dropout
        build_unet_body(self, in_channel, out_channel, inner_channel, norm_groups, channel_mults, attn_res, res_blocks,
                        dropout, inner_channel, image_height, mid_attn=(False,))
        self.precision = precision
        self.time_act = "swish"
