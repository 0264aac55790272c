"""SRDiff (RRDB-conditioned) UNet -- drop-in for the reference's models/diffusion_models/srdiff/unet.py:6-141.
``forward((rrdb_features, x_t), time)``: 18 feature maps (B,64,H/4,W/4); features [2::3] are concatenated,
projected by ConvTranspose2d(384->64, k8, s4, p2) (hoisted: condition-only) and added after ``downs[2]``."""
import torch
from torch import nn

from ..nn_modules.functional_layers import Mish
from ..resdiff.unet import PlannedUNet, build_unet_body, noise_level_mlp


class UNet(PlannedUNet):
    def __init__(self, in_channel=9, out_channel=3, inner_channel=32, norm_groups=32, channel_mults=(1, 2, 4, 8, 8),
                 attn_res=(8,), res_blocks=3, dropout=0, with_noise_level_emb=True, image_width=128, image_height=128,
                 image_channels=1, precision="bf16"):
        super().__init__()
        if not with_noise_level_emb:
            raise NotImplementedError("with_noise_level_emb=False is never used on the reference's path")
        self.hidden_size = 64
        self.num_block = 17
        self.cond_proj = nn.ConvTranspose2d(self.hidden_size * ((self.num_block + 1) // 3), self.hidden_size, 8, 4, 2)
        self.noise_level_mlp = noise_level_mlp(inner_channel, Mish())
        self.image_channels = image_channels
        self.image_height, self.image_width = image_height, image_width
        self.inner_channel, self.norm_groups, self.dropout = inner_channel, norm_groups, dropout
        build_unet_body(self, in_channel, out_channel, inner_channel, norm_groups, channel_mults, attn_res, res_blocks,
                        dropout, inner_channel, image_height)
        self.precision = precision
        self.time_act = "mish"

    def _split(self, x):
        """x = (rrdb_features, x_t): the condition is cat(features[2::3], 1), or -- joint training with a trainable encoder --
        that concatenation already made by ``RRDBNet.forward_joint`` as one differentiable tensor."""
        feas, x_t = x
        return (feas if torch.is_tensor(feas) else torch.cat(list(feas[2::3]), dim=1)), x_t
