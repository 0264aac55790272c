"""PhyDiff ("ResDiff+Physics") noise-prediction UNet -- drop-in for the reference's models/diffusion_models/phydiff/unet.py:
140-346 (SURVEY.md 8f N1; the architecture of the reference's README example and of 30 of its 55 configs).

ResDiff without the FD splitter: the stem sees ``cat([condition, x_t, Kx(c), Ky(c), Kxy(c)])`` where the three fixed
stencils (x / y forward differences, 5-point Laplacian) act on the REFLECT-padded condition and sum over the image channels
(:189-196, :311-314), and the HF-guided cross-attention queries are the three Haar detail bands kept apart
(``wavelet_components = 3``, :265-276).  Everything that depends only on the condition is computed once per batch
(``UNetPlan.set_condition``, kind 'phydiff').  The reference's ``PhyConv`` / ``K2M`` classes (:11-137) are never
instantiated by it and are not reproduced.  state_dict: 386 tensors for the canonical config (the stencil kernels are plain
tensors in the reference, not parameters or buffers).
"""
from torch import nn

from ..nn_modules.functional_layers import Swish
from ..resdiff.guided_cross_attention import HF_guided_CA
from ..resdiff.unet import PlannedUNet, build_unet_body, noise_level_mlp


class UNet(PlannedUNet):
    def __init__(self, in_channel=9, out_channel=3, inner_channel=32, norm_groups=32, channel_mults=(1, 2, 4, 8, 8),
                 attn_res=(8,), res_blocks=3, dropout=0, with_noise_level_emb=True, image_width=128, image_height=128,
                 image_channels=1, device='cuda', precision="bf16"):
        super().__init__()
        if not with_noise_level_emb:
            raise NotImplementedError("with_noise_level_emb=False is never used on the reference's path")
        if in_channel != 2 * image_channels + 3:
            raise AssertionError("PhyDiff's stem consumes cat([condition, x_t, 3 stencil maps]): in_channel must be 2 * image_channels + 3")
        self.noise_level_mlp = noise_level_mlp(inner_channel, Swish())
        self.image_channels = image_channels
        self.wavelet_components = 3
        self.J = 4
        self.image_height, self.image_width = image_height, image_width
        self.inner_channel, self.norm_groups, self.dropout = inner_channel, norm_groups, dropout
        self.hf_ca_list = nn.ModuleList(
            [HF_guided_CA(inner_channel * (2 ** i), image_channels=image_channels, wavelet_components=self.wavelet_components)
             for i in range(self.J)])
        build_unet_body(self, in_channel, out_channel, inner_channel, norm_groups, channel_mults, attn_res, res_blocks,
                        dropout, inner_channel, image_height)
        self.precision = precision
        self.time_act = "swish"
        del device
