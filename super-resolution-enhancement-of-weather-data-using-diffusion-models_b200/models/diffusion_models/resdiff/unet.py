"""ResDiff noise-prediction UNet -- drop-in for the reference's models/diffusion_models/resdiff/unet.py:11-177.

Same constructor signature, attribute names and state_dict keys (396 tensors for the canonical config), so reference
checkpoints load unchanged.  ``forward(x, time)`` has the reference's meaning -- ``x = cat([condition, x_t], 1)``
(B, 2*C_img, H, W) fp32 NCHW, ``time`` (B, 1) continuous noise level, returns eps_hat (B, C_img, H, W) fp32 -- but runs
entirely in hand-written sm_100a kernels through ``UNetPlan``.  ``precision`` selects ``'bf16'`` (tcgen05 path,
default) or ``'fp32'`` (check mode).
"""
from torch import nn

import torch

from ....unet_plan import UNetPlan
from ..nn_modules.functional_layers import Downsample, PositionalEncoding, Swish, Upsample, default
from ..nn_modules.resnet import Block, ResnetBlocWithAttn
from .fd_info_spliter import FD_Info_Spliter
from .guided_cross_attention import HF_guided_CA


def build_unet_body(net, in_channel, out_channel, inner_channel, norm_groups, channel_mults, attn_res, res_blocks,
                    dropout, noise_level_channel, image_height, mid_attn=(True, False)):
    """Down / mid / up module lists shared by the ResDiff and SRDiff UNets (reference resdiff/unet.py:62-119,
    srdiff/unet.py:58-110).  Attention placement is keyed on the image HEIGHT, as in the reference."""
    n_levels = len(channel_mults)
    width = inner_channel
    skip_widths = [width]
    res = image_height
    downs = [nn.Conv2d(in_channel, inner_channel, kernel_size=3, padding=1)]
    for lvl, mult in enumerate(channel_mults):
        out_w = inner_channel * mult
        for _ in range(res_blocks):
            downs.append(ResnetBlocWithAttn(width, out_w, noise_level_emb_dim=noise_level_channel, norm_groups=norm_groups,
                                            dropout=dropout, with_attn=(res in attn_res)))
            width = out_w
            skip_widths.append(width)
        if lvl != n_levels - 1:
            downs.append(Downsample(width))
            skip_widths.append(width)
            res //= 2
    net.downs = nn.ModuleList(downs)
    # mid_attn: one entry per mid block (ResDiff / SRDiff / PhyDiff: attention then plain; SR3: ONE plain block, sr3/unet.py:77-81)
    net.mid = nn.ModuleList([
        ResnetBlocWithAttn(width, width, noise_level_emb_dim=noise_level_channel, norm_groups=norm_groups, dropout=dropout, with_attn=a)
        for a in mid_attn])
    ups = []
    for lvl in reversed(range(n_levels)):
        out_w = inner_channel * channel_mults[lvl]
        for _ in range(res_blocks + 1):
            ups.append(ResnetBlocWithAttn(width + skip_widths.pop(), out_w, noise_level_emb_dim=noise_level_channel,
                                          norm_groups=norm_groups, dropout=dropout, with_attn=(res in attn_res)))
            width = out_w
        if lvl != 0:
            ups.append(Upsample(width))
            res *= 2
    net.ups = nn.ModuleList(ups)
    net.final_conv = Block(width, default(out_channel, in_channel), groups=norm_groups)


def noise_level_mlp(inner_channel, act):
    """PositionalEncoding -> Linear -> act -> Linear: the noise-level embedding of every UNet of the family."""
    return nn.Sequential(
        PositionalEncoding(inner_channel),
        nn.Linear(inner_channel, inner_channel * 4),
        act,
        nn.Linear(inner_channel * 4, inner_channel),
    )


class PlannedUNet(nn.Module):
    """The engine glue shared by the four UNets: plan caches and ``forward`` through ``UNetPlan`` / ``UNetTrainPlan``.
    Subclasses build their modules and say how ``forward``'s input splits into (condition, x_t) (``_split``)."""

    def __init__(self):
        super().__init__()
        self._plans = {}

    def plan(self, batch, device=None, precision=None, strict_tc=False):
        """The compiled launch schedule for a given local batch size (cached)."""
        device = device or next(self.parameters()).device
        key = (batch, str(device), precision or self.precision, strict_tc)
        pl = self._plans.get(key)
        if pl is None:
            pl = UNetPlan(self, batch, device, precision or self.precision, strict_tc=strict_tc)
            self._plans[key] = pl
        pl.refresh_weights()
        return pl

    def train_plan(self, batch, device=None, precision=None):
        """Forward + backward schedule (``UNetTrainPlan``) for a given local batch size (cached)."""
        from ....unet_train import UNetTrainPlan
        device = device or next(self.parameters()).device
        key = ("train", batch, str(device), precision or self.precision)
        pl = self._plans.get(key)
        if pl is None:
            pl = UNetTrainPlan(self, batch, device, precision or self.precision)
            self._plans[key] = pl
        return pl

    def _apply(self, fn, *args, **kwargs):
        self._plans = {}           # .to() / .cuda() re-allocate the parameters: drop plans that point at the old storage
        return super()._apply(fn, *args, **kwargs)

    def _split(self, x):
        """forward's input -> (condition, x_t): x = cat([condition, x_t], 1) (ResDiff, PhyDiff, SR3)."""
        c = self.image_channels
        if x.shape[1] != 2 * c:
            raise AssertionError("expected cat([condition, x_t]) with %d channels, got %d" % (2 * c, x.shape[1]))
        return x[:, :c], x[:, c:]

    def forward(self, x, time):
        cond, x_t = self._split(x)
        b = x_t.shape[0]
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            # training step: the autograd node runs the hand-written backward pass (unet_train.py)
            from ....autograd_glue import DenoiseFn
            anchor = next(p for p in self.parameters() if p.requires_grad)
            return DenoiseFn.apply(anchor, self, cond, x_t, time)
        if self.training and self.dropout:
            pl = self.train_plan(b, x_t.device)
            pl.train_mode = True
        else:
            pl = self.plan(b, x_t.device)
        pl.set_condition(cond)
        pl.set_levels(time.reshape(b))
        return pl.denoise(x_t)


class UNet(PlannedUNet):
    def __init__(self, in_channel=9, out_channel=3, inner_channel=32, norm_groups=32, channel_mults=(1, 2, 4, 8, 8),
                 attn_res=(8,), res_blocks=3, dropout=0, with_noise_level_emb=True, image_width=128, image_height=128,
                 image_channels=3, precision="bf16"):
        super().__init__()
        if not with_noise_level_emb:
            raise NotImplementedError("with_noise_level_emb=False is never used on the reference's path")
        self.noise_level_mlp = noise_level_mlp(inner_channel, Swish())
        self.image_channels = image_channels
        self.fd_spliter = FD_Info_Spliter(dim=inner_channel, in_channels=image_channels, out_channels=out_channel,
                                          image_height=image_height, image_width=image_width)
        self.image_height, self.image_width = image_height, image_width
        self.inner_channel, self.norm_groups, self.dropout = inner_channel, norm_groups, dropout
        self.J = 4
        self.hf_ca_list = nn.ModuleList(
            [HF_guided_CA(inner_channel * (2 ** i), image_channels=image_channels) for i in range(self.J)])
        build_unet_body(self, in_channel, out_channel, inner_channel, norm_groups, channel_mults, attn_res, res_blocks,
                        dropout, inner_channel, image_height)
        self.precision = precision
        self.time_act = "swish"
