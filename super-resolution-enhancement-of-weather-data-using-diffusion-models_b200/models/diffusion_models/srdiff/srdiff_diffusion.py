"""SRDiffDiffusion -- drop-in for the reference's srdiff/srdiff_diffusion.py:9-219: RRDB encoder once per batch, then T reverse
steps of the SRDiff UNet conditioned on 6 of its 18 feature maps; training with a frozen (``lock_weights=True``) or a jointly trained
encoder."""
import torch

from ...rrdb_encoder.RRDBNet import RRDBNet
from ..diffusion import GaussianDiffusion
from ..nn_modules.functional_layers import default


class SRDiffDiffusion(GaussianDiffusion):
    def __init__(self, denoise_fn, image_height, image_width, channels=1, loss_type='l1', conditional=True,
                 schedule_opt=None, pretrained_model_path=None, lock_weights=True):
        super().__init__(denoise_fn=denoise_fn, channels=channels, loss_type=loss_type, conditional=conditional,
                         schedule_opt=schedule_opt, image_height=image_height, image_width=image_width,
                         pretrained_model_path=pretrained_model_path, lock_weights=lock_weights)
        self.lock_weights = lock_weights
        self.rrdb_encoder = None
        if pretrained_model_path is not None:
            self.init_rrdb_encoder(pretrained_model_path, lock_weights)

    def init_rrdb_encoder(self, pretrained_model_path, lock_weights=True):
        hidden_size, num_block = 64, 17
        self.rrdb_encoder = RRDBNet(self.channels, self.channels, hidden_size, num_block, hidden_size // 2,
                                    precision=getattr(self.denoise_fn, "precision", "bf16"))
        if pretrained_model_path:
            self.rrdb_encoder.load_state_dict(torch.load(pretrained_model_path))
        if lock_weights:
            self.rrdb_encoder.eval()
            for p in self.rrdb_encoder.parameters():
                p.requires_grad_(False)

    def _condition(self, lr):
        """cat(feas[2::3], 1) as an NCHW fp32 tensor (B, 384, h, w)."""
        if self.rrdb_encoder is None:
            raise NotImplementedError("SRDiff without an RRDB encoder conditions on raw LR, which the reference's UNet cannot consume")
        pl, feas = self.rrdb_encoder.features_device(lr)
        return torch.cat([f.to_nchw(pl.eng) for f in feas[2::3]], dim=1)

    def _loop_input(self, x_in):
        """p_sample_loop takes the whole dict (reference :77-117): 'LR' feeds the encoder, 'SR' is added back."""
        return x_in

    def _loop_condition(self, x_in):
        """The RRDB encoder runs once on the B LR fields; the bicubic SR is added back."""
        dev = self.betas.device
        return self._condition(x_in['LR'].to(dev)), x_in['SR'].to(device=dev, dtype=torch.float32)

    @torch.no_grad()
    def p_sample(self, x, t, clip_denoised=True, condition_x=None):
        """condition_x: the list of 18 RRDB feature maps (reference :133-159)."""
        cond = torch.cat(list(condition_x[2::3]), dim=1)
        return super().p_sample(x, t, clip_denoised=clip_denoised, condition_x=cond)

    def p_losses(self, x_in, noise=None):
        """reference :161-216.  Locked encoder: the noise loss alone.  ``lock_weights=False``: ``loss + F.l1_loss(rrdb_sr, HR)`` (:212-214)
        with the gradient flowing into the encoder both through its SR image and through the six condition features."""
        sr_up, lr, hr = x_in['SR'], x_in['LR'], x_in['HR']
        dev = sr_up.device
        b = sr_up.shape[0]
        joint = (self.rrdb_encoder is not None and not self.lock_weights and torch.is_grad_enabled()
                 and any(p.requires_grad for p in self.rrdb_encoder.parameters()))
        if joint:
            rrdb_sr, feas = self.rrdb_encoder.forward_joint(lr.to(dev))
        else:
            rrdb_sr, feas = self.rrdb_encoder(lr, True)
        level = self._draw_levels(b, dev)
        noise = default(noise, lambda: torch.randn_like(sr_up)).to(torch.float32).contiguous()
        hr32, sr32 = hr.to(torch.float32).contiguous(), sr_up.to(torch.float32).contiguous()
        x_noisy = self.q_sample(hr32, level, noise, offset=sr32)
        loss = self._loss(noise, self.denoise_fn((feas, x_noisy), level.view(b, -1)))
        if self.rrdb_encoder is not None and not self.lock_weights:
            return loss + torch.nn.functional.l1_loss(rrdb_sr, hr.to(torch.float32))          # reference :212-214
        return loss
