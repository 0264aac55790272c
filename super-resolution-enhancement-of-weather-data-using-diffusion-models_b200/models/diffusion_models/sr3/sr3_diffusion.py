"""SR3Diffusion -- drop-in for the reference's sr3/sr3_diffusion.py:8-140: the condition is ``x_in['SR']``, the target of the
forward process is HR itself (no residual), and the sampler returns the final image WITHOUT adding the condition (:84)."""
import numpy as np
import torch

from .... import _native as nat
from ..diffusion import GaussianDiffusion
from ..nn_modules.functional_layers import default


class SR3Diffusion(GaussianDiffusion):
    def __init__(self, denoise_fn, channels=1, image_height=128, image_width=256, loss_type='l1', conditional=True,
                 schedule_opt=None, pretrained_model_path=None, lock_weights=True):
        super().__init__(denoise_fn=denoise_fn, channels=channels, loss_type=loss_type, conditional=conditional,
                         schedule_opt=schedule_opt, image_height=image_height, image_width=image_width,
                         pretrained_model_path=pretrained_model_path, lock_weights=lock_weights)

    @torch.no_grad()
    def p_sample_loop(self, x_in, continous=False, noise_chain=None, seed=None):
        """reference :49-84 (conditional branch): x_in is the condition (B,C,H,W); returns the final image."""
        if not self.conditional:
            raise NotImplementedError("unconditional sampling is not part of the accelerated path")
        cond = x_in
        plan = self._plan(cond.shape[0], self.betas.device)
        plan.set_condition(cond.to(self.betas.device))
        return self._reverse_loop(plan, tuple(cond.shape), noise_chain=noise_chain, seed=seed).clone()

    @torch.no_grad()
    def super_resolution(self, x_in, continous=False):
        return self.p_sample_loop(x_in["SR"], continous)

    def _ensemble_condition(self, x_in):
        """SR3 returns the final image itself: nothing is added back."""
        return x_in["SR"].to(device=self.betas.device, dtype=torch.float32), None

    def p_losses(self, x_in, noise=None):
        """reference :101-137: x_start = HR, one t per batch, per-sample continuous level, sum-reduced loss."""
        hr, sr = x_in['HR'], x_in['SR']
        b = hr.shape[0]
        dev = hr.device
        t = np.random.randint(1, self.num_timesteps + 1)
        level = torch.FloatTensor(np.random.uniform(self.sqrt_alphas_cumprod_prev[t - 1],
                                                    self.sqrt_alphas_cumprod_prev[t], size=b)).to(dev)
        noise = default(noise, lambda: torch.randn_like(hr)).to(torch.float32).contiguous()
        hr32, sr32 = hr.to(torch.float32).contiguous(), sr.to(torch.float32).contiguous()
        zero = torch.zeros_like(hr32)
        x_noisy = torch.empty_like(hr32)
        nat.call("wsr_q_sample", hr32.data_ptr(), zero.data_ptr(), noise.data_ptr(), level.data_ptr(), b,
                 hr32[0].numel(), x_noisy.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
        if not self.conditional:
            raise NotImplementedError("unconditional training is not part of the accelerated path")
        eps = self.denoise_fn(torch.cat([sr32, x_noisy], dim=1), level.view(b, -1))
        if eps.requires_grad:
            from ....autograd_glue import NoiseLossFn
            return NoiseLossFn.apply(noise, eps, self.loss_type == 'l2')
        return self._noise_loss(noise, eps)
