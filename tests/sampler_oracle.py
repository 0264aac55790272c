"""float64 reference chains of the fewer-step samplers, written from the papers' x0 / eps / lambda form rather than from the folded
coefficient tables of ``models/diffusion_models/samplers.py``, so that they check the folding independently.

  DDIM(eta)        Song et al., "Denoising Diffusion Implicit Models" (2021), eq. 12 and 16, with the reference's x0 clamp.
  DPM-Solver++(2M) Lu et al., "DPM-Solver++" (2022), Algorithm 2 (data prediction, multistep second order), first order on the first
                   step and on the step into the last timestep.

``denoise(x, level)`` -> eps_hat for x (fp32) and level (B, 1) fp32 = sqrt(alphas_cumprod[tau]).  Noise is injected in the chain
layout of the parity tests: noise[0] is the initial image, noise[k + 1] the z of the k-th step (unused by DPM-Solver++(2M))."""
import numpy as np
import torch

from oracle import schedule


def alphas_cumprod(schedule_opt):
    b = schedule.betas_for(schedule_opt["schedule"], schedule_opt["n_timestep"], schedule_opt["linear_start"], schedule_opt["linear_end"])
    return np.cumprod(1.0 - b)


def taus(T, S):
    return [int(t) for t in np.rint(np.linspace(T - 1, 0, S))]


def _eps_x0(denoise, x, a, clip):
    level = torch.full((x.shape[0], 1), float(np.float32(np.sqrt(a))), dtype=torch.float32)
    eps = denoise(x.float(), level).double()
    x0 = (x - np.sqrt(1.0 - a) * eps) / np.sqrt(a)
    return x0.clamp(-1.0, 1.0) if clip else x0


def ddim_chain(denoise, abar, S, noise, eta=0.0, clip=True):
    ts = taus(len(abar), S)
    x = noise[0].double()
    for k, t in enumerate(ts):
        a = abar[t]
        x0 = _eps_x0(denoise, x, a, clip)
        if k == S - 1:
            return x0
        a_next = abar[ts[k + 1]]
        sigma = eta * np.sqrt((1.0 - a_next) / (1.0 - a)) * np.sqrt(1.0 - a / a_next)
        eps = (x - np.sqrt(a) * x0) / np.sqrt(1.0 - a)          # the noise direction implied by the (clamped) x0
        x = np.sqrt(a_next) * x0 + np.sqrt(max(1.0 - a_next - sigma ** 2, 0.0)) * eps
        if sigma > 0:
            x = x + sigma * noise[k + 1].double()
    return x


def dpmpp2m_chain(denoise, abar, S, noise, clip=True):
    ts = taus(len(abar), S)
    x = noise[0].double()
    x0_prev = h_prev = None
    for k, t in enumerate(ts):
        a = abar[t]
        x0 = _eps_x0(denoise, x, a, clip)
        if k == S - 1:
            return x0
        a_next = abar[ts[k + 1]]
        alpha_n, sig, sig_n = np.sqrt(a_next), np.sqrt(1.0 - a), np.sqrt(1.0 - a_next)
        lam, lam_n = np.log(np.sqrt(a) / sig), np.log(alpha_n / sig_n)
        h = lam_n - lam
        if x0_prev is None or k + 1 == S - 1:
            D = x0
        else:
            r = h_prev / h
            D = (1.0 + 1.0 / (2.0 * r)) * x0 - (1.0 / (2.0 * r)) * x0_prev
        x = (sig_n / sig) * x - alpha_n * (np.exp(-h) - 1.0) * D
        x0_prev, h_prev = x0, h
    return x
