"""GaussianDiffusion -- drop-in for the reference's models/diffusion_models/diffusion.py:10-273.

Same constructor, buffers (12 fp32 schedule tables under the reference's names, so checkpoints round-trip),
attributes (``num_timesteps``, ``sqrt_alphas_cumprod_prev`` as a host numpy array) and methods.  The arithmetic of
``p_sample`` / ``q_sample`` / the loss runs in the fused CUDA kernels (wsr_sampler_step, wsr_q_sample,
wsr_noise_loss); the reverse loop keeps the step counter on the device and replays one captured CUDA graph per step
instead of ~610 eager launches plus a host->device copy (reference diffusion.py:159-160).
"""
import numpy as np
import torch
from torch import nn

from ... import _native as nat
from . import samplers
from .nn_modules.functional_layers import default
from .sheduler import make_beta_schedule

_TABLE_ORDER = ("sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod", "posterior_mean_coef1",
                "posterior_mean_coef2", "posterior_log_variance_clipped")


def rank_stream_seed(seed, rank=None):
    """seed -> a per-rank Philox key: rank 0 (and single-process runs) keep ``seed``; rank r > 0 gets splitmix64(seed + r * golden),
    so shards of one batch hold independent noise realisations while a single-GPU run with the same seed is unchanged."""
    if rank is None:
        import torch.distributed as dist
        rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
    if rank == 0:
        return int(seed) & ((1 << 62) - 1)
    m = (1 << 64) - 1
    z = (int(seed) + int(rank) * 0x9E3779B97F4A7C15) & m
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & m
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & m
    return (z ^ (z >> 31)) & ((1 << 62) - 1)


def member_key(seed, m):
    """Philox key of ensemble member m: the splitmix derivation of ``rank_stream_seed`` with the member index in place of the rank.
    Member 0 keeps ``seed`` (it is the single-GPU ``super_resolution`` run with that seed), and the key never depends on the rank,
    the chunking or the batch a member is sampled in."""
    return rank_stream_seed(seed, int(m))


def ensemble_chunks(n_members, batch, max_images=64, member_offset=0):
    """Member ranges [(first member, count)] sampled together: whole members, R = max(1, max_images // batch) per chunk."""
    per = max(1, int(max_images) // int(batch))
    return [(member_offset + c, min(per, n_members - c)) for c in range(0, int(n_members), per)]


class GaussianDiffusion(nn.Module):
    # ResDiff, PhyDiff, SRDiff: the forward process runs on HR - SR (q_sample around SR) and the sampler returns image + SR.
    # SR3 sets False: the target is HR itself and nothing is added back.
    residual = True

    def __init__(self, denoise_fn, channels=1, loss_type='l1', conditional=True, schedule_opt=None, image_height=128,
                 image_width=256, pretrained_model_path=None, lock_weights=True):
        super().__init__()
        self.channels = channels
        self.image_height = image_height
        self.image_width = image_width
        self.denoise_fn = denoise_fn
        self.loss_type = loss_type
        self.conditional = conditional
        self.use_cuda_graph = True
        self.sample_seed = None          # None -> derive from torch's global generator at every loop
        self._sampler_tables = None
        self.sampler = ("ddpm", None, None)   # set_sampler's (name, steps, eta)
        self._fewer_step_tables = None

    # ---- schedule (reference :49-96) --------------------------------------------------------------------------------
    def set_new_noise_schedule(self, schedule_opt, device):
        betas = make_beta_schedule(schedule=schedule_opt['schedule'], n_timestep=schedule_opt['n_timestep'],
                                   linear_start=schedule_opt['linear_start'], linear_end=schedule_opt['linear_end'])
        betas = np.asarray(betas, dtype=np.float64)
        alphas = 1.0 - betas
        abar = np.cumprod(alphas, axis=0)
        abar_prev = np.append(1.0, abar[:-1])
        self.sqrt_alphas_cumprod_prev = np.sqrt(np.append(1.0, abar))
        self.num_timesteps = int(betas.shape[0])
        post_var = betas * (1.0 - abar_prev) / (1.0 - abar)
        with np.errstate(divide="ignore", invalid="ignore"):
            tables = {
                'betas': betas,
                'alphas_cumprod': abar,
                'alphas_cumprod_prev': abar_prev,
                'sqrt_alphas_cumprod': np.sqrt(abar),
                'sqrt_one_minus_alphas_cumprod': np.sqrt(1.0 - abar),
                'log_one_minus_alphas_cumprod': np.log(1.0 - abar),
                'sqrt_recip_alphas_cumprod': np.sqrt(1.0 / abar),
                'sqrt_recipm1_alphas_cumprod': np.sqrt(1.0 / abar - 1),
                'posterior_variance': post_var,
                'posterior_log_variance_clipped': np.log(np.maximum(post_var, 1e-20)),
                'posterior_mean_coef1': betas * np.sqrt(abar_prev) / (1.0 - abar),
                'posterior_mean_coef2': (1.0 - abar_prev) * np.sqrt(alphas) / (1.0 - abar),
            }
        for name, arr in tables.items():
            self.register_buffer(name, torch.tensor(arr, dtype=torch.float32, device=device))
        self._sampler_tables = None
        self._fewer_step_tables = None

    def set_sampler(self, name="ddpm", steps=None, eta=None):
        """Select the reverse loop's sampler (samplers.py): 'ddpm' (the reference's ancestral loop over all T steps, the default),
        'ddim' (``steps`` of the T timesteps, ``eta`` in [0, inf), default 0; eta = 1 is the respaced ancestral sampler) or 'dpmpp2m'
        (DPM-Solver++(2M), deterministic).  steps=None is every timestep.  ``super_resolution``, ``p_sample_loop``,
        ``super_resolution_ensemble`` and ``begin_loop`` follow it; ``p_sample`` stays the DDPM step."""
        T = getattr(self, "num_timesteps", None)
        if T is None:
            raise ValueError("set_sampler needs the noise schedule (set_new_noise_schedule) first")
        samplers.check(name, steps, eta, T)
        self.sampler = (name, steps, eta)
        self._fewer_step_tables = None

    def _ddpm_tables_dev(self):
        """[5][T] fp32 table consumed by wsr_sampler_step + the T noise levels sqrt(abar_prev[t+1]) (:159-160)."""
        if self._sampler_tables is None or self._sampler_tables[0].device != self.betas.device:
            tab = torch.stack([getattr(self, n) for n in _TABLE_ORDER], 0).contiguous()
            levels = torch.tensor(self.sqrt_alphas_cumprod_prev[1:].astype(np.float32), device=self.betas.device)
            self._sampler_tables = (tab, levels)
        return self._sampler_tables

    def _tables_dev(self):
        """The selected sampler's [5][S] fp32 table and its S noise levels, rows in device-counter order (samplers.py)."""
        name, steps, eta = self.sampler
        if name == "ddpm":
            return self._ddpm_tables_dev()
        if self._fewer_step_tables is None or self._fewer_step_tables[0].device != self.betas.device:
            # the schedule may have changed since set_sampler: re-validate against the current T
            name, S, eta = samplers.check(name, steps, eta, self.num_timesteps)
            abar = np.square(self.sqrt_alphas_cumprod_prev[1:])
            tab, levels = samplers.tables(name, abar, S, eta)
            self._fewer_step_tables = (torch.tensor(tab, dtype=torch.float32, device=self.betas.device),
                                       torch.tensor(levels, dtype=torch.float32, device=self.betas.device))
        return self._fewer_step_tables

    def set_loss(self, device):
        if self.loss_type not in ('l1', 'l2'):
            raise NotImplementedError()
        self.loss_device = device

    # ---- closed-form pieces kept for API compatibility (reference :112-142) -----------------------------------------
    def predict_start_from_noise(self, x_t, t, noise):
        return self.sqrt_recip_alphas_cumprod[t] * x_t - self.sqrt_recipm1_alphas_cumprod[t] * noise

    def q_posterior(self, x_start, x_t, t):
        mean = self.posterior_mean_coef1[t] * x_start + self.posterior_mean_coef2[t] * x_t
        return mean, self.posterior_log_variance_clipped[t]

    # ---- engine glue ------------------------------------------------------------------------------------------------
    def _plan(self, batch, device):
        return self.denoise_fn.plan(batch, device)

    def _set_condition(self, plan, condition_x):
        plan.set_condition(condition_x)

    def _next_seed(self):
        """Philox seed of the next loop.  Under ``torch.distributed`` (batch-sharded sampling, parallel.py) every rank must draw
        DIFFERENT noise for its shard: the Philox counter is the local element index, and torch's default CPU generator starts
        from the same state in every process, so the rank is folded into the key (``rank_stream_seed``)."""
        base = int(self.sample_seed) if self.sample_seed is not None else int(torch.randint(0, 2 ** 62, (1,)).item())
        return rank_stream_seed(base)

    @torch.no_grad()
    def p_sample(self, x, t, clip_denoised=True, condition_x=None):
        """One reverse step x_t -> x_{t-1} (reference :175-192), generic (un-hoisted) entry."""
        if condition_x is None:
            raise NotImplementedError("unconditional sampling is not part of the accelerated path")
        plan = self._plan(x.shape[0], x.device)
        self._set_condition(plan, condition_x)
        tab, levels = self._ddpm_tables_dev()
        plan.set_level_table(levels)
        t_dev = torch.tensor([int(t)], dtype=torch.int32, device=x.device)
        xb = x.to(torch.float32).contiguous().clone()
        self._step(plan, xb, t_dev, tab, None, 0, self._next_seed(), clip_denoised)
        return xb

    def _step(self, plan, x, t_dev, tab, z, z_stride, seed, clip=True, members=None, hist=None):
        """members: None, or (device int64 key table, elements per member) -- an ensemble batch with member-keyed noise.
        hist: None (DDPM / DDIM tables), or the fp32 x0 history of a multistep (DPM-Solver++(2M)) table; the step then draws no noise.
        The table's row count is the loop length (T for DDPM, S for the fewer-step samplers)."""
        st = plan.eng.stream
        S = tab.shape[1]
        plan.select_level_row(t_dev)
        if plan.can_fuse_head():
            # head (GroupNorm + Swish + conv3x3) and the reverse-step update in one HBM-bound kernel
            feat = plan.run(x, head=False)
            plan.head_sampler_step(feat, x, tab, S, t_dev, z, z_stride, seed, clip, members=members, hist=hist)
            plan.eng.call("wsr_step_counter_add", t_dev.data_ptr(), -1, st)
            return
        plan.run(x)
        zp = 0 if z is None else z.data_ptr()
        if hist is not None:
            plan.eng.call("wsr_sampler_step_multistep", x.data_ptr(), plan.eps.data_ptr(), nat.F32, hist.data_ptr(), tab.data_ptr(), S,
                          t_dev.data_ptr(), 1 if clip else 0, x.data_ptr(), x.numel(), st, nbytes=x.numel() * 20)
        elif members is None:
            plan.eng.call("wsr_sampler_step", x.data_ptr(), plan.eps.data_ptr(), nat.F32, zp, z_stride, seed, tab.data_ptr(),
                          S, t_dev.data_ptr(), 1 if clip else 0, x.data_ptr(), x.numel(), st,
                          nbytes=x.numel() * (16 if z is not None else 12))
        else:
            plan.eng.call("wsr_sampler_step_members", x.data_ptr(), plan.eps.data_ptr(), nat.F32, zp, z_stride, members[0].data_ptr(),
                          members[1], tab.data_ptr(), S, t_dev.data_ptr(), 1 if clip else 0, x.data_ptr(), x.numel(),
                          st, nbytes=x.numel() * (16 if z is not None else 12))
        plan.eng.call("wsr_step_counter_add", t_dev.data_ptr(), -1, st)

    @torch.no_grad()
    def begin_loop(self, plan, shape, noise_chain=None, seed=None, member_keys=None):
        """Set up a reverse loop on the plan's current condition and return its state object (see ReverseLoop)."""
        return ReverseLoop(self, plan, shape, noise_chain, seed, member_keys)

    @torch.no_grad()
    def _reverse_loop(self, plan, shape, noise_chain=None, seed=None, steps=None, collect_eps=False, member_keys=None):
        """S reverse steps of the selected sampler (S = T for DDPM) on the plan's current condition.  noise_chain: optional injected
        noise [S+1, *shape] (index 0 = initial image, index S-t = noise of the step at counter t) for parity runs; otherwise Philox
        noise from ``seed``, or, with ``member_keys`` (R Philox keys), from key member_keys[m] for the m-th of R equal member slices of
        the batch.  Returns the final x_0 (fp32 NCHW)."""
        loop = self.begin_loop(plan, shape, noise_chain, seed, member_keys)
        n_steps = loop.S if steps is None else min(int(steps), loop.S)
        eps_log = []
        # first step eagerly (lazy initialisation of kernel attributes happens here), the rest as graph replays
        loop.step()
        if collect_eps:
            eps_log.append(plan.eps.clone())
        remaining = n_steps - 1
        if remaining > 0 and self.use_cuda_graph and not collect_eps:
            loop.capture()
            for _ in range(remaining):
                loop.replay()
        else:
            for _ in range(remaining):
                loop.step()
                if collect_eps:
                    eps_log.append(plan.eps.clone())
        if collect_eps:
            return loop.x, eps_log
        return loop.x

    def _loop_input(self, x_in):
        """super_resolution's dict -> p_sample_loop's input: the condition x_in['SR']."""
        return x_in["SR"]

    def _loop_condition(self, x):
        """p_sample_loop's input -> (condition tensor for the plan, field added to the sampled image or None).  Here x is the
        condition itself, which is added back when the process is ``residual``."""
        cond = x.to(device=self.betas.device, dtype=torch.float32)
        return cond, (cond if self.residual else None)

    @torch.no_grad()
    def p_sample_loop(self, x_in, continous=False, noise_chain=None, seed=None):
        """The conditional reverse loop (reference :58-94): x_in is ``_loop_input``'s form of the batch."""
        if not self.conditional:
            raise NotImplementedError("unconditional sampling is not part of the accelerated path")
        cond, add = self._loop_condition(x_in)
        shape = tuple((cond if add is None else add).shape)       # the image's: the added field's, or (SR3) the condition's
        plan = self._plan(shape[0], self.betas.device)
        plan.set_condition(cond)
        img = self._reverse_loop(plan, shape, noise_chain=noise_chain, seed=seed)
        return img if add is None else img + add

    @torch.no_grad()
    def super_resolution(self, x_in, continous=False):
        return self.p_sample_loop(self._loop_input(x_in), continous)

    @torch.no_grad()
    def super_resolution_ensemble(self, x_in, n_members, seed=None, member_offset=0, max_images=64):
        """``n_members`` samples per condition: (n_members, B, C, H, W) fp32.  Member k is global member member_offset + k, whose
        noise is Philox key ``member_key(seed, member_offset + k)``: it equals ``p_sample_loop`` on the B conditions with that seed,
        independently of the chunking and of ``member_offset``.  Members run in chunks of R = max(1, max_images // B) whole members;
        a chunk is one reverse loop over R * B images whose condition-only work runs once on the B conditions
        (``UNetPlan.set_condition(cond, repeats=R)``)."""
        if not self.conditional:
            raise NotImplementedError("unconditional sampling is not part of the accelerated path")
        n_members = int(n_members)
        if n_members < 1:
            raise ValueError("n_members must be >= 1")
        dev = self.betas.device
        shape = tuple(x_in["SR"].shape)
        B = shape[0]
        base = int(seed) if seed is not None else (int(self.sample_seed) if self.sample_seed is not None
                                                   else int(torch.randint(0, 2 ** 62, (1,)).item()))
        cond, add = self._loop_condition(self._loop_input(x_in))
        out = torch.empty((n_members,) + shape, device=dev, dtype=torch.float32)
        for first, r in ensemble_chunks(n_members, B, max_images, member_offset):
            plan = self._plan(r * B, dev)
            plan.set_condition(cond, repeats=r)
            keys = torch.tensor([member_key(base, first + k) for k in range(r)], dtype=torch.int64).to(dev)
            img = self._reverse_loop(plan, (r * B,) + shape[1:], member_keys=keys)
            k0 = first - member_offset
            dst = out[k0:k0 + r]
            dst.copy_(img.view((r,) + shape))
            if add is not None:
                dst.add_(add.unsqueeze(0))
        return out

    @torch.no_grad()
    def sample(self, batch_size=1, continous=False):
        return self.p_sample_loop((batch_size, self.channels, self.image_height, self.image_height), continous)

    def q_sample(self, x_start, continuous_sqrt_alpha_cumprod, noise=None, offset=None):
        """reference :209-228.  x_start (B,C,H,W), continuous_sqrt_alpha_cumprod (B,1,1,1).  offset: x_t is centred on
        ``offset + a * x_start`` (the residual processes' SR; None = 0)."""
        noise = default(noise, lambda: torch.randn_like(x_start))
        x0 = x_start.to(torch.float32).contiguous()
        a = continuous_sqrt_alpha_cumprod.reshape(-1).to(torch.float32).contiguous()
        nz = noise.to(torch.float32).contiguous()
        off = torch.zeros_like(x0) if offset is None else offset.to(torch.float32).contiguous()
        out = torch.empty_like(x0)
        nat.call("wsr_q_sample", x0.data_ptr(), off.data_ptr(), nz.data_ptr(), a.data_ptr(), x0.shape[0],
                 x0[0].numel(), out.data_ptr(), torch.cuda.current_stream(x0.device).cuda_stream)
        return out

    def _draw_levels(self, b, device):
        """ONE t per batch, then b continuous noise levels in [sqrt(abar[t-1]), sqrt(abar[t])), from numpy's global RNG in the
        reference's order: randint, then uniform (reference :116-121)."""
        t = np.random.randint(1, self.num_timesteps + 1)
        return torch.FloatTensor(np.random.uniform(self.sqrt_alphas_cumprod_prev[t - 1],
                                                   self.sqrt_alphas_cumprod_prev[t], size=b)).to(device)

    def _loss(self, noise, eps):
        """The noise loss, through the autograd node when eps carries a gradient."""
        if eps.requires_grad:
            from ...autograd_glue import NoiseLossFn
            return NoiseLossFn.apply(noise, eps, self.loss_type == 'l2')
        return self._noise_loss(noise, eps)

    def _noise_loss(self, noise, eps):
        """Sum-reduced L1/L2 (reference :98-110) computed by wsr_noise_loss; returns a 0-dim fp32 tensor."""
        acc = torch.zeros(1, dtype=torch.float64, device=noise.device)
        nat.call("wsr_noise_loss", noise.data_ptr(), eps.data_ptr(), noise.numel(), 1 if self.loss_type == 'l2' else 0,
                 acc.data_ptr(), 0, 0.0, torch.cuda.current_stream(noise.device).cuda_stream)
        return acc.to(torch.float32)[0]

    def forward(self, x, *args, **kwargs):
        return self.p_losses(x, *args, **kwargs)

    def p_losses(self, x_in, noise=None):
        """reference :111-152: one t per batch and per-sample continuous level (``_draw_levels``), q_sample of HR around SR
        (``residual``) or 0, the denoiser on cat([SR, x_t]), sum-reduced loss."""
        sr, hr = x_in['SR'], x_in['HR']
        b = sr.shape[0]
        level = self._draw_levels(b, sr.device)
        noise = default(noise, lambda: torch.randn_like(sr)).to(torch.float32).contiguous()
        hr32, sr32 = hr.to(torch.float32).contiguous(), sr.to(torch.float32).contiguous()
        x_noisy = self.q_sample(hr32, level, noise, offset=sr32 if self.residual else None)
        if not self.conditional:
            raise NotImplementedError("unconditional training is not part of the accelerated path")
        eps = self.denoise_fn(torch.cat([sr32, x_noisy], dim=1), level.view(b, -1))
        return self._loss(noise, eps)


class ReverseLoop:
    """State of one reverse loop of the diffusion's sampler: the image x (updated in place), the device-side step counter
    (S-1 -> 0, S = T for DDPM), the x0 history of a multistep sampler and the captured CUDA graph of one step.  ``step()``
    launches one step eagerly, ``capture()`` records the same launches into a graph, ``replay()`` replays it -- the step index
    and the history live on the device, so every replay advances the chain."""

    def __init__(self, diffusion, plan, shape, noise_chain=None, seed=None, member_keys=None):
        self.diffusion, self.plan = diffusion, plan
        dev = plan.eng.device
        self.tab, levels = diffusion._tables_dev()
        self.S = S = self.tab.shape[1]
        plan.set_level_table(levels)
        self.x = torch.empty(shape, device=dev, dtype=torch.float32)
        self.hist = torch.zeros(shape, device=dev, dtype=torch.float32) if diffusion.sampler[0] == "dpmpp2m" else None
        # an explicit seed is still made rank-distinct: sharded ranks pass the same value (bench.py, sample.py)
        self.seed = diffusion._next_seed() if seed is None else rank_stream_seed(int(seed))
        self.members = None
        if member_keys is not None:
            # ensemble batch: R equal member slices, each keyed by its own entry of the (constant, graph-safe) device key table
            keys = member_keys.to(device=dev, dtype=torch.int64).contiguous()
            n = 1
            for d in shape:
                n *= int(d)
            assert n % keys.numel() == 0
            self.members = (keys, n // keys.numel())
        if noise_chain is not None:
            self.z = noise_chain.to(device=dev, dtype=torch.float32).contiguous()
            assert self.z.shape[0] == S + 1 and tuple(self.z.shape[1:]) == tuple(shape)
            self.x.copy_(self.z[0])
            self.z_stride = self.x.numel()
        else:
            self.z, self.z_stride = None, 0
            if self.members is None:
                nat.call("wsr_randn", self.x.data_ptr(), self.x.numel(), self.seed, 0xFFFFFFFF, plan.eng.stream)
            else:
                nat.call("wsr_randn_members", self.x.data_ptr(), self.x.numel(), self.members[0].data_ptr(), self.members[1],
                         0xFFFFFFFF, plan.eng.stream)
        self.t_dev = torch.tensor([S - 1], dtype=torch.int32, device=dev)
        self.graph = None

    def reset_counter(self, t=None):
        self.t_dev.fill_(self.S - 1 if t is None else int(t))

    def step(self):
        self.diffusion._step(self.plan, self.x, self.t_dev, self.tab, self.z, self.z_stride, self.seed, members=self.members, hist=self.hist)

    def capture(self):
        torch.cuda.synchronize(self.plan.eng.device)
        self.graph = torch.cuda.CUDAGraph()
        # small batches (<= 8 images of 128x256 per GPU -- the sharded benchmark): the ~190 launches of a step are short enough for the
        # gaps between them to show, so the graph is captured with programmatic dependent launch (wsr.h: wsr_set_pdl)
        small = self.x.shape[0] * self.x.shape[-2] * self.x.shape[-1] <= 8 * 128 * 256
        prev = nat.call("wsr_set_pdl", 1) if small else None
        try:
            with torch.cuda.graph(self.graph):
                self.step()
        finally:
            if prev is not None:
                nat.call("wsr_set_pdl", prev)
        return self.graph

    def replay(self):
        self.graph.replay()
