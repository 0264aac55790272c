"""Bridges between torch.autograd and the hand-written backward pass, so that the reference's training code
(``l_pix = netG(data); l_pix = l_pix.sum() / n; l_pix.backward(); optG.step()``, models/diffusion_models/model.py:61-69)
runs unchanged on the CUDA path.

``DenoiseFn``   eps_hat = UNet(cat([cond, x_t]), level).  backward() runs ``UNetTrainPlan.backward`` and installs every
                parameter gradient as ``p.grad`` (a view into the plan's flat gradient buffer).
``NoiseLossFn`` sum-reduced L1 / L2 between the injected noise and eps_hat (diffusion.py:98-110) via ``wsr_noise_loss``.
``FusedAdam``   torch.optim.Adam-compatible optimizer (same state_dict layout) whose update is ``wsr_adam_step``: one
                launch over the flat parameter buffer when the parameters were flattened by the train plan.  Optionally keeps
                an EMA of the weights, updated in the same launch (``wsr_adam_step_ema``).
"""
import torch

from . import _native as nat

weights_epoch = 0          # bumped by every optimizer step that writes parameters through raw pointers
weights_swapped = False    # True inside DDPM.ema_weights(): a training forward there is refused (see its docstring)


class DenoiseFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, anchor, net, cond, x_t, time):
        """cond, x_t: the split of the UNet's input (``PlannedUNet._split``).  A condition that requires grad -- SRDiff with a
        trainable encoder, cat(feas[2::3]) -- gets its gradient (``UNetTrainPlan.cond_grad``) back into the encoder's backward pass."""
        if weights_swapped:
            raise RuntimeError("training forward inside DDPM.ema_weights(): the train plan would keep EMA-derived level projections "
                               "and condition weights for the first training forward after the swap back")
        b = x_t.shape[0]
        pl = net.train_plan(b, x_t.device)
        pl.train_mode = bool(net.training)
        pl.want_cond_grad = ctx.needs_input_grad[2]
        pl.set_condition(cond.detach())
        pl.set_levels(time.reshape(b))
        eps = pl.denoise(x_t)
        ctx.pl, ctx.net = pl, net
        return eps

    @staticmethod
    def backward(ctx, d_eps):
        pl, net = ctx.pl, ctx.net
        pairs = pl.param_grads()
        stale = None
        if any(p.grad is not None and p.grad.data_ptr() == g.data_ptr() for p, g in pairs):
            stale = pl.gflat.clone()          # gradients of an earlier backward were not cleared: accumulate
        pl.backward(d_eps)
        if stale is not None:
            pl.gflat.add_(stale)
        for p, g in pairs:
            if not p.requires_grad:
                continue
            if p.grad is None or p.grad.data_ptr() == g.data_ptr():
                p.grad = g
            else:
                p.grad.add_(g)
        return None, None, (pl.cond_grad() if ctx.needs_input_grad[2] else None), None, None


class NoiseLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, noise, eps, l2):
        acc = torch.zeros(1, dtype=torch.float64, device=noise.device)
        grad = torch.empty_like(eps)               # d loss / d eps for an upstream gradient of 1 (same kernel, same pass)
        nat.call("wsr_noise_loss", noise.data_ptr(), eps.data_ptr(), noise.numel(), 1 if l2 else 0, acc.data_ptr(), grad.data_ptr(), 1.0,
                 torch.cuda.current_stream(noise.device).cuda_stream)
        ctx.save_for_backward(grad)
        return acc.to(torch.float32)[0]

    @staticmethod
    def backward(ctx, go):
        (grad,) = ctx.saved_tensors
        # scaling by the 0-dim upstream gradient stays on the device: reading it on the host would stall the launch queue
        # between the forward and the backward pass
        return None, grad * go.to(grad.dtype), None


def check_ema_schedule(sched):
    """``train.ema_scheduler`` of a config -> (step_start_ema, update_ema_every, ema_decay); ValueError when a key is missing or
    out of range."""
    if not isinstance(sched, dict):
        raise ValueError("EMA needs train.ema_scheduler {step_start_ema, update_ema_every, ema_decay} in the config")
    missing = [k for k in ("step_start_ema", "update_ema_every", "ema_decay") if sched.get(k) is None]
    if missing:
        raise ValueError("train.ema_scheduler lacks %s" % ", ".join(missing))
    start, every, decay = int(sched["step_start_ema"]), int(sched["update_ema_every"]), float(sched["ema_decay"])
    if every < 1:
        raise ValueError("train.ema_scheduler.update_ema_every must be >= 1 (got %d)" % every)
    if start < 0:
        raise ValueError("train.ema_scheduler.step_start_ema must be >= 0 (got %d)" % start)
    if not 0.0 <= decay < 1.0:
        raise ValueError("train.ema_scheduler.ema_decay must be in [0, 1) (got %r)" % decay)
    return start, every, decay


def ema_action(step, start, every):
    """What the s-th optimizer step (s = 1, 2, ...) does to the EMA, with k = s - 1: 'skip' when k % every != 0, else 'copy'
    (ema = p) while k < start, else 'blend' (ema = ema * d + (1 - d) * p)."""
    k = step - 1
    if k % every != 0:
        return "skip"
    return "copy" if k < start else "blend"


class FusedAdam(torch.optim.Optimizer):
    """Adam with torch.optim.Adam's arithmetic and state layout (``step``, ``exp_avg``, ``exp_avg_sq`` per parameter);
    amsgrad / maximize / capturable are not supported (the reference uses none of them).

    ``ema=(step_start_ema, update_ema_every, ema_decay)`` also keeps an exponential moving average of every parameter it steps
    (``ema_action``), updated inside the Adam launch by ``wsr_adam_step_ema``.  The averages live in ``self.ema`` (parameter ->
    tensor), outside ``state_dict()``, which stays torch.optim.Adam's."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, ema=None):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        self._flat = None
        self.ema, self.ema_schedule = None, None
        if ema is not None:
            self.enable_ema(ema)

    @torch.no_grad()
    def enable_ema(self, schedule):
        """Start the EMA from the current parameter values."""
        start, every, decay = schedule
        self.ema_schedule = (int(start), int(every), float(decay))
        self.ema = {p: p.detach().clone() for group in self.param_groups for p in group["params"] if p.requires_grad}
        if self._flat is not None:
            self.attach_flat(self._flat["plan"])

    def attach_flat(self, plan):
        """Use the train plan's flat parameter / gradient buffers: one kernel launch per step.  Existing per-parameter state
        (a loaded checkpoint, or steps already taken one by one) is COPIED into the flat moment buffers, so attaching before or
        after ``load_state_dict`` keeps the optimizer state.  The same holds for the EMA."""
        pflat = plan.flatten_parameters()
        m, v = torch.zeros_like(pflat), torch.zeros_like(pflat)
        e = pflat.clone() if self.ema is not None else None
        step = 0
        for p in plan.param_order:
            off = plan._goff[id(p)]
            st = self.state.get(p)
            if st:
                m[off:off + p.numel()].copy_(st["exp_avg"].reshape(-1))
                v[off:off + p.numel()].copy_(st["exp_avg_sq"].reshape(-1))
                step = max(step, int(float(st["step"])))
            if e is not None and p in self.ema:
                e[off:off + p.numel()].copy_(self.ema[p].reshape(-1))
        self._flat = dict(plan=plan, p=pflat, m=m, v=v, ema=e, step=step)
        step_t = torch.tensor(float(step))
        for p in plan.param_order:
            off = plan._goff[id(p)]
            st = self.state[p]
            st["step"] = step_t
            st["exp_avg"] = m[off:off + p.numel()].view(p.shape)
            st["exp_avg_sq"] = v[off:off + p.numel()].view(p.shape)
            if e is not None and p in self.ema:
                self.ema[p] = e[off:off + p.numel()].view(p.shape)

    def load_state_dict(self, state_dict):
        """torch.optim.Optimizer.load_state_dict replaces the state tensors: the per-parameter ``step`` counters are moved back to
        the host (a CUDA ``step`` would cost one device->host read per parameter per step in ``_step_each``), and an attached
        flat plan is re-synchronised with the loaded moments instead of silently keeping its zeros."""
        super().load_state_dict(state_dict)
        for st in self.state.values():
            if torch.is_tensor(st.get("step")) and st["step"].is_cuda:
                st["step"] = st["step"].cpu()
        if self._flat is not None:
            self.attach_flat(self._flat["plan"])

    def _flat_ok(self):
        f = self._flat
        if f is None or len(self.param_groups) != 1:
            return False
        plan = f["plan"]
        if not plan.parameters_are_flat():
            return False
        for p, g in plan.param_grads():
            if p.grad is None or p.grad.data_ptr() != g.data_ptr():
                return False
        return True

    @torch.no_grad()
    def step(self, closure=None):
        global weights_epoch
        loss = closure() if closure is not None else None
        if self._flat_ok():
            f, group = self._flat, self.param_groups[0]
            plan = f["plan"]
            f["step"] += 1
            self._launch(f["p"], plan.gflat, f["m"], f["v"], f["ema"], f["step"], group)
            step_t = torch.tensor(float(f["step"]))
            for p in plan.param_order:
                self.state[p]["step"] = step_t
            # parameters of the group that are NOT part of the flat plan (e.g. a jointly trained RRDB encoder) step one by one
            in_plan = f.get("ids")
            if in_plan is None:
                in_plan = f["ids"] = {id(p) for p in plan.param_order}
            self._step_each([p for p in group["params"] if id(p) not in in_plan], group)
            weights_epoch += 1
            return loss
        for group in self.param_groups:
            self._step_each(group["params"], group)
        weights_epoch += 1
        return loss

    def _step_each(self, params, group):
        for p in params:
            if p.grad is None:
                continue
            if p.dtype != torch.float32 or not p.is_contiguous() or not p.is_cuda:
                raise nat.WsrError("FusedAdam: parameters must be contiguous fp32 CUDA tensors")
            g = p.grad if p.grad.is_contiguous() else p.grad.contiguous()
            st = self.state[p]
            if len(st) == 0:
                st["step"] = torch.tensor(0.0)
                st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
            st["step"] = st["step"] + 1
            self._launch(p, g, st["exp_avg"], st["exp_avg_sq"], None if self.ema is None else self.ema.get(p),
                         int(st["step"].item()), group)

    def _launch(self, p, g, m, v, ema, step, group):
        """One Adam update; with EMA, the fused variant on the steps where the schedule writes the EMA (d = 0 copies)."""
        b1, b2 = group["betas"]
        args = (float(group["lr"]), float(b1), float(b2), float(group["eps"]), float(group["weight_decay"]), int(step))
        stream = torch.cuda.current_stream(p.device).cuda_stream
        action = "skip" if ema is None else ema_action(step, *self.ema_schedule[:2])
        if action == "skip":
            nat.call("wsr_adam_step", p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), *args, stream)
        else:
            decay = 0.0 if action == "copy" else self.ema_schedule[2]
            nat.call("wsr_adam_step_ema", p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), ema.data_ptr(), p.numel(), *args,
                     decay, stream)
