"""Bridges between torch.autograd and the hand-written backward pass, so that the reference's training code
(``l_pix = netG(data); l_pix = l_pix.sum() / n; l_pix.backward(); optG.step()``, models/diffusion_models/model.py:61-69)
runs unchanged on the CUDA path.

``DenoiseFn``   eps_hat = UNet(cat([cond, x_t]), level).  backward() runs ``UNetTrainPlan.backward`` and installs every
                parameter gradient as ``p.grad`` (a view into the plan's flat gradient buffer).
``NoiseLossFn`` sum-reduced L1 / L2 between the injected noise and eps_hat (diffusion.py:98-110) via ``wsr_noise_loss``.
``FusedAdam``   torch.optim.Adam-compatible optimizer (same state_dict layout) whose update is ``wsr_adam_step``: one
                launch over the flat parameter buffer when the parameters were flattened by the train plan.
"""
import torch

from . import _native as nat

weights_epoch = 0          # bumped by every optimizer step that writes parameters through raw pointers


class DenoiseFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, anchor, net, cond, x_t, time):
        """cond, x_t: the split of the UNet's input (``PlannedUNet._split``).  A condition that requires grad -- SRDiff with a
        trainable encoder, cat(feas[2::3]) -- gets its gradient (``UNetTrainPlan.cond_grad``) back into the encoder's backward pass."""
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


class FusedAdam(torch.optim.Optimizer):
    """Adam with torch.optim.Adam's arithmetic and state layout (``step``, ``exp_avg``, ``exp_avg_sq`` per parameter);
    amsgrad / maximize / capturable are not supported (the reference uses none of them)."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        self._flat = None

    def attach_flat(self, plan):
        """Use the train plan's flat parameter / gradient buffers: one kernel launch per step.  Existing per-parameter state
        (a loaded checkpoint, or steps already taken one by one) is COPIED into the flat moment buffers, so attaching before or
        after ``load_state_dict`` keeps the optimizer state."""
        pflat = plan.flatten_parameters()
        m, v = torch.zeros_like(pflat), torch.zeros_like(pflat)
        step = 0
        for p in plan.param_order:
            st = self.state.get(p)
            if st:
                off = plan._goff[id(p)]
                m[off:off + p.numel()].copy_(st["exp_avg"].reshape(-1))
                v[off:off + p.numel()].copy_(st["exp_avg_sq"].reshape(-1))
                step = max(step, int(float(st["step"])))
        self._flat = dict(plan=plan, p=pflat, m=m, v=v, step=step)
        step_t = torch.tensor(float(step))
        for p in plan.param_order:
            off = plan._goff[id(p)]
            st = self.state[p]
            st["step"] = step_t
            st["exp_avg"] = m[off:off + p.numel()].view(p.shape)
            st["exp_avg_sq"] = v[off:off + p.numel()].view(p.shape)

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
            b1, b2 = group["betas"]
            nat.call("wsr_adam_step", f["p"].data_ptr(), plan.gflat.data_ptr(), f["m"].data_ptr(), f["v"].data_ptr(), f["p"].numel(),
                     float(group["lr"]), float(b1), float(b2), float(group["eps"]), float(group["weight_decay"]), int(f["step"]),
                     torch.cuda.current_stream(f["p"].device).cuda_stream)
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
        b1, b2 = group["betas"]
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
            nat.call("wsr_adam_step", p.data_ptr(), g.data_ptr(), st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr(), p.numel(),
                     float(group["lr"]), float(b1), float(b2), float(group["eps"]), float(group["weight_decay"]),
                     int(st["step"].item()), torch.cuda.current_stream(p.device).cuda_stream)
