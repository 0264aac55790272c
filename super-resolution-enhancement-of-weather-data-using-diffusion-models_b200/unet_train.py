"""UNetTrainPlan -- forward + backward launch schedule of the ResDiff denoiser for the training step
(reference models/diffusion_models/model.py:61-69: loss -> ``backward()`` through resdiff/unet.py:121-177).

The forward is ``UNetPlan.run`` with the training-mode dropout of ``Block`` (nn_modules/resnet.py:23).  Every forward
buffer is distinct, so all activations needed by the backward pass are still resident when it starts; the backward is
a second fixed sequence of C-ABI calls:

  * data gradients of the convolutions run on the FORWARD convolution kernels with transposed / flipped weights
    (``taps.py``): tcgen05 in bf16 mode, SIMT in the fp32 check mode;
  * weight / bias gradients: ``wsr_conv_wgrad_simt`` writes straight into the reference's OIHW layout;
  * GroupNorm + Swish (+ dropout) backward: ``wsr_gn_bwd_reduce`` / ``wsr_gn_bwd_apply``; the per-image column sums
    that feed the FeatureWiseAffine linears (resnet.py:145-157) come out of the same kernel in closed form;
  * attention backward: recompute S, P with the GEMM + softmax kernels, then five GEMMs and ``wsr_softmax_bwd_rows``;
  * noise-level MLP, the 27 stacked FeatureWiseAffine linears, the FD_Info_Spliter gate and its FFT branch.

Parameter gradients live in ONE flat fp32 buffer (``gflat``) laid out in the order in which the backward pass finishes
them, so a data-parallel trainer can all-reduce contiguous buckets while the rest of the backward is still running
(``on_ready`` callback).  ``param_grads()`` maps every ``nn.Parameter`` to its view of that buffer.
"""
import ctypes
import functools
import math

import torch

from . import _native as nat
from . import taps as T
from .engine import Act
from .unet_plan import UNetPlan, _L


class UNetTrainPlan(UNetPlan):
    feeds_backward = True

    def __init__(self, net, batch, device, precision="bf16", strict_tc=False):
        self.drop_p = float(getattr(net, "dropout", 0.0) or 0.0)
        self.drop_seed = 0
        self.on_ready = None           # callback(lo, hi): gflat[lo:hi] is final (launch its all-reduce now)
        self._dw = None
        # Launch lists: a training step issues ~1100 kernel launches whose arguments (device pointers, descriptors, tap
        # tables) never change, while building them in Python costs ~30 us each -- more than the GPU needs to execute
        # them at batch 4.  The forward and the backward schedule are therefore RECORDED once (Engine.rec) and replayed
        # with ~2 us per launch; the only per-step value, the dropout seed, lives in a shared ctypes object.
        self._seed = ctypes.c_uint64(0)
        self._lists = {}
        self._n_bwd = 0
        self.replay_enabled = True
        self._jobtab = None            # (device WsrPackJob table, njobs, total units, parameter-address signature)
        self.batched_refresh = True     # False: re-pack weights tensor by tensor (the reference the tests compare with)
        super().__init__(net, batch, device, precision, strict_tc)
        self._grad_layout()
        self._grad_buffers()

    # ------------------------------------------------------------------------------------------------------------------
    # forward: dropout in block2
    # ------------------------------------------------------------------------------------------------------------------
    def _block2_norm(self, r):
        if self.drop_p > 0.0 and self.train_mode:
            self.eng.gn_apply_dropout(r.hbuf, r.g2, r.b2, self.groups, nat.ACT_SWISH, r.a2, self.drop_p, self._seed, r.drop_tag)
        else:
            self.eng.gn_apply(r.hbuf, r.g2, r.b2, self.groups, nat.ACT_SWISH, r.a2)

    train_mode = True

    def _res_records(self):
        return [r for r in list(self.downs) + list(self.mids) + list(self.ups) if r.kind == "res"]

    # ------------------------------------------------------------------------------------------------------------------
    # flat gradient buffer, in completion order of the backward pass
    # ------------------------------------------------------------------------------------------------------------------
    def _grad_layout(self):
        net = self.net
        order = []          # parameters in the order their gradients become final

        def add(*ps):
            for p in ps:
                if p is not None:
                    order.append(p)

        def res_params(r):
            rb = r.mod.res_block
            if r.attn:
                at = r.mod.attn
                add(at.out.weight, at.out.bias, at.qkv.weight, at.norm.weight, at.norm.bias)
            add(rb.block2.block[3].weight, rb.block2.block[3].bias)
            if r.has_res_conv:
                add(rb.res_conv.weight, rb.res_conv.bias)
            add(rb.block2.block[0].weight, rb.block2.block[0].bias, rb.block1.block[3].weight, rb.block1.block[3].bias,
                rb.block1.block[0].weight, rb.block1.block[0].bias)

        fc = net.final_conv.block
        add(fc[3].weight, fc[3].bias, fc[0].weight, fc[0].bias)
        self._marks = []                  # (number of parameters finished, label) after each stage
        for r in reversed(self.ups):
            if r.kind == "res":
                res_params(r)
            else:
                add(r.mod.conv.weight, r.mod.conv.bias)
        self._marks.append(len(order))
        for r in reversed(self.mids):
            res_params(r)
        self._marks.append(len(order))    # most parameters sit in the up path, the mid blocks and the two deepest levels: a mark after each
        for r in reversed(self.downs[1:]):   # lets their all-reduce start while the shallow, parameter-poor levels are still being walked
            if r.kind == "res":
                res_params(r)
            else:
                if self.has_hfca:
                    m = r.ca.mod
                    add(m.out.weight, m.out.bias, m.kv.weight, m.q.weight, m.norm.weight, m.norm.bias)
                add(r.mod.conv.weight, r.mod.conv.bias)
                self._marks.append(len(order))
        if self._marks[-1] != len(order):
            self._marks.append(len(order))
        stem = self.downs[0].mod
        add(stem.weight, stem.bias)
        if self.kind == "srdiff":
            add(net.cond_proj.weight, net.cond_proj.bias)
        fd = getattr(net, "fd_spliter", None)
        if fd is not None:
            add(fd.noise_resSE.fc[0].weight, fd.noise_resSE.fc[2].weight, fd.sigma_resSE.fc[0].weight, fd.sigma_resSE.fc[2].weight,
                fd.HF_guided_resSE.fc[0].weight, fd.HF_guided_resSE.fc[2].weight, fd.channel_transform.weight, fd.channel_transform.bias)
        # the stacked FeatureWiseAffine linears: weights, then biases, in projection order (= rows of proj_w / proj_b)
        lins = [r.mod.res_block.noise_func.noise_func[0] for r in self._res_records()] + ([fd.noise_func] if fd is not None else [])
        proj_w_first = len(order)
        add(*[l.weight for l in lins])
        proj_b_first = len(order)
        add(*[l.bias for l in lins])
        mlp = net.noise_level_mlp
        add(mlp[1].weight, mlp[1].bias, mlp[3].weight, mlp[3].bias)

        seen = set()
        for p in order:
            assert id(p) not in seen, "parameter listed twice"
            seen.add(id(p))
        missing = [n for n, p in net.named_parameters() if id(p) not in seen]
        assert not missing, "parameters without a gradient slot: %s" % missing[:5]
        self.param_order = order
        offs, off = {}, 0
        for p in order:
            offs[id(p)] = off
            off += (p.numel() + 3) // 4 * 4          # keep every view 16-byte aligned
        self.gflat = torch.zeros(off, device=self.eng.device, dtype=torch.float32)
        self._goff = offs
        self._gview = {id(p): self.gflat[offs[id(p)]:offs[id(p)] + p.numel()].view(p.shape) for p in order}
        # the projection weights / biases are contiguous blocks (no padding needed: cout*inner and cout are multiples of 4)
        self.dproj_w = self.gflat[offs[id(order[proj_w_first])]:offs[id(order[proj_w_first])] + self.P * self.inner].view(self.P, self.inner)
        self.dproj_b = self.gflat[offs[id(order[proj_b_first])]:offs[id(order[proj_b_first])] + self.P]
        assert all(l.weight.numel() % 4 == 0 and l.bias.numel() % 4 == 0 for l in lins)
        self._mark_offsets = [offs[id(order[m])] if m < len(order) else off for m in self._marks]

    def gv(self, p):
        return self._gview[id(p)]

    def flatten_parameters(self):
        """Re-point every parameter's storage into one flat fp32 buffer with the same layout as ``gflat`` (values are
        preserved), so that the optimizer update is a single launch.  Idempotent."""
        if self.parameters_are_flat():
            return self._pflat
        pflat = torch.zeros_like(self.gflat)
        with torch.no_grad():
            for p in self.param_order:
                off = self._goff[id(p)]
                view = pflat[off:off + p.numel()].view(p.shape)
                view.copy_(p.data)
                p.data = view
        self._pflat = pflat
        self._wver = None
        # the packed buffers, the job table and the launch lists were keyed on the old parameter addresses
        self.eng._pack_cache.clear()
        self._jobtab = None
        self._lists.clear()
        return pflat

    def parameters_are_flat(self):
        pf = getattr(self, "_pflat", None)
        if pf is None:
            return False
        base = pf.data_ptr()
        return all(p.data_ptr() == base + 4 * self._goff[id(p)] for p in self.param_order)

    def param_grads(self):
        """[(parameter, fp32 gradient view into gflat)] in completion order."""
        return [(p, self._gview[id(p)]) for p in self.param_order]

    # ------------------------------------------------------------------------------------------------------------------
    # gradient buffers of the activations
    # ------------------------------------------------------------------------------------------------------------------
    def _grad_buffers(self):
        e, B = self.eng, self.B
        self._gbuf = {}
        self._gtensors = []
        self._garena = None
        red = self._red_sizes = []

        def gn_slot(c):
            off = sum(red)
            red.append(B * 2 * c)
            return off

        for i, r in enumerate(self._res_records()):
            r.drop_tag = i + 1
            r.red1, r.red2 = gn_slot(r.cin), gn_slot(r.cout)
            if r.attn:
                r.red3 = gn_slot(r.cout)
                r.dvT = e.empty(tuple(r.vT.shape))
        for ca in self.hfca:
            ca.red = gn_slot(ca.c)
            ca.dvT = e.empty(tuple(ca.vT.shape))
        self.red_final = gn_slot(self.final_cin)
        self.red = torch.zeros(max(sum(red), 1), device=e.device, dtype=torch.float64)
        n = self.scores.numel() if self.scores is not None else 0
        self.dP = e.empty((n,), torch.float32) if n else None
        self.dS = e.empty((n,)) if n else None
        self.dproj = torch.zeros((B, self.P), device=e.device, dtype=torch.float32)
        self.dtemb = e.empty((B, self.inner), torch.float32)
        self.deps = e.new_act(B, self.H, self.W, self.C_img)
        self.deps_in = e.empty((B, self.C_img, self.H, self.W), torch.float32)
        if self.kind == "resdiff":
            self.dxin = e.new_act(B, self.H, self.W, 5 * self.C_img, dt=nat.F32)
            self.g_lf = e.empty((B, self.C_img, self.H, self.W), torch.float32)
            self.g_hf = e.empty((B, self.C_img, self.H, self.W), torch.float32)
            nb = nat.call("wsr_fd_backward_workspace_bytes", B, self.C_img, self.H, self.W)
            self.fd_bwork = e.empty((nb,), torch.uint8)

    def G(self, a):
        """Gradient buffer mirroring the activation slice ``a`` (same geometry; created on first use, zeroed per step)."""
        key = a.buf.data_ptr()
        g = self._gbuf.get(key)
        if g is None:
            g = torch.zeros_like(a.buf)
            self._garena = None        # a late buffer lives outside the arena: fall back to per-buffer clearing
            self._gbuf[key] = g
            self._gtensors.append(g)
        return Act(g, a.N, a.H, a.W, a.C, a.ld, a.coff, a.dt)

    # ------------------------------------------------------------------------------------------------------------------
    # weights: forward packs + data-gradient packs
    # ------------------------------------------------------------------------------------------------------------------
    def refresh_weights(self):
        """Re-pack every forward and data-gradient weight from the fp32 parameters.  The first call goes through the
        per-tensor pack entry points and records a WsrPackJob table; as long as the parameters keep their addresses, later
        calls (after every optimizer step) are ONE ``wsr_repack_batch`` launch writing the same destination buffers."""
        v = self._weights_version()
        if v == self._wver:
            return
        e = self.eng
        sig = tuple(p.data_ptr() for p in self.net.parameters())
        if self._jobtab is not None and self._jobtab[3] == sig and self.batched_refresh:
            tab, n, total, _ = self._jobtab
            e.call("wsr_repack_batch", tab.data_ptr(), n, total, e.stream)
            self._wver = v
            self.proj_table = None
            return
        e.jobs, e.jobs_ok = [], True
        try:
            self._refresh_eager()
            if e.jobs_ok and e.jobs:
                self._jobtab = e.job_table() + (sig,)
            else:
                self._jobtab = None
        finally:
            e.jobs = None

    def _refresh_eager(self):
        super().refresh_weights()
        e = self.eng
        with torch.no_grad():
            def dg(weight):
                return e.pack_conv(T.dgrad_weight(weight), None, key=("dgrad",) + e._src_key(weight), src=(weight.data_ptr(), 1))

            for r in self._res_records():
                rb = r.mod.res_block
                r.dconv1, r.dconv2 = dg(rb.block1.block[3].weight), dg(rb.block2.block[3].weight)
                if r.has_res_conv:
                    r.dresw = dg(rb.res_conv.weight)
                if r.attn:
                    at = r.mod.attn
                    cc = r.cout
                    r.dwqk = dg(at.qkv.weight[:2 * cc])
                    r.dwout = dg(at.out.weight)
                    r.wv_f = e.pack_rows(at.qkv.weight[2 * cc:].reshape(cc, cc))
            for r in self.downs:
                if r.kind == "stem":
                    r.dconv = dg(r.mod.weight)
                elif r.kind == "down":
                    r.dconv = dg(r.mod.conv.weight)
                    if self.has_hfca:
                        m = r.ca.mod
                        r.ca.dwk = dg(m.kv.weight[:r.ca.c])
                        r.ca.dwout = dg(m.out.weight)
            for r in self.ups:
                if r.kind == "up":
                    w = r.mod.conv.weight
                    r.dconv = e.pack_conv(T.upsample_dgrad_weight(w), None, key=("updgrad",) + e._src_key(w),
                                          src=(w.data_ptr(), 1), job_kind=nat.PACK_UPSAMPLE_DGRAD)
            self.dfinal = dg(self.net.final_conv.block[3].weight)
            if self.kind == "srdiff":
                # data gradient of cond_proj (joint training of the encoder): its OIHW weight is the parameter itself
                cp = self.net.cond_proj
                self.cond_dgrad_pc = e.pack_conv(cp.weight, None, key=("cond_dgrad",) + e._src_key(cp.weight))
        e._keep.clear()

    # ------------------------------------------------------------------------------------------------------------------
    # backward building blocks
    # ------------------------------------------------------------------------------------------------------------------
    # ---- weight-gradient side stream ---------------------------------------------------------------------------------
    # Nothing in the backward chain waits for a weight gradient: dW / db of a layer only feed the optimizer (and the gradient
    # all-reduce), while the chain itself is data gradient -> GroupNorm backward -> data gradient ...  At the reference's batch of 4
    # per GPU every one of these ~900 launches is far too small to fill 148 SMs, so the weight-gradient launches (a third of the
    # step's kernel time) go to a second stream and run BESIDE the chain: fork = the side stream waits for everything the main
    # stream has issued so far (x and dy of the layer are final by then and are not written again during this backward), join =
    # the main stream waits for the side stream before a gradient range is handed to the all-reduce / optimizer.  Both are host
    # callbacks in the recorded launch list, so replays fork and join exactly like the recording run.
    def _wstream(self):
        if not hasattr(self, "_wside"):
            on = self.eng.device.type == "cuda"
            self._wside = torch.cuda.Stream(device=self.eng.device) if on else None
            self._wev_fork = torch.cuda.Event() if on else None
            self._wev_join = torch.cuda.Event() if on else None
            self._wforked = False
        return self._wside

    def _host(self, fn):
        """Run a host callback now and at the same place in every replay of the launch list being recorded."""
        if self.eng.rec is not None:
            self.eng.rec.append((None, fn, "host"))
        fn()

    def _wfork_fire(self, src=None):
        # src: the stream the launches being forked from were issued on when that is NOT the caller's current stream (the HF-CA branch
        # stream below); replays run these callbacks with the main stream current
        self._wev_fork.record(src if src is not None else torch.cuda.current_stream(self.eng.device))
        self._wside.wait_event(self._wev_fork)
        self._wforked = True

    def _wjoin_fire(self, final):
        # the chain itself joins the side stream only at the end of the backward pass; gradient ranges handed to the bucketed all-reduce
        # earlier are ordered after the side stream without blocking the chain (_ready_fire)
        if self._wforked and final:
            self._wev_join.record(self._wside)
            torch.cuda.current_stream(self.eng.device).wait_event(self._wev_join)
            self._wforked = False

    def _wjoin(self, final):
        if self._wstream() is not None:
            self._host(functools.partial(self._wjoin_fire, final))

    def _on_side(self, launch):
        """Issue ``launch()`` on the weight-gradient stream (after everything the main stream has issued so far)."""
        side = self._wstream()
        if side is None or self.eng.prof is not None:      # per-launch event timing brackets launches on the main stream
            launch()
            return
        cur = torch.cuda.current_stream(self.eng.device)
        src = cur if (getattr(self, "_hside", None) is not None and cur == self._hside) else None
        self._host(functools.partial(self._wfork_fire, src))
        with torch.cuda.stream(side):
            launch()

    # ---- HF-guided cross-attention backward on a third stream ------------------------------------------------------------
    # HF_guided_CA only produces SKIP tensors (resdiff/unet.py:156-163), so the gradient of its output is final as soon as the up path
    # has been walked back, while its own gradient (into the down-path feature it read) is only needed when the backward pass reaches
    # that Downsample again -- half a pass later.  In between sits the most expensive single piece of the step, the N = 8192 attention
    # backward through four (B, 8192, 8192) matrices.  The branches therefore run on their own stream from the end of the up path on
    # (deepest level first, the order in which the chain will ask for them), each into a private dx buffer and private attention
    # scratch; the chain joins a branch where it used to compute it and adds the private dx.
    def _hstream(self):
        if not hasattr(self, "_hside"):
            on = self.eng.device.type == "cuda" and self.has_hfca and self.scores is not None
            if on:
                # the branch needs its own (B, N, N) scratch set (3.2 GB at batch 4): beyond 8 GB the batch is large enough to fill the
                # machine without the overlap, and the memory is better left to the activations
                extra = sum(t.numel() * t.element_size() for t in (self.scores, self.probs, self.dP, self.dS))
                on = extra <= 8 * (1 << 30)
            self._hside = torch.cuda.Stream(device=self.eng.device) if on else None
            if on:
                e = self.eng
                self._hscratch = (torch.empty_like(self.scores), torch.empty_like(self.probs), torch.empty_like(self.dP), torch.empty_like(self.dS))
                self._hev_fork = torch.cuda.Event()
                for ca in self.hfca:
                    ca.dx_side = e.new_act(self.B, ca.h, ca.w, ca.c)
                    ca.ev_done = torch.cuda.Event()
        return self._hside

    def _hfork_fire(self):
        self._hev_fork.record(torch.cuda.current_stream(self.eng.device))
        self._hside.wait_event(self._hev_fork)

    def _hdone_fire(self, ca):
        ca.ev_done.record(self._hside)

    def _hjoin_fire(self, ca):
        torch.cuda.current_stream(self.eng.device).wait_event(ca.ev_done)

    def _hf_ca_bwd_all_on_side(self, order):
        """Issue the backward of every HF-CA branch in ``order`` on the branch stream; returns False when the stream is off."""
        side = self._hstream()
        if side is None or self.eng.prof is not None:
            return False
        self._host(self._hfork_fire)
        with torch.cuda.stream(side):
            for ca in order:
                self._hf_ca_bwd(ca, dx=ca.dx_side, scratch=self._hscratch)
                self._host(functools.partial(self._hdone_fire, ca))
        return True

    def _wgrad(self, x, dy, conv_mod, taps, up=1, rows=None, bias=True):
        """Weight (+ bias) gradient of ``conv_mod`` (an nn.Conv2d) straight into its OIHW gradient view.
        rows = (lo, hi): only output channels [lo, hi) of the module (split qkv / kv projections)."""
        w = conv_mod.weight
        co, ci, kh, kw = w.shape
        gw = self.gv(w)
        lo, hi = rows if rows is not None else (0, co)
        view = gw[lo:hi]
        assert dy.C == hi - lo and x.C >= ci
        xs = x if x.C == ci else x.slice(0, ci)
        gb = None
        if bias and conv_mod.bias is not None:
            gb = self.gv(conv_mod.bias)[lo:hi]
        self._on_side(lambda: self.eng.wgrad(xs, dy, taps, view, (1, ci * kh * kw, kh * kw), gb, up))

    def _gn_bwd(self, x, gn_mod, act, da, dx, red_off, colsum=0, colsum_ld=0, drop=(0.0, 0, 0), gamma=None, beta=None, groups=None):
        self.eng.gn_bwd(x, gamma, beta, groups or self.groups, act, da, dx, self.red.data_ptr() + 8 * red_off,
                        self.gv(gn_mod.weight), self.gv(gn_mod.bias), True, colsum, colsum_ld, drop)

    def _attention_bwd(self, q, k, vT, do, dq, dk, dvT, scratch=None):
        """Backward of o = softmax(q k^T / sqrt(C)) v (nn_modules/resnet.py:90-97, guided_cross_attention.py:34-41).
        q, k, do, dq, dk: Acts (B, ., ., C); vT, dvT: (B, C, Nk) tensors.  dq / dk are written (not accumulated)."""
        e, B = self.eng, self.B
        Nq, Nk, Cc = q.H * q.W, k.H * k.W, q.C
        scale = 1.0 / math.sqrt(Cc)
        n = B * Nq * Nk
        S, P, dP, dS = (t[:n] for t in (scratch or (self.scores, self.probs, self.dP, self.dS)))
        s_dt = nat.BF16 if S.dtype == torch.bfloat16 else nat.F32
        p_dt = nat.BF16 if P.dtype == torch.bfloat16 else nat.F32
        ds_dt = nat.BF16 if dS.dtype == torch.bfloat16 else nat.F32
        e.gemm(q.ptr, q.dt, (Nq * q.ld, q.ld, 1), k.ptr, k.dt, (Nk * k.ld, k.ld, 1), S.data_ptr(), s_dt, (Nq * Nk, Nk, 1), B, Nq, Nk, Cc)
        e.softmax(S, s_dt, B * Nq, Nk, scale, P, p_dt)
        # dvT[c][j] = sum_i do[i][c] P[i][j]
        e.gemm(do.ptr, do.dt, (Nq * do.ld, 1, do.ld), P.data_ptr(), p_dt, (Nq * Nk, 1, Nk), dvT.data_ptr(), e.dt, (Cc * Nk, Nk, 1),
               B, Cc, Nk, Nq)
        # dP[i][j] = sum_c do[i][c] vT[c][j]
        e.gemm(do.ptr, do.dt, (Nq * do.ld, do.ld, 1), vT.data_ptr(), e.dt, (Cc * Nk, 1, Nk), dP.data_ptr(), nat.F32, (Nq * Nk, Nk, 1),
               B, Nq, Nk, Cc)
        e.softmax_bwd(P, p_dt, dP, nat.F32, B * Nq, Nk, scale, dS, ds_dt)
        # dq[i][c] = sum_j dS[i][j] k[j][c] ;  dk[j][c] = sum_i dS[i][j] q[i][c]
        e.gemm(dS.data_ptr(), ds_dt, (Nq * Nk, Nk, 1), k.ptr, k.dt, (Nk * k.ld, 1, k.ld), dq.ptr, dq.dt, (Nq * dq.ld, dq.ld, 1),
               B, Nq, Cc, Nk)
        e.gemm(dS.data_ptr(), ds_dt, (Nq * Nk, 1, Nk), q.ptr, q.dt, (Nq * q.ld, 1, q.ld), dk.ptr, dk.dt, (Nk * dk.ld, dk.ld, 1),
               B, Nk, Cc, Nq)

    def _v_bwd(self, wv_packed, nact, dvT, dn, dw_rows):
        """v^T = Wv n^T  ->  dn[pix][k] += sum_c dvT[c][pix] Wv[c][k];  dWv[c][k] += sum_{b,pix} dvT[b][c][pix] n[b][pix][k]."""
        e, B = self.eng, self.B
        cc, n = wv_packed.shape[0], nact.H * nact.W
        e.gemm(dvT.data_ptr(), e.dt, (cc * n, 1, n), wv_packed.data_ptr(), e.dt, (0, 1, cc), dn.ptr, dn.dt, (n * dn.ld, dn.ld, 1),
               B, n, cc, cc, res=(dn.ptr, dn.dt, (n * dn.ld, dn.ld, 1)))
        es = 2 if e.dt == nat.BF16 else 4

        def dw_launches():
            for b in range(B):
                e.gemm(dvT.data_ptr() + b * cc * n * es, e.dt, (0, n, 1), nact.ptr + b * n * nact.ld * es, nact.dt, (0, 1, nact.ld),
                       dw_rows.data_ptr(), nat.F32, (0, cc, 1), 1, cc, cc, n, res=(dw_rows.data_ptr(), nat.F32, (0, cc, 1)))
        self._on_side(dw_launches)

    def _res_block_bwd(self, r, x):
        """Backward of UNetPlan._res_block; reads G(r.y), accumulates into G(x)."""
        e, B, G = self.eng, self.B, self.G
        SW = nat.ACT_SWISH
        rb = r.mod.res_block
        taps3 = T.forward_taps(3, 1, r.h, r.w)
        taps1 = T.forward_taps(1, 1, r.h, r.w)
        dy = G(r.y)
        if r.attn:
            at = r.mod.attn
            cc = r.cout
            d_rbuf, d_o, d_qk, d_n = G(r.rbuf), G(r.obuf), G(r.qk), G(r.nbuf)
            # y = out(o) + rbuf
            e.conv(dy, r.dwout, d_o, bias=False)
            self._wgrad(r.obuf, dy, at.out, taps1)
            e.call("wsr_axpby", dy.ptr, dy.dt, dy.ld, 1.0, d_rbuf.ptr, d_rbuf.dt, d_rbuf.ld, 1.0, d_rbuf.ptr, d_rbuf.dt, d_rbuf.ld,
                   B * r.h * r.w, cc, e.stream)
            self._attention_bwd(r.qk.slice(0, cc), r.qk.slice(cc, cc), r.vT, d_o, d_qk.slice(0, cc), d_qk.slice(cc, cc), r.dvT)
            e.conv(d_qk, r.dwqk, d_n, bias=False)
            self._wgrad(r.nbuf, d_qk, at.qkv, taps1, rows=(0, 2 * cc), bias=False)
            self._v_bwd(r.wv_f, r.nbuf, r.dvT, d_n, self.gv(at.qkv.weight)[2 * cc:].view(cc, cc))
            self._gn_bwd(r.rbuf, at.norm, nat.ACT_NONE, d_n, d_rbuf, r.red3, gamma=r.g3, beta=r.b3)
            dy = d_rbuf
        # dst = conv2(a2) + (res_conv(x) | x)
        d_a2, d_h, d_a1, dx = G(r.a2), G(r.hbuf), G(r.a1), G(x)
        e.conv(dy, r.dconv2, d_a2, bias=False)
        self._wgrad(r.a2, dy, rb.block2.block[3], taps3)
        if r.has_res_conv:
            e.conv(dy, r.dresw, dx, bias=False, res=dx)
            self._wgrad(x, dy, rb.res_conv, taps1)
        else:
            e.call("wsr_axpby", dy.ptr, dy.dt, dy.ld, 1.0, dx.ptr, dx.dt, dx.ld, 1.0, dx.ptr, dx.dt, dx.ld, B * r.h * r.w, r.cout, e.stream)
        # a2 = dropout(swish(GN2(h)));  h = conv1(a1) + bias + proj[b]
        drop = (self.drop_p, self._seed, r.drop_tag) if (self.drop_p > 0.0 and self.train_mode) else (0.0, 0, 0)
        self._gn_bwd(r.hbuf, rb.block2.block[0], SW, d_a2, d_h, r.red2, colsum=self.dproj.data_ptr() + 4 * r.proj_off,
                     colsum_ld=self.P, drop=drop, gamma=r.g2, beta=r.b2)
        e.conv(d_h, r.dconv1, d_a1, bias=False)
        self._wgrad(r.a1, d_h, rb.block1.block[3], taps3)
        self._gn_bwd(x, rb.block1.block[0], SW, d_a1, dx, r.red1, gamma=r.g1, beta=r.b1)

    def _hf_ca_bwd(self, ca, dx=None, scratch=None):
        """Backward of UNetPlan._hf_ca; reads G(ca.y), accumulates into G(ca.x) -- or, dx given, WRITES the branch's gradient w.r.t.
        ca.x into that private buffer (branch stream: the chain adds it to G(ca.x) at the join)."""
        e, B, G = self.eng, self.B, self.G
        m = ca.mod
        cc = ca.c
        taps1 = T.forward_taps(1, 1, ca.h, ca.w)
        dy = G(ca.y)
        private = dx is not None
        if not private:
            dx = G(ca.x)
        d_o, d_k, d_q, d_n = G(ca.obuf), G(ca.kbuf), G(ca.q), G(ca.nbuf)
        e.conv(dy, ca.dwout, d_o, bias=False)
        self._wgrad(ca.obuf, dy, m.out, taps1)
        if private:      # dx = dy (z = dy with weight 0: never reads what the private buffer held)
            e.call("wsr_axpby", dy.ptr, dy.dt, dy.ld, 1.0, dy.ptr, dy.dt, dy.ld, 0.0, dx.ptr, dx.dt, dx.ld, B * ca.h * ca.w, cc, e.stream)
        else:
            e.call("wsr_axpby", dy.ptr, dy.dt, dy.ld, 1.0, dx.ptr, dx.dt, dx.ld, 1.0, dx.ptr, dx.dt, dx.ld, B * ca.h * ca.w, cc, e.stream)
        self._attention_bwd(ca.q, ca.kbuf, ca.vT, d_o, d_q, d_k, ca.dvT, scratch=scratch)
        self._wgrad(ca.qimg, d_q, m.q, taps1, bias=False)
        e.conv(d_k, ca.dwk, d_n, bias=False)
        self._wgrad(ca.nbuf, d_k, m.kv, taps1, rows=(0, cc), bias=False)
        self._v_bwd(ca.wv, ca.nbuf, ca.dvT, d_n, self.gv(m.kv.weight)[cc:].view(cc, cc))
        self._gn_bwd(ca.x, m.norm, nat.ACT_NONE, d_n, dx, ca.red, gamma=ca.g, beta=ca.b, groups=32)

    def _ready(self):
        """The gradient range that ends at the next mark is final (call order = order of ``self._marks``, then the tail)."""
        mark = self._mark_i
        self._mark_i += 1
        assert mark <= len(self._marks)
        final = mark == len(self._marks)
        if final:
            self._wjoin(True)          # end of the pass: the optimizer reads every gradient
        if self.eng.rec is not None:
            self.eng.rec.append((None, functools.partial(self._ready_fire, mark, final), "on_ready"))
        self._ready_fire(mark, final)

    def _ready_fire(self, mark, final=True):
        if self.on_ready is None:
            return
        lo = 0 if mark == 0 else self._mark_offsets[mark - 1]
        hi = self._mark_offsets[mark] if mark < len(self._mark_offsets) else self.gflat.numel()
        if hi <= lo:
            return
        side = getattr(self, "_wside", None)
        if final or side is None or not self._wforked:
            self.on_ready(lo, hi)
            return
        # The range's weight gradients may still be running on the side stream.  Making the chain wait for them here would serialise
        # the two streams at every mark (measured: 1.3 -> 2.0 ms of exposed all-reduce with 7 marks); instead a third stream waits for
        # BOTH and the hook -- whose collectives order themselves after the stream they are issued from -- is called on it.
        if not hasattr(self, "_rsync"):
            self._rsync = torch.cuda.Stream(device=self.eng.device)
            self._rev_m, self._rev_s = torch.cuda.Event(), torch.cuda.Event()
        self._rev_m.record(torch.cuda.current_stream(self.eng.device))
        self._rev_s.record(side)
        self._rsync.wait_event(self._rev_m)
        self._rsync.wait_event(self._rev_s)
        with torch.cuda.stream(self._rsync):
            self.on_ready(lo, hi)

    # ------------------------------------------------------------------------------------------------------------------
    # the backward pass
    # ------------------------------------------------------------------------------------------------------------------
    def backward(self, d_eps):
        """d_eps: (B, C_img, H, W) fp32 gradient of the loss w.r.t. ``self.eps``.  Fills ``gflat`` (all parameter
        gradients of this step; the buffer is overwritten, accumulation across steps is the caller's business)."""
        e = self.eng
        self.deps_in.copy_(d_eps.to(torch.float32))
        self._n_bwd += 1
        key = ("bwd", self.train_mode, getattr(self, "want_cond_grad", False), self._ptr_sig())
        if self.replay_enabled and self._lists.get("bwd_key") == key:
            e.replay(self._lists["bwd"])
            return self.gflat
        # the first call creates the activation-gradient buffers lazily (their memsets are not in its launch sequence):
        # record from the second call on
        record = self.replay_enabled and self._n_bwd >= 2
        if record:
            e.rec = []
        try:
            self._backward_body(self.deps_in)
        finally:
            lst, e.rec = e.rec, None
        if record:
            self._lists["bwd"], self._lists["bwd_key"] = lst, key
        elif self._garena is None and self._gtensors:
            self._consolidate_gbufs()
        return self.gflat

    def _cond_grad_launches(self, gy):
        """SRDiff with a trainable encoder (``lock_weights=False``, srdiff_diffusion.py:212-214): gradient of the loss w.r.t. the
        condition cat(feas[2::3]) (B, 384, h, w).  cond_up = ConvTranspose2d(k8, s4, p2)(cond) was added to the output of downs[2], so
        d cond[n, ci, i, j] = sum_{co, ky, kx} dY[n, co, 4i + ky - 2, 4j + kx - 2] W[ci, co, ky, kx]: a stride-4 8x8 convolution over dY
        whose OIHW weight IS the transposed convolution's (in, out, 8, 8) parameter, run as four 16-tap launches on the tap tables the
        weight gradient already uses.  Part of the backward launch sequence (and of its recorded list)."""
        e = self.eng
        cp = self.net.cond_proj
        pc = self.cond_dgrad_pc                      # packed with the other backward weights (refresh_weights)
        cf = self.cond_feat
        if getattr(self, "_dcond", None) is None:
            self._dcond = e.new_act(self.B, cf.H, cf.W, cf.C)
        for q, tp in enumerate(T.conv_transpose_k8s4_wgrad_taps(cf.H, cf.W)):
            e.conv(gy, pc, self._dcond, taps=tp, bias=False, res=self._dcond if q else None, force_simt=True)

    def cond_grad(self):
        """(B, 384, h, w) fp32 NCHW gradient w.r.t. the condition, computed by the last ``backward`` (``want_cond_grad`` set)."""
        assert self.kind == "srdiff" and getattr(self, "_dcond", None) is not None
        return self._dcond.to_nchw(self.eng)

    def _consolidate_gbufs(self):
        """After the first backward pass every activation-gradient buffer exists: move them into ONE arena so that the
        per-step clearing is a single memset instead of ~150."""
        sizes = [(g.numel() * g.element_size() + 255) // 256 * 256 for g in self._gtensors]
        arena = torch.zeros((sum(sizes),), device=self.eng.device, dtype=torch.uint8)
        new, off = {}, 0
        old_to_new = {}
        for g, nb in zip(self._gtensors, sizes):
            v = arena[off:off + g.numel() * g.element_size()].view(g.dtype).view(g.shape)
            old_to_new[g.data_ptr()] = v
            off += nb
        for key, g in self._gbuf.items():
            new[key] = old_to_new[g.data_ptr()]
        self._gbuf = new
        self._gtensors = list(new.values())
        self._garena = arena

    def _fd_bwd(self, dy):
        """Backward of FD_Info_Spliter (fd_info_spliter.py:37-117) from the gradient of the stem convolution's output."""
        e, B = self.eng, self.B
        st = e.stream
        net = self.net
        stem = self.downs[0]
        C = self.C_img
        e.conv(dy, stem.dconv, self.dxin, bias=False)
        fd = net.fd_spliter
        e.call("wsr_fd_gate_bwd", self.dxin.ptr, self.dxin.dt, self.dxin.ld, 2 * C, self.x_t.data_ptr(),
               self.cur_proj.data_ptr() + 4 * self.ne_off, self.P, B, C, self.H, self.W, self.fd_n0.data_ptr(), self.fd_n2.data_ptr(),
               self.fd_hidden, self.dproj.data_ptr() + 4 * self.ne_off, self.P, self.gv(fd.noise_resSE.fc[0].weight).data_ptr(),
               self.gv(fd.noise_resSE.fc[2].weight).data_ptr(), st)
        e.call("wsr_nhwc_to_nchw", self.dxin.ptr + 4 * 3 * C, nat.F32, self.dxin.ld, B, C, self.H, self.W, self.g_lf.data_ptr(), st)
        e.call("wsr_nhwc_to_nchw", self.dxin.ptr + 4 * 4 * C, nat.F32, self.dxin.ld, B, C, self.H, self.W, self.g_hf.data_ptr(), st)
        e.call("wsr_fd_backward", self.cond.data_ptr(), B, C, self.H, self.W, self.fd_s0.data_ptr(), self.fd_s2.data_ptr(),
               self.fd_h0.data_ptr(), self.fd_h2.data_ptr(), self.fd_ctw.data_ptr(), self.g_lf.data_ptr(), self.g_hf.data_ptr(),
               self.fd_work.data_ptr(), self.fd_bwork.data_ptr(), self.gv(fd.sigma_resSE.fc[0].weight).data_ptr(),
               self.gv(fd.sigma_resSE.fc[2].weight).data_ptr(), self.gv(fd.HF_guided_resSE.fc[0].weight).data_ptr(),
               self.gv(fd.HF_guided_resSE.fc[2].weight).data_ptr(), self.gv(fd.channel_transform.weight).data_ptr(),
               self.gv(fd.channel_transform.bias).data_ptr(), st)


    def _ptr_sig(self):
        return tuple(p.data_ptr() for p in self.param_order)

    def _backward_body(self, d_eps):
        e, B, G = self.eng, self.B, self.G
        self._mark_i = 0
        st = e.stream
        net = self.net
        SW = nat.ACT_SWISH
        e.call("wsr_fill_zero", self.gflat.data_ptr(), self.gflat.numel() * 4, st)
        e.call("wsr_fill_zero", self.red.data_ptr(), self.red.numel() * 8, st)
        e.call("wsr_fill_zero", self.dproj.data_ptr(), self.dproj.numel() * 4, st)
        if self._garena is not None:
            e.call("wsr_fill_zero", self._garena.data_ptr(), self._garena.numel(), st)
        else:
            for g in self._gtensors:
                e.call("wsr_fill_zero", g.data_ptr(), g.numel() * g.element_size(), st)
        e.call("wsr_nchw_to_nhwc", d_eps.data_ptr(), B, self.C_img, self.H, self.W, self.deps.ptr, self.deps.dt, self.deps.ld, st)

        # head: eps = conv(swish(GN(x_last)))
        fc = net.final_conv.block
        x_last = self._x_last
        d_fa = G(self.final_a)
        e.conv(self.deps, self.dfinal, d_fa, bias=False)
        self._wgrad(self.final_a, self.deps, fc[3], T.forward_taps(3, 1, self.H, self.W))
        self._gn_bwd(x_last, fc[0], SW, d_fa, G(x_last), self.red_final, gamma=self.gf, beta=self.bf_)

        # up path, reversed
        for k in range(len(self.ups) - 1, -1, -1):
            r = self.ups[k]
            if r.kind == "res":
                self._res_block_bwd(r, r.cat)
            else:
                x = self._up_inputs[k]
                e.conv(G(r.y), r.dconv, G(x), taps=T.dgrad_upsample_taps(x.H, x.W), bias=False, res=G(x))
                self._wgrad(x, G(r.y), r.mod.conv, T.forward_upsample_taps(x.H, x.W), up=2)
        # HF-CA branches: their output gradients (skip slots of the up path's concat buffers) are final now
        hf_on_side = False
        if self.has_hfca:
            order = [self.downs[i].ca for i in range(len(self.downs) - 1, 0, -1) if self.downs[i].kind != "res"]
            hf_on_side = self._hf_ca_bwd_all_on_side(order)
        self._ready()
        for i in range(len(self.mids) - 1, -1, -1):
            self._res_block_bwd(self.mids[i], self._mid_inputs[i])
        self._ready()
        for i in range(len(self.downs) - 1, 0, -1):
            r = self.downs[i]
            x = self._down_inputs[i]
            if r.kind == "res":
                self._res_block_bwd(r, x)
            else:
                if self.has_hfca and hf_on_side:
                    ca, gx = r.ca, G(r.ca.x)
                    self._host(functools.partial(self._hjoin_fire, ca))
                    e.call("wsr_axpby", ca.dx_side.ptr, ca.dx_side.dt, ca.dx_side.ld, 1.0, gx.ptr, gx.dt, gx.ld, 1.0, gx.ptr, gx.dt, gx.ld,
                           B * ca.h * ca.w, ca.c, e.stream)
                elif self.has_hfca:
                    self._hf_ca_bwd(r.ca)
                dy, dx = G(r.y), G(x)
                for tp in T.dgrad_down_taps(x.H, x.W):
                    e.conv(dy, r.dconv, dx, taps=tp, bias=False, res=dx)
                self._wgrad(x, dy, r.mod.conv, T.forward_taps(3, 2, x.H, x.W))
                self._ready()
        if self.downs[1].kind == "res":
            self._ready()

        # stem (its input is not a function of any parameter except through ResDiff's FD_Info_Spliter)
        stem = self.downs[0]
        C = self.C_img
        dy = G(stem.y)
        self._wgrad(stem.xin, dy, stem.mod, T.forward_taps(3, 1, self.H, self.W))
        if self.kind == "resdiff":
            self._fd_bwd(dy)
        elif self.kind == "srdiff":
            # cond = cond_proj(cat(feas[2::3])) was added to the output of downs[2] (srdiff/unet.py:118,126-127): its gradient is
            # the gradient of that output; the RRDB encoder is frozen (lock_weights), so only cond_proj's parameters need it
            cp = net.cond_proj
            gy = G(self.downs[2].y)
            gw = self.gv(cp.weight)
            co_t = cp.out_channels
            for tp in T.conv_transpose_k8s4_wgrad_taps(self.cond_feat.H, self.cond_feat.W):
                e.wgrad(gy, self.cond_feat, tp, gw, (1, co_t * 64, 64), None, 1, force_simt=True)
            e.call("wsr_col_sums", gy.ptr, gy.dt, B * gy.H * gy.W, gy.C, gy.ld, self.gv(cp.bias).data_ptr(), st)
            if getattr(self, "want_cond_grad", False):
                self._cond_grad_launches(gy)

        # level embedding: all FeatureWiseAffine linears at once, then the noise MLP
        e.call("wsr_linear_rows_bwd", self.cur_temb.data_ptr(), B, self.inner, self.proj_w.data_ptr(), self.dproj.data_ptr(), self.P,
               self.dtemb.data_ptr(), self.dproj_w.data_ptr(), self.dproj_b.data_ptr(), st)
        mlp = net.noise_level_mlp
        e.call("wsr_noise_embed_bwd", self.levels.data_ptr(), B, self.inner, self.mlp_w1.data_ptr(), self.mlp_b1.data_ptr(),
               self.mlp_w2.data_ptr(), self.time_act, self.dtemb.data_ptr(), self.gv(mlp[1].weight).data_ptr(),
               self.gv(mlp[1].bias).data_ptr(), self.gv(mlp[3].weight).data_ptr(), self.gv(mlp[3].bias).data_ptr(), st)
        self._ready()
        assert self._mark_i == len(self._marks) + 1
        return self.gflat

    # ------------------------------------------------------------------------------------------------------------------
    # forward: UNetPlan.run, recorded once and then replayed
    # ------------------------------------------------------------------------------------------------------------------
    def run(self, x_t):
        """UNetPlan.run after a weight refresh and a fresh dropout seed; from the second identical call on, a replay of its
        recorded launch list."""
        e = self.eng
        self.refresh_weights()
        if self.drop_p > 0.0 and self.train_mode:
            self.drop_seed = int(torch.randint(0, 2 ** 62, (1,)).item())
            self._seed.value = self.drop_seed
        key = ("fwd", x_t.data_ptr(), self.train_mode, self._ptr_sig())
        if self.replay_enabled and self._lists.get("fwd_key") == key:
            e.replay(self._lists["fwd"])
            return self.eps
        record = self.replay_enabled and self._lists.get("fwd_seen") == key      # second identical call
        self._lists["fwd_seen"] = key
        if record:
            e.rec = []
        try:
            super().run(x_t)
        finally:
            lst, e.rec = e.rec, None
        if record:
            self._lists["fwd"], self._lists["fwd_key"] = lst, key
        return self.eps
