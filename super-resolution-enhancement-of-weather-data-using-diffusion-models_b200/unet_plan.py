"""UNetPlan -- the launch schedule of one denoiser call (reference resdiff/unet.py:121-177, srdiff/unet.py:112-141).

Built once per (UNet module, local batch, precision): packs the reference-layout fp32 parameters into kernel
layouts, allocates every activation buffer (NHWC, skip tensors written straight into the channel slice of the
up-block's concat buffer, so ``torch.cat`` never happens), and then replays a fixed sequence of C-ABI calls per step.
Because the sequence and all pointers are fixed, a whole reverse step can be captured in a CUDA graph (``sampler.py``).

Hoisting (SURVEY.md 0.3) -- results identical, work done once instead of T times:
  * condition-only: FD splitter FFT branch (lf, hf), Haar detail queries and the HF-CA ``q`` convolutions,
    SRDiff's ``cond_proj`` transposed convolution                       -> ``set_condition``
  * level-only: positional encoding, noise MLP, the 27 FeatureWiseAffine projections and ``fd_spliter.noise_func``
    for all T levels                                                    -> ``set_level_table`` (sampling)
"""
import math

import torch

from . import _native as nat
from .engine import Act, Engine, StatsArena


class _L:
    """Plain record."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


def _is_res(m):
    return type(m).__name__ == "ResnetBlocWithAttn"


class UNetPlan:
    # True for the train plan, whose forward is followed by the hand-written backward pass: every activation that pass reads stays
    # materialised (no GroupNorm fused into the consuming convolution, q | k and V^T kept apart), and, because its forward is replayed
    # from a recorded launch list that holds no stream events, there is no fused head and no HF-CA side stream.
    feeds_backward = False

    def __init__(self, net, batch, device, precision="bf16", strict_tc=False):
        self.net = net
        self.B = int(batch)
        self.eng = Engine(device, precision, strict_tc=strict_tc)
        # resdiff: FD splitter + HF-guided cross attention; phydiff: stencil channels + 3-band HF-CA queries (phydiff/unet.py);
        # srdiff: RRDB features through cond_proj; sr3: plain conditional UNet on cat([cond, x_t]) (sr3/unet.py)
        self.kind = ("resdiff" if hasattr(net, "fd_spliter") else "srdiff" if hasattr(net, "cond_proj") else
                     "phydiff" if hasattr(net, "hf_ca_list") else "sr3")
        self.has_hfca = self.kind in ("resdiff", "phydiff")
        self.C_img = net.image_channels
        self.H, self.W = net.image_height, net.image_width
        self.inner = net.inner_channel
        self.groups = net.norm_groups
        self.time_act = nat.ACT_MISH if net.time_act == "mish" else nat.ACT_SWISH
        self._wver = None
        # GroupNorm + Swish fused into the consuming convolution's operand path (transform warps rewrite the TMA-landed halo tile
        # in shared memory row by row; wsr_conv_tc with WsrConvDesc.gn_table).  Round 2 (8 transform warps on their own register
        # budget, packed bf16x2 arithmetic, row-by-row hand-over TMA -> transform -> MMA), measured on B200 at B = 64
        # (profiles/r02_fused_gn_decomposition.txt):  128->128 @64x128: 0.166 ms fused vs 0.141 conv + 0.061 gn_apply;
        # 384->128: 0.441 vs 0.358 + 0.138;  but 64->64 @128x256: 0.326 vs 0.163 + 0.094 and 192->64: 0.719 vs 0.364 + 0.260 --
        # the N = 64 layers are bound by the tensor core's own shared-memory operand fetch, and the transform's traffic on the same
        # banks slows both.  So only layers with at least 128 output channels fuse (_res_block); fusing every eligible layer measured
        # slower at every batch size (DESIGN.md section 8).
        self.fuse_gn = not self.feeds_backward and self.eng.mode == "bf16"
        self._structure()
        self._buffers()
        self.refresh_weights()

    # ------------------------------------------------------------------------------------------------------------------
    # structure: layer records with shapes, projection offsets
    # ------------------------------------------------------------------------------------------------------------------
    def _res_record(self, mod, name, cin, cout, h, w):
        rb = mod.res_block
        rec = _L(kind="res", mod=mod, name=name, cin=cin, cout=cout, h=h, w=w, attn=mod.with_attn,
                 has_res_conv=not isinstance(rb.res_conv, torch.nn.Identity), proj_off=self.P)
        self.P += cout
        return rec

    def _structure(self):
        net = self.net
        self.P = 0                       # width of the concatenated level projection (all FeatureWiseAffine linears)
        h, w = self.H, self.W
        downs, feat_shapes = [], []
        stem = net.downs[0]
        c = stem.out_channels
        downs.append(_L(kind="stem", mod=stem, name="downs.0", cin=stem.in_channels, cout=c, h=h, w=w))
        feat_shapes.append((c, h, w))
        for i, m in enumerate(list(net.downs)[1:], start=1):
            if _is_res(m):
                cout = m.res_block.block1.block[3].out_channels
                downs.append(self._res_record(m, "downs.%d" % i, c, cout, h, w))
                c = cout
            else:
                h, w = h // 2, w // 2
                downs.append(_L(kind="down", mod=m, name="downs.%d" % i, cin=c, cout=c, h=h, w=w))
            feat_shapes.append((c, h, w))
        mids = [self._res_record(m, "mid.%d" % i, c, c, h, w) for i, m in enumerate(net.mid)]
        ups = []
        fs = list(feat_shapes)
        for i, m in enumerate(net.ups):
            if _is_res(m):
                sc, sh, sw = fs.pop()
                assert (sh, sw) == (h, w)
                cout = m.res_block.block1.block[3].out_channels
                rec = self._res_record(m, "ups.%d" % i, c + sc, cout, h, w)
                rec.cx, rec.cs = c, sc
                ups.append(rec)
                c = cout
            else:
                ups.append(_L(kind="up", mod=m, name="ups.%d" % i, cin=c, cout=c, h=h * 2, w=w * 2))
                h, w = h * 2, w * 2
        self.downs, self.mids, self.ups, self.feat_shapes = downs, mids, ups, feat_shapes
        self.final_cin = c
        if self.kind == "resdiff":
            self.ne_off = self.P         # fd_spliter.noise_func output (W values) lives at the tail of the projection
            self.P += self.W

    # ------------------------------------------------------------------------------------------------------------------
    # buffers
    # ------------------------------------------------------------------------------------------------------------------
    def _buffers(self):
        e, B = self.eng, self.B
        bf = e.mode == "bf16"
        arena = self.arena = StatsArena()
        # concat buffers of the up path: ups res-block j reads cat([x, feats.pop()])
        up_res = [r for r in self.ups if r.kind == "res"]
        for r in up_res:
            r.cat = e.new_act(B, r.h, r.w, r.cx + r.cs, stats=arena)
        nfeat = len(self.feat_shapes)
        assert nfeat == len(up_res)
        feat_dst = [None] * nfeat
        for j, r in enumerate(up_res):
            feat_dst[nfeat - 1 - j] = r.cat.slice(r.cx, r.cs)
        # destination of each layer's main-path output
        max_scores = 0

        def res_scratch(r, y):
            nonlocal max_scores
            r.y = y
            r.a1 = e.new_act(B, r.h, r.w, r.cin)
            r.hbuf = e.new_act(B, r.h, r.w, r.cout, stats=arena)
            r.a2 = e.new_act(B, r.h, r.w, r.cout)
            if r.attn:
                n = r.h * r.w
                r.rbuf = e.new_act(B, r.h, r.w, r.cout, stats=arena)
                r.nbuf = e.new_act(B, r.h, r.w, r.cout)
                # sampling plans at the low-resolution levels: ONE q | k | v projection, V consumed as pixels x channels by the fused
                # attention kernel (no V^T GEMM); the train plan keeps q | k + V^T (its backward pass reads them)
                r.v_nhwc = not self.feeds_backward and bf and e.small_attention_takes_nhwc_v(n, n, r.cout)
                if r.v_nhwc:
                    r.qkv = e.new_act(B, r.h, r.w, 3 * r.cout)
                    r.qk, r.vT = r.qkv.slice(0, 2 * r.cout), None
                else:
                    r.qk = e.new_act(B, r.h, r.w, 2 * r.cout)
                    r.vT = e.empty((B, r.cout, n))
                    max_scores = max(max_scores, B * n * n)
                r.obuf = e.new_act(B, r.h, r.w, r.cout)

        # down path
        hf_i = 0
        self.hfca = []
        for i, r in enumerate(self.downs):
            if r.kind == "stem":
                cpad = 64 if bf else r.cin
                r.cin_pad = max(cpad, r.cin)
                r.xin = e.new_act(B, r.h, r.w, r.cin_pad, zero=True)
                r.y = feat_dst[i]
            elif r.kind == "res":
                res_scratch(r, feat_dst[i])
            else:
                if self.has_hfca:
                    # main path continues with the plain strided-conv output; the skip is its HF-guided attention
                    r.y = e.new_act(B, r.h, r.w, r.cout, stats=arena)
                    n = r.h * r.w
                    ca = _L(mod=self.net.hf_ca_list[hf_i], c=r.cout, h=r.h, w=r.w, x=r.y, y=feat_dst[i], level=hf_i)
                    ca.nbuf = e.new_act(B, r.h, r.w, r.cout)
                    ca.v_nhwc = not self.feeds_backward and bf and e.small_attention_takes_nhwc_v(n, n, r.cout)
                    if ca.v_nhwc:
                        ca.kv = e.new_act(B, r.h, r.w, 2 * r.cout)           # one k | v projection
                        ca.kbuf, ca.vT = ca.kv.slice(0, r.cout), None
                    else:
                        ca.kbuf = e.new_act(B, r.h, r.w, r.cout)
                        ca.vT = e.empty((B, r.cout, n))
                    ca.obuf = e.new_act(B, r.h, r.w, r.cout)
                    ca.q = e.new_act(B, r.h, r.w, r.cout)
                    ca.qimg = e.new_act(B, r.h, r.w, self.C_img * (3 if self.kind == "phydiff" else 1), dt=nat.F32)
                    if not ca.v_nhwc:
                        max_scores = max(max_scores, B * n * n)
                    r.ca = ca
                    self.hfca.append(ca)
                    hf_i += 1
                else:
                    r.y = feat_dst[i]
        # mid: mid.0 -> temp, mid.1 -> x slot of the first up concat buffer
        # (SR3 has a single mid block, sr3/unet.py:77-81): the LAST one writes into the first up concat buffer
        for m in self.mids[:-1]:
            res_scratch(m, e.new_act(B, m.h, m.w, m.cout, stats=arena))
        res_scratch(self.mids[-1], up_res[0].cat.slice(0, up_res[0].cx))
        # up path: each layer writes into the x slot of the next res block's concat buffer
        for k, r in enumerate(self.ups):
            following = self.ups[k + 1] if k + 1 < len(self.ups) else None
            if following is not None and following.kind == "res":
                dst = following.cat.slice(0, following.cx)
            else:
                dst = e.new_act(B, r.h, r.w, r.cout, stats=arena)
            if r.kind == "res":
                res_scratch(r, dst)
            else:
                r.y = dst
        # head
        self.final_a = e.new_act(B, self.H, self.W, self.final_cin)
        self.eps_nhwc = e.new_act(B, self.H, self.W, self.C_img, dt=nat.F32)
        self.eps = self.eps_nhwc.buf.view(B, self.C_img, self.H, self.W) if self.C_img == 1 else \
            e.empty((B, self.C_img, self.H, self.W), torch.float32)
        self.stats = arena.finalize(e.device)
        self.scores = e.empty((max_scores,), torch.float32) if max_scores else None
        self.probs = e.empty((max_scores,)) if max_scores else None
        # level embedding
        self.cur_proj = e.empty((B, self.P), torch.float32)
        self.cur_temb = e.empty((B, self.inner), torch.float32)
        self.levels = e.empty((B,), torch.float32)
        self.proj_table = None
        # condition state
        self.cond = e.empty((B, self.C_img, self.H, self.W), torch.float32)
        self.x_t = e.empty((B, self.C_img, self.H, self.W), torch.float32)
        if self.kind == "resdiff":
            self.lf = e.empty((B, self.C_img, self.H, self.W), torch.float32)
            self.hf = e.empty((B, self.C_img, self.H, self.W), torch.float32)
            self.gate = e.empty((B, self.C_img, self.W), torch.float32)
            nb = nat.call("wsr_fd_precompute_workspace_bytes", B, self.C_img, self.H, self.W)
            self.fd_work = e.empty((nb,), torch.uint8)
            tot = sum(B * self.C_img * (self.H >> (j + 1)) * (self.W >> (j + 1)) for j in range(4))
            self.haar_out = e.empty((tot,), torch.float32)
            self.haar_work = e.empty((B * self.C_img * self.H * self.W // 2 + 16,), torch.float32)
        elif self.kind == "phydiff":
            tot = sum(B * 3 * self.C_img * (self.H >> (j + 1)) * (self.W >> (j + 1)) for j in range(4))
            self.haar_out = e.empty((tot,), torch.float32)
            self.haar_work = e.empty((B * self.C_img * self.H * self.W // 2 + 16,), torch.float32)
            self.stencils = e.empty((B, 3, self.H, self.W), torch.float32)
        elif self.kind == "srdiff":
            self.cond_feat = e.new_act(B, self.H // 4, self.W // 4, self.net.cond_proj.in_channels)
            self.cond_up = e.new_act(B, self.H, self.W, self.net.cond_proj.out_channels)

    # ------------------------------------------------------------------------------------------------------------------
    # weights
    # ------------------------------------------------------------------------------------------------------------------
    def _weights_version(self):
        from . import autograd_glue
        return ((autograd_glue.weights_epoch,) + tuple(p._version for p in self.net.parameters())
                + tuple(p.data_ptr() for p in self.net.parameters()))

    def refresh_weights(self):
        v = self._weights_version()
        if v == self._wver:
            return
        self._wver = v
        e = self.eng
        with torch.no_grad():
            proj_w, proj_b = [], []

            def pack_res(r):
                rb = r.mod.res_block
                gn1, conv1 = rb.block1.block[0], rb.block1.block[3]
                gn2, conv2 = rb.block2.block[0], rb.block2.block[3]
                r.g1, r.b1 = e.f32(gn1.weight), e.f32(gn1.bias)
                r.g2, r.b2 = e.f32(gn2.weight), e.f32(gn2.bias)
                r.conv1 = e.pack_conv(conv1.weight, conv1.bias)
                r.conv2 = e.pack_conv(conv2.weight, conv2.bias)
                if r.has_res_conv:
                    r.resw = e.pack_conv(rb.res_conv.weight, None)
                    r.bias2 = e.static_f32(("bias2", conv2.bias.data_ptr()), conv2.bias + rb.res_conv.bias,
                                           addend=(conv2.bias.detach(), rb.res_conv.bias.detach()))
                lin = rb.noise_func.noise_func[0]
                proj_w.append(e.f32(lin.weight)); proj_b.append(e.f32(lin.bias))
                if r.attn:
                    at = r.mod.attn
                    r.g3, r.b3 = e.f32(at.norm.weight), e.f32(at.norm.bias)
                    wqkv = at.qkv.weight
                    cc = r.cout
                    if r.v_nhwc:
                        r.wqkv = e.pack_conv(wqkv, None)
                    else:
                        r.wqk = e.pack_conv(wqkv[:2 * cc], None)
                        r.wv = e.pack_rows(wqkv[2 * cc:].reshape(cc, cc))
                    r.wout = e.pack_conv(at.out.weight, at.out.bias)

            for r in self.downs:
                if r.kind == "stem":
                    r.conv = e.pack_conv(r.mod.weight, r.mod.bias, cin_pad=r.cin_pad)
                elif r.kind == "res":
                    pack_res(r)
                else:
                    r.conv = e.pack_conv(r.mod.conv.weight, r.mod.conv.bias)
                    if self.has_hfca:
                        ca, m = r.ca, r.ca.mod
                        ca.g, ca.b = e.f32(m.norm.weight), e.f32(m.norm.bias)
                        cc = ca.c
                        if ca.v_nhwc:
                            ca.wkv = e.pack_conv(m.kv.weight, None)
                        else:
                            ca.wk = e.pack_conv(m.kv.weight[:cc], None)
                            ca.wv = e.pack_rows(m.kv.weight[cc:].reshape(cc, cc))
                        ca.wout = e.pack_conv(m.out.weight, m.out.bias)
                        ca.wq = self._pack_f32_conv(m.q.weight)
            for r in self.mids:
                pack_res(r)
            for r in self.ups:
                if r.kind == "res":
                    pack_res(r)
                else:
                    r.conv = e.pack_upsample_conv(r.mod.conv.weight, r.mod.conv.bias)
            fc = self.net.final_conv.block
            self.gf, self.bf_ = e.f32(fc[0].weight), e.f32(fc[0].bias)
            self.final = e.pack_conv(fc[3].weight, fc[3].bias, rows=64 if e.mode == "bf16" else None)
            # fp32 [9][Cout][Cin] copy of the head's weights for the fused head + reverse-step kernel (wsr_final_conv_sampler_step)
            self.final_f32 = self._pack_f32_conv(fc[3].weight) if (e.mode == "bf16" and not self.feeds_backward) else None
            if (self.final_f32 is not None
                    and nat.call("wsr_head_sampler_supported", self.final_cin, self.C_img, self.groups)):
                # ldmatrix-ready bf16 blocks of the head's weights for wsr_final_conv_sampler_step
                key = ("headw", fc[3].weight.data_ptr())
                self.final_hw = e._pack_cache.get(key)
                if self.final_hw is None:
                    self.final_hw = e._pack_cache[key] = e.empty((self.final_cin // 64) * 9 * 4 * 2 * 64, torch.bfloat16)
                nat.call("wsr_pack_head_weight", self.final_f32.w.data_ptr(), self.C_img, self.final_cin, self.final_hw.data_ptr(), e.stream)
            mlp = self.net.noise_level_mlp
            self.mlp_w1, self.mlp_b1 = e.f32(mlp[1].weight), e.f32(mlp[1].bias)
            self.mlp_w2, self.mlp_b2 = e.f32(mlp[3].weight), e.f32(mlp[3].bias)
            if self.kind == "resdiff":
                fd = self.net.fd_spliter
                proj_w.append(e.f32(fd.noise_func.weight)); proj_b.append(e.f32(fd.noise_func.bias))
                self.fd_n0, self.fd_n2 = e.f32(fd.noise_resSE.fc[0].weight), e.f32(fd.noise_resSE.fc[2].weight)
                self.fd_s0, self.fd_s2 = e.f32(fd.sigma_resSE.fc[0].weight), e.f32(fd.sigma_resSE.fc[2].weight)
                self.fd_h0, self.fd_h2 = e.f32(fd.HF_guided_resSE.fc[0].weight), e.f32(fd.HF_guided_resSE.fc[2].weight)
                self.fd_ctw = e.f32(fd.channel_transform.weight.reshape(fd.channel_transform.out_channels, -1))
                self.fd_ctb = e.f32(fd.channel_transform.bias)
                self.fd_hidden = self.fd_n0.shape[0]
            elif self.kind == "srdiff":
                cp = self.net.cond_proj
                self.cp_w = e.empty((64, cp.out_channels, cp.in_channels))
                w = e.f32(cp.weight)
                e.jobs_ok = False        # no batched kind for the transposed-convolution packing
                nat.call("wsr_pack_convT_weight", w.data_ptr(), cp.in_channels, cp.out_channels, 8, 8, self.cp_w.data_ptr(), e.dt, e.stream)
                self.cp_b = e.f32(cp.bias)
                e._keep.append(w)
            self.proj_w = e.static_f32(("proj_w", id(self)), torch.cat(proj_w, 0), parts=proj_w)
            self.proj_b = e.static_f32(("proj_b", id(self)), torch.cat(proj_b, 0), parts=proj_b)
            assert self.proj_w.shape == (self.P, self.inner), (self.proj_w.shape, self.P)
        self.proj_table = None
        # no host synchronisation: the temporaries were consumed by kernels launched on torch's current stream, and the
        # caching allocator only hands a freed block to later work on that same stream
        e._keep.clear()

    def _pack_f32_conv(self, weight):
        """fp32-packed conv weight (used for the 1-channel Haar query convolution, kept in fp32 in both modes)."""
        e = self.eng
        w = e.f32(weight)
        Cout, Cin, KH, KW = w.shape
        from .engine import PackedConv
        key = ("f32conv", e._src_key(weight))
        pc = e._pack_cache.get(key)
        if pc is None:
            pc = e._pack_cache[key] = PackedConv()
            pc.Cout, pc.Cin, pc.k, pc.Cin_pad, pc.rows, pc.bias = Cout, Cin, KH, Cin, Cout, None
            pc.w = e.empty((KH * KW, Cout, Cin), torch.float32)
        nat.call("wsr_pack_conv_weight", w.data_ptr(), Cout, Cin, KH, KW, pc.w.data_ptr(), nat.F32, Cout, Cin, e.stream)
        e._job(nat.PACK_CONV, w.data_ptr(), pc.w.data_ptr(), nat.F32, Cout, Cin, KH * KW, Cout, Cin, stable=w.data_ptr() == weight.data_ptr())
        e._keep.append(w)
        return pc

    # ------------------------------------------------------------------------------------------------------------------
    # condition-only and level-only precompute
    # ------------------------------------------------------------------------------------------------------------------
    def set_condition(self, cond, repeats=1):
        """resdiff: cond = x_in['SR'] (B,C,H,W).  srdiff: cond = cat(feas[2::3], 1) (B,384,H/4,W/4).
        repeats = R > 1 (ensembles): cond holds B / R conditions; the condition-only work runs once on them and its outputs are copied
        into the other R - 1 member slices of the batch, so every member sees exactly what a run on the B / R conditions alone sees
        (for resdiff the FD splitter's 4-D FFT couples the batch: each member gets the spectrum of its own B / R group)."""
        e = self.eng
        repeats = int(repeats)
        if repeats < 1 or self.B % repeats or cond.shape[0] * repeats != self.B:
            raise ValueError("set_condition: %d conditions x %d repeats != plan batch %d" % (cond.shape[0], repeats, self.B))
        B = self.B // repeats
        st = e.stream

        def head(a):
            # the first B images of an activation buffer (Act is image-major, so this is a prefix of the same buffer)
            return Act(a.buf, B, a.H, a.W, a.C, a.ld, a.coff, a.dt)
        if self.kind == "resdiff":
            self.cond[:B].copy_(cond.to(torch.float32))
            nat.call("wsr_fd_precompute", self.cond.data_ptr(), B, self.C_img, self.H, self.W, self.fd_s0.data_ptr(),
                     self.fd_s2.data_ptr(), self.fd_h0.data_ptr(), self.fd_h2.data_ptr(), self.fd_ctw.data_ptr(),
                     self.fd_ctb.data_ptr(), self.fd_ctw.shape[0], self.lf.data_ptr(), self.hf.data_ptr(),
                     self.fd_work.data_ptr(), st)
            nat.call("wsr_haar_detail_sums", self.cond.data_ptr(), B, self.C_img, self.H, self.W, 4, self.haar_out.data_ptr(),
                     self.haar_work.data_ptr(), st)
            off = 0
            for ca in self.hfca:
                n = B * self.C_img * ca.h * ca.w
                j = ca.level
                assert (ca.h, ca.w) == (self.H >> (j + 1), self.W >> (j + 1))
                nat.call("wsr_nchw_to_nhwc", self.haar_out.data_ptr() + 4 * off, B, self.C_img, ca.h, ca.w, ca.qimg.ptr,
                         nat.F32, ca.qimg.ld, st)
                e.conv(head(ca.qimg), ca.wq, head(ca.q), bias=False, force_simt=True)
                off += n
            shared = [self.cond, self.lf, self.hf] + [ca.q.buf for ca in self.hfca]
        elif self.kind == "phydiff":
            # condition-only work of phydiff/unet.py:262-314, done once per batch: stencil channels of the reflect-padded
            # condition, the 3-band Haar queries and their 1x1 projections; cond and the stencils are written straight into
            # their channel slices of the stem input [cond | x_t | Kx Ky Kxy]
            C = self.C_img
            stem = self.downs[0]
            self.cond[:B].copy_(cond.to(torch.float32))
            nat.call("wsr_phy_stencils", self.cond.data_ptr(), B, C, self.H, self.W, self.stencils.data_ptr(), st)
            e.nchw_to_act(self.cond[:B], head(stem.xin.slice(0, C)))
            e.nchw_to_act(self.stencils[:B], head(stem.xin.slice(2 * C, 3)))
            nat.call("wsr_haar_detail_bands", self.cond.data_ptr(), B, C, self.H, self.W, 4, self.haar_out.data_ptr(),
                     self.haar_work.data_ptr(), st)
            off = 0
            for ca in self.hfca:
                n = B * 3 * C * ca.h * ca.w
                j = ca.level
                assert (ca.h, ca.w) == (self.H >> (j + 1), self.W >> (j + 1))
                nat.call("wsr_nchw_to_nhwc", self.haar_out.data_ptr() + 4 * off, B, 3 * C, ca.h, ca.w, ca.qimg.ptr,
                         nat.F32, ca.qimg.ld, st)
                e.conv(head(ca.qimg), ca.wq, head(ca.q), bias=False, force_simt=True)
                off += n
            shared = [stem.xin.buf] + [ca.q.buf for ca in self.hfca]     # stem input: its x_t slice is rewritten every step
        elif self.kind == "sr3":
            self.cond[:B].copy_(cond.to(torch.float32))
            e.nchw_to_act(self.cond[:B], head(self.downs[0].xin.slice(0, self.C_img)))
            shared = [self.downs[0].xin.buf]
        else:
            src = cond.to(torch.float32).contiguous()
            e.nchw_to_act(src, head(self.cond_feat))
            nat.call("wsr_conv_transpose_k8s4", self.cond_feat.ptr, self.cond_feat.dt, B, self.cond_feat.H, self.cond_feat.W,
                     self.cond_feat.C, self.cond_feat.ld, self.cp_w.data_ptr(), self.cp_b.data_ptr(), self.cond_up.C,
                     self.cond_up.ptr, self.cond_up.dt, self.cond_up.ld, st)
            shared = [self.cond_up.buf]
        for t in shared if repeats > 1 else ():
            for r in range(1, repeats):
                t[r * B:(r + 1) * B].copy_(t[:B])          # contiguous device-to-device copies

    def _embed(self, levels, n_rows, temb, proj):
        st = self.eng.stream
        nat.call("wsr_noise_embed", levels.data_ptr(), n_rows, self.inner, self.mlp_w1.data_ptr(), self.mlp_b1.data_ptr(),
                 self.mlp_w2.data_ptr(), self.mlp_b2.data_ptr(), self.time_act, temb.data_ptr(), st)
        nat.call("wsr_linear_rows", temb.data_ptr(), n_rows, self.inner, self.proj_w.data_ptr(), self.proj_b.data_ptr(),
                 self.P, proj.data_ptr(), st)

    def set_levels(self, levels):
        """Per-sample continuous noise levels (B,) -- the training / generic ``forward`` path."""
        self.levels.copy_(levels.to(torch.float32))
        self._embed(self.levels, self.B, self.cur_temb, self.cur_proj)

    def set_level_table(self, levels_T):
        """All T levels of a sampling schedule: proj_table[r] is the projection of level r (computed once)."""
        e = self.eng
        lv = levels_T.to(device=e.device, dtype=torch.float32).contiguous()
        T = lv.numel()
        self.table_levels = lv
        self.temb_table = e.empty((T, self.inner), torch.float32)
        self.proj_table = e.empty((T, self.P), torch.float32)
        self._embed(lv, T, self.temb_table, self.proj_table)

    def select_level_row(self, row_index_dev):
        """cur_proj[b] = proj_table[*row_index] for every b (device-side index: CUDA-graph friendly)."""
        self.eng.call("wsr_broadcast_row", self.proj_table.data_ptr(), self.P, row_index_dev.data_ptr(), self.B,
                      self.cur_proj.data_ptr(), self.eng.stream)

    # ------------------------------------------------------------------------------------------------------------------
    # the denoiser
    # ------------------------------------------------------------------------------------------------------------------
    def denoise(self, x_t):
        """Generic entry: x_t (B,C,H,W) fp32 NCHW -> eps_hat (B,C,H,W) fp32 (a fresh tensor)."""
        self.x_t.copy_(x_t.to(torch.float32))
        self.run(self.x_t)
        return self.eps.clone()

    def _rowvec(self, r):
        return self.cur_proj.data_ptr() + 4 * r.proj_off

    def _res_block(self, r, x, extra_res=None):
        e, B, G = self.eng, self.B, self.groups
        SW = nat.ACT_SWISH
        if not hasattr(r, "fuse1"):
            wide = r.cout >= 128
            r.fuse1 = self.fuse_gn and wide and e.conv_can_fuse_gn(x, r.conv1)
            r.fuse2 = self.fuse_gn and wide and e.conv_can_fuse_gn(r.hbuf, r.conv2, x2=x if r.has_res_conv else None)
            r.tab1 = e.empty((B, r.cin, 2), torch.float32) if r.fuse1 else None
            r.tab2 = e.empty((B, r.cout, 2), torch.float32) if r.fuse2 else None
        if r.fuse1:
            e.gn_finalize(x, r.g1, r.b1, G, r.tab1)
            e.conv(x, r.conv1, r.hbuf, rowvec=self._rowvec(r), rowvec_ld=self.P, gn=(r.tab1, SW))
        else:
            e.gn_apply(x, r.g1, r.b1, G, SW, r.a1)
            e.conv(r.a1, r.conv1, r.hbuf, rowvec=self._rowvec(r), rowvec_ld=self.P)
        dst = r.rbuf if r.attn else r.y
        er = None if r.attn else extra_res
        if r.fuse2:
            e.gn_finalize(r.hbuf, r.g2, r.b2, G, r.tab2)
            a2, gn2 = r.hbuf, (r.tab2, SW)
        else:
            self._block2_norm(r)
            a2, gn2 = r.a2, None
        if r.has_res_conv:
            e.conv(a2, r.conv2, dst, x2=x, w2=r.resw, extra_bias=r.bias2, res2=er, gn=gn2)
        else:
            e.conv(a2, r.conv2, dst, res=x, res2=er, gn=gn2)
        if r.attn:
            e.gn_apply(r.rbuf, r.g3, r.b3, G, nat.ACT_NONE, r.nbuf)
            n = r.h * r.w
            if r.v_nhwc:
                e.conv(r.nbuf, r.wqkv, r.qkv, bias=False)
                e.attention(r.qkv.slice(0, r.cout), r.qkv.slice(r.cout, r.cout), None, r.obuf, None, None, v=r.qkv.slice(2 * r.cout, r.cout))
            else:
                e.conv(r.nbuf, r.wqk, r.qk, bias=False)
                self._v_transposed(r.wv, r.nbuf, r.vT)
                e.attention(r.qk.slice(0, r.cout), r.qk.slice(r.cout, r.cout), r.vT, r.obuf,
                            self.scores[:B * n * n], self.probs[:B * n * n])
            e.conv(r.obuf, r.wout, r.y, res=r.rbuf, res2=extra_res)
        return r.y

    def _block2_norm(self, r):
        """GroupNorm + Swish of block2 (nn_modules/resnet.py:21-22); the training plan adds the dropout of :23 here."""
        self.eng.gn_apply(r.hbuf, r.g2, r.b2, self.groups, nat.ACT_SWISH, r.a2)

    def _v_transposed(self, wv, nact, vT):
        """vT[b][c][pix] = sum_k Wv[c][k] * n[b][pix][k]  (V produced already transposed = K-major for P*V)."""
        e = self.eng
        cc, n = wv.shape[0], nact.H * nact.W
        e.gemm(wv.data_ptr(), e.dt, (0, cc, 1), nact.ptr, nact.dt, (n * nact.ld, nact.ld, 1),
               vT.data_ptr(), e.dt, (cc * n, n, 1), self.B, cc, n, cc)

    def _side_stream(self):
        """The HF-guided cross-attention branches (resdiff/unet.py:156-163: they only produce the SKIP tensors; the main path continues
        with the un-attended x) run on a second stream, forked after each Downsample and joined before the up path: the N = 8192 /
        2048 attention launches then overlap the deep levels of the down path, whose kernels leave most SMs idle at small batch.
        Works eagerly and inside a captured CUDA graph (event fork / join).  Only when every branch launch is a fused kernel -- the
        unfused fallback shares the score scratch with the main path's self-attention -- and not while per-launch timing is on."""
        if self.feeds_backward or not self.has_hfca or self.eng.prof is not None:
            return None
        ok = getattr(self, "_side_ok", None)
        if ok is None:
            e = self.eng
            ok = e.use_tc and e.mode == "bf16" and not e.no_fused_attention
            for ca in self.hfca:
                n = ca.h * ca.w
                fused_long = ca.c in (64, 128) and n % 128 == 0
                fused_small = bool(nat.call("wsr_attention_small_tc_supported", n, n, ca.c))
                ok = ok and (fused_long or fused_small)
            self._side_ok = ok
            self._side = torch.cuda.Stream(device=e.device) if ok else None
        return self._side if ok else None

    def _hf_ca(self, ca):
        e, B = self.eng, self.B
        e.gn_apply(ca.x, ca.g, ca.b, 32, nat.ACT_NONE, ca.nbuf)       # norm_groups fixed at 32 (guided_cross_attention.py:15)
        n = ca.h * ca.w
        if ca.v_nhwc:
            e.conv(ca.nbuf, ca.wkv, ca.kv, bias=False)
            e.attention(ca.q, ca.kbuf, None, ca.obuf, None, None, v=ca.kv.slice(ca.c, ca.c))
        else:
            e.conv(ca.nbuf, ca.wk, ca.kbuf, bias=False)
            self._v_transposed(ca.wv, ca.nbuf, ca.vT)
            e.attention(ca.q, ca.kbuf, ca.vT, ca.obuf, self.scores[:B * n * n], self.probs[:B * n * n])
        e.conv(ca.obuf, ca.wout, ca.y, res=ca.x)

    def _stem_input(self, x_t):
        """Per-step part of the stem input: ResDiff's noise gate + 5-channel assembly (fd_info_spliter.py:44-47,117), or x_t
        written into its channel slice next to the condition-only channels (sr3 / phydiff), or x_t alone (srdiff)."""
        e, B = self.eng, self.B
        st = e.stream
        stem = self.downs[0]
        if self.kind == "resdiff":
            e.call("wsr_fd_gate", self.cur_proj.data_ptr() + 4 * self.ne_off, self.P, 0, B, self.C_img, self.W,
                     self.fd_n0.data_ptr(), self.fd_n2.data_ptr(), self.fd_hidden, self.gate.data_ptr(), st)
            e.call("wsr_stem_assemble", x_t.data_ptr(), self.cond.data_ptr(), self.gate.data_ptr(), self.lf.data_ptr(),
                     self.hf.data_ptr(), B, self.C_img, self.H, self.W, stem.xin.ptr, stem.xin.dt, stem.xin.ld, st)
        elif self.kind in ("phydiff", "sr3"):
            xs = stem.xin.slice(self.C_img, self.C_img)         # channels [C, 2C) of [cond | x_t | ...]
            e.call("wsr_nchw_to_nhwc", x_t.data_ptr(), B, self.C_img, self.H, self.W, xs.ptr, xs.dt, xs.ld, st)
        else:
            e.call("wsr_nchw_to_nhwc", x_t.data_ptr(), B, self.C_img, self.H, self.W, stem.xin.ptr, stem.xin.dt, stem.xin.ld, st)

    def can_fuse_head(self):
        """True when the head (GroupNorm + Swish + conv3x3 to <= 4 channels) can run fused with the reverse-step update
        (wsr_final_conv_sampler_step): bf16 sampling plan, head input produced by a convolution that emitted its statistics."""
        ok = getattr(self, "_fuse_head", None)
        if ok is None:
            ok = self._fuse_head = (not self.feeds_backward and self.eng.mode == "bf16" and self.eng.use_tc
                                    and bool(nat.call("wsr_head_sampler_supported", self.final_cin, self.C_img, self.groups)))
        return ok

    def head_sampler_step(self, feat, x_state, tab, T, t_dev, z, z_stride, seed, clip, members=None, hist=None):
        """eps_hat = final_conv(feat) and x_state <- reverse-step update, one launch; eps_hat is also left in ``self.eps``.
        members: None, or (device key table, elements per member) for member-keyed noise (wsr_final_conv_sampler_step_members).
        hist: None, or the fp32 x0 history of a multistep table (wsr_final_conv_sampler_step_multistep; z, seed and members unused)."""
        e = self.eng
        assert feat.stats_ptr and feat.C == self.final_cin and feat.dt == nat.BF16
        npix = self.B * self.H * self.W
        head = (feat.ptr, feat.ld, self.B, self.H, self.W, feat.C, feat.stats_ptr, feat.st_ld, self.gf.data_ptr(), self.bf_.data_ptr(),
                self.groups, 1e-5, self.final_hw.data_ptr(), self.final.bias.data_ptr(), self.C_img, self.eps.data_ptr(),
                x_state.data_ptr(), 0 if z is None else z.data_ptr(), z_stride)
        tail = (tab.data_ptr(), T, t_dev.data_ptr(), 1 if clip else 0, e.stream)
        cost = dict(tag="head_sampler", flops=2 * npix * 9 * feat.C * self.C_img,
                    nbytes=npix * (feat.C * 2 + self.C_img * (16 if z is not None else 12)))
        if hist is not None:
            cost["nbytes"] = npix * (feat.C * 2 + self.C_img * 20)
            e.call("wsr_final_conv_sampler_step_multistep", *head[:-2], hist.data_ptr(), *tail, **cost)
        elif members is None:
            e.call("wsr_final_conv_sampler_step", *head, seed, *tail, **cost)
        else:
            e.call("wsr_final_conv_sampler_step_members", *head, members[0].data_ptr(), members[1], *tail, **cost)

    def run(self, x_t, head=True):
        """One denoiser call on the current condition / level projection.  x_t: fp32 NCHW device tensor (B,C,H,W).
        Leaves eps_hat in ``self.eps`` (fp32 NCHW).  head=False: stop before ``final_conv`` and return its (raw) input Act --
        the caller runs the head fused with the sampler update (``head_sampler_step``).  Records which buffer fed each layer
        (``_down_inputs``, ``_mid_inputs``, ``_up_inputs``, ``_x_last``): the train plan's backward walks them in reverse."""
        e, B = self.eng, self.B
        st = e.stream
        e.call("wsr_fill_zero", self.stats.data_ptr(), self.stats.numel() * 8, st)
        main, side = torch.cuda.current_stream(e.device), self._side_stream()
        stem = self.downs[0]
        self._stem_input(x_t)
        x = e.conv(stem.xin, stem.conv, stem.y)
        self._down_inputs, self._mid_inputs, self._up_inputs = {}, {}, {}
        for i, r in enumerate(self.downs[1:], start=1):
            self._down_inputs[i] = x
            extra = self.cond_up if (self.kind == "srdiff" and i == 2) else None
            if r.kind == "res":
                x = self._res_block(r, x, extra_res=extra)
            else:
                x = e.conv(x, r.conv, r.y, stride=2, res=extra)
                if self.has_hfca:
                    if side is None:
                        self._hf_ca(r.ca)
                    else:
                        # fork: the branch only reads r.y (complete on the main stream at this point) and writes its own scratch and
                        # the skip slot of an up-path concat buffer, which nothing touches before the join below
                        ev = torch.cuda.Event()
                        ev.record(main)
                        side.wait_event(ev)
                        with torch.cuda.stream(side):
                            self._hf_ca(r.ca)
        for i, r in enumerate(self.mids):
            self._mid_inputs[i] = x
            x = self._res_block(r, x)
        if side is not None:
            ev = torch.cuda.Event()
            ev.record(side)
            main.wait_event(ev)            # join: the up path consumes the skips written by the branch
        for k, r in enumerate(self.ups):
            if r.kind == "res":
                x = self._res_block(r, r.cat)
            else:
                self._up_inputs[k] = x
                x = e.conv(x, r.conv, r.y, upsample=True)
        self._x_last = x
        if not head:
            return x
        self._head(x)
        if self.C_img != 1:
            e.call("wsr_nhwc_to_nchw", self.eps_nhwc.ptr, nat.F32, self.eps_nhwc.ld, B, self.C_img, self.H, self.W,
                     self.eps.data_ptr(), st)
        return self.eps

    def _head(self, x):
        """final_conv = GroupNorm -> Swish -> conv3x3 (resdiff/unet.py:119, nn_modules/resnet.py:19-28)."""
        e = self.eng
        e.gn_apply(x, self.gf, self.bf_, self.groups, nat.ACT_SWISH, self.final_a)
        e.conv(self.final_a, self.final, self.eps_nhwc)
