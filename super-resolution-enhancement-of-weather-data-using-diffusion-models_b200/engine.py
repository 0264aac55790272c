"""Host-side engine: device buffers, packed weights and typed wrappers over the C ABI (libwsr.so).

PyTorch is used here only as plumbing: it owns device memory (``torch.empty``) and the CUDA stream; every arithmetic
operation is a call into the hand-written kernels through ``_native.call``.  Activations are NHWC slices (``Act``)
with an explicit channel pitch so that skip-concatenation and dense blocks never copy.

Precision modes
---------------
``bf16``   bf16 activations/weights, tcgen05 tensor-core kernels (``wsr_conv_tc`` / ``wsr_gemm_tc``), fp32 accumulation.
           Shapes the tensor-core kernel does not take (channel counts that are not multiples of 64, e.g. the 1-channel
           Haar query convolution) run on the SIMT kernel; with ``strict_tc=True`` that raises instead.
``fp32``   "fp32 check mode": fp32 activations/weights on the SIMT kernels; matches the reference to ~1e-5.
"""
import ctypes as C
import math

import torch

from . import _native as nat

_DT = {"bf16": (nat.BF16, torch.bfloat16), "fp32": (nat.F32, torch.float32)}


def _ptr(t):
    return 0 if t is None else t.data_ptr()


class StatsArena:
    """Bump allocator for the per-(image, channel) GroupNorm statistics (doubles).  Offsets are handed out while the
    plan is being laid out; ``finalize`` allocates the single zero-initialised tensor that is cleared once per step."""

    def __init__(self):
        self.size = 0
        self.tensor = None

    def alloc(self, n):
        off = self.size
        self.size += n
        return off

    def finalize(self, device):
        self.tensor = torch.zeros(max(self.size, 1), device=device, dtype=torch.float64)
        return self.tensor


class Act:
    """A channel slice [coff, coff+C) of an NHWC buffer (N, H, W, ld).  ``st*`` optionally locate the GroupNorm
    statistics of these channels: doubles at arena[st_off + n*st_ld + 2*c + {0,1}]."""

    __slots__ = ("buf", "N", "H", "W", "C", "ld", "coff", "dt", "st", "st_off", "st_ld")

    def __init__(self, buf, N, H, W, C, ld, coff, dt, st=None, st_off=0, st_ld=0):
        self.buf, self.N, self.H, self.W, self.C, self.ld, self.coff, self.dt = buf, N, H, W, C, ld, coff, dt
        self.st, self.st_off, self.st_ld = st, st_off, st_ld

    @property
    def ptr(self):
        return self.buf.data_ptr() + self.coff * self.buf.element_size()

    @property
    def stats_ptr(self):
        return 0 if self.st is None else self.st.tensor.data_ptr() + 8 * self.st_off

    def slice(self, c0, c):
        assert 0 <= c0 and c0 + c <= self.C
        return Act(self.buf, self.N, self.H, self.W, c, self.ld, self.coff + c0, self.dt, self.st, self.st_off + 2 * c0, self.st_ld)

    def to_nchw(self, eng):
        out = torch.empty((self.N, self.C, self.H, self.W), device=self.buf.device, dtype=torch.float32)
        nat.call("wsr_nhwc_to_nchw", self.ptr, self.dt, self.ld, self.N, self.C, self.H, self.W, out.data_ptr(), eng.stream)
        return out


class PackedConv:
    """Conv weight packed as [tap][rows][Cin_pad] in the engine dtype, fp32 bias."""

    def __init__(self):
        self.w = self.bias = None
        self.Cout = self.Cin = self.Cin_pad = self.rows = self.k = 0
        self.merged_up = False          # True: phase-merged taps of an upsample conv (wsr_pack_upsample_weight)
        self.w_vm = None                # vertical-tap-merge packing (3x3, Cout <= 64, bf16 mode): see wsr_conv_tc


class Engine:
    def __init__(self, device, mode="bf16", strict_tc=False):
        if mode not in _DT:
            raise ValueError("mode must be 'bf16' or 'fp32', got %r" % (mode,))
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise nat.WsrError("the B200 engine needs a CUDA device; there is no CPU fallback (got %s)" % device)
        self.mode = mode
        self.dt, self.tdt = _DT[mode]
        self.strict_tc = strict_tc
        self.use_tc = mode == "bf16" and bool(nat.call("wsr_device_is_sm100"))
        if mode == "bf16" and not self.use_tc and strict_tc:
            raise nat.WsrError("bf16 tensor-core mode needs an sm_100 device")
        self.n_tc = 0
        self.n_simt = 0
        self._keep = []          # tensors that must outlive async launches
        self._pack_cache = {}    # key -> packed buffers: re-packing after an optimizer step writes the SAME device buffers,
                                 # so pointers recorded in launch lists stay valid
        self.jobs = None         # when a list: every pack_* call also appends its WsrPackJob description (batched refresh)
        self.jobs_ok = True      # False once a pack read from a temporary (no stable source address): batching impossible
        self.rec = None          # when a list: every launch made through call() is appended as (fn, args) for replay()
        self.prof = None         # list of (name, flops, bytes, start_event, end_event) when profiling
        self.prof_detail = False
        self.no_fused_attention = False

    # ---- plumbing -------------------------------------------------------------------------------------------------
    def call(self, name, *args, flops=0, nbytes=0, tag=None, xflops=None):
        """nat.call with optional per-launch CUDA-event timing (bench.py roofline pass).  flops = ALGORITHMIC FLOPs (as the
        reference executes the op); xflops = FLOPs the kernel actually EXECUTES when they differ (phase-merged upsample taps)."""
        if self.prof is None:
            rc = nat.call(name, *args)
            if self.rec is not None:
                self.rec.append((nat.fn(name), args, name))
            return rc
        s = torch.cuda.Event(enable_timing=True)
        t = torch.cuda.Event(enable_timing=True)
        s.record(torch.cuda.current_stream(self.device))
        rc = nat.call(name, *args)
        t.record(torch.cuda.current_stream(self.device))
        self.prof.append((tag or name, flops, nbytes, s, t, flops if xflops is None else xflops))
        return rc

    def replay(self, entries):
        """Re-issue a recorded launch list: same entry points, same argument objects (device pointers, descriptors and
        tap tables are fixed per plan; values that change per step -- dropout seeds -- are shared ctypes objects whose
        .value is updated before the replay).  Entries with fn None are host callbacks (gradient-bucket hooks)."""
        if self.prof is not None:
            for fn, args, name in entries:
                if fn is None:
                    args()
                else:
                    self.call(name, *args)
            return
        for fn, args, name in entries:
            if fn is None:
                args()
            else:
                rc = fn(*args)
                if rc != 0:
                    raise nat.WsrError("%s failed (%d) during replay: %s" % (name, rc, nat.last_error()))
        nat.launches += len(entries)

    def prof_summary(self):
        """name -> [launches, ms, algorithmic flops, bytes, executed flops] from the recorded events (synchronises)."""
        torch.cuda.synchronize(self.device)
        out = {}
        for name, fl, nb, s, t, xf in self.prof:
            r = out.setdefault(name, [0, 0.0, 0, 0, 0])
            r[0] += 1; r[1] += s.elapsed_time(t); r[2] += fl; r[3] += nb; r[4] += xf
        return out

    @property
    def stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def empty(self, shape, dtype=None):
        return torch.empty(shape, device=self.device, dtype=dtype or self.tdt)

    def zeros(self, shape, dtype=None):
        return torch.zeros(shape, device=self.device, dtype=dtype or self.tdt)

    def new_act(self, N, H, W, C, ld=None, dt=None, zero=False, stats=None):
        """stats: a StatsArena to reserve GroupNorm statistics for this buffer (it will be the input of a GroupNorm)."""
        ld = ld or C
        tdt = self.tdt if dt is None else (torch.bfloat16 if dt == nat.BF16 else torch.float32)
        buf = (torch.zeros if zero else torch.empty)((N, H, W, ld), device=self.device, dtype=tdt)
        a = Act(buf, N, H, W, C, ld, 0, self.dt if dt is None else dt)
        if stats is not None:
            a.st, a.st_off, a.st_ld = stats, stats.alloc(N * ld * 2), ld * 2
        return a

    def f32(self, t, track=True):
        r = t.detach().to(device=self.device, dtype=torch.float32).contiguous()
        if track and self.jobs is not None and r.data_ptr() != t.data_ptr():
            self.jobs_ok = False     # a converted COPY of a parameter would go stale under the batched refresh
        return r

    # ---- packing ---------------------------------------------------------------------------------------------------
    def _src_key(self, t):
        return (t.data_ptr(), tuple(t.shape), tuple(t.stride()))

    def _job(self, kind, src, dst, dt, Cout, Cin, taps, Cout_pad, Cin_pad, transposed=0, src2=0, stable=True):
        if self.jobs is None:
            return
        if not stable:
            self.jobs_ok = False
        units = Cout if kind == nat.PACK_COPY else Cout_pad * Cin_pad
        self.jobs.append((kind, src, src2, dst, dt, Cout, Cin, taps, Cout_pad, Cin_pad, transposed, units))

    def job_table(self):
        """Device copy of the recorded jobs -> (tensor holding the WsrPackJob array, njobs, total units)."""
        arr = (nat.PackJob * len(self.jobs))()
        first = 0
        for a, (kind, src, src2, dst, dt, Cout, Cin, taps, Cout_pad, Cin_pad, transposed, units) in zip(arr, self.jobs):
            a.src, a.src2, a.dst, a.first_unit = src, src2 or None, dst, first
            a.kind, a.transposed, a.dst_dtype, a.Cout, a.Cin, a.taps, a.Cout_pad, a.Cin_pad = kind, transposed, dt, Cout, Cin, taps, Cout_pad, Cin_pad
            first += units
        host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)
        return host.to(self.device), len(self.jobs), first

    def pack_conv(self, weight, bias=None, cin_pad=None, rows=None, key=None, src=None, job_kind=None):
        """weight: OIHW fp32 parameter (or a tensor derived from one; then pass ``key`` = a stable identity for the cache,
        e.g. ('dgrad', param.data_ptr()), because a derived temporary has a new address on every call)."""
        w = self.f32(weight, track=False)
        Cout, Cin, KH, KW = w.shape
        key = ("conv", key if key is not None else self._src_key(weight), cin_pad, rows)
        pc = self._pack_cache.get(key)
        if pc is None:
            pc = self._pack_cache[key] = PackedConv()
            pc.Cout, pc.Cin, pc.k = Cout, Cin, KH
            pc.Cin_pad = cin_pad or Cin
            pc.rows = rows or Cout
            pc.merged_up = False
            pc.w = self.empty((KH * KW, pc.rows, pc.Cin_pad))
            if self.use_tc and KH == 3 and KW == 3 and Cout <= 64 and pc.Cin_pad % 64 == 0:
                pc.w_vm = self.empty((3, 192, pc.Cin_pad))
        nat.call("wsr_pack_conv_weight", w.data_ptr(), Cout, Cin, KH, KW, pc.w.data_ptr(), self.dt, pc.rows, pc.Cin_pad, self.stream)
        # the batched refresh reads the PARAMETER: either `weight` itself (src None) or the parameter that `weight` is the
        # data-gradient view of (src = (parameter address, 1))
        jsrc, jtr = src if src is not None else (w.data_ptr(), 0)
        stable = src is not None or w.data_ptr() == weight.data_ptr()
        self._job(nat.PACK_CONV if job_kind is None else job_kind, jsrc, pc.w.data_ptr(), self.dt, Cout, Cin,
                  9 if job_kind is not None else KH * KW, pc.rows, pc.Cin_pad, jtr, stable=stable)
        if pc.w_vm is not None:
            nat.call("wsr_pack_conv_weight_vmerge", w.data_ptr(), Cout, Cin, pc.w_vm.data_ptr(), self.dt, pc.Cin_pad, self.stream)
            self._job(nat.PACK_VMERGE, jsrc, pc.w_vm.data_ptr(), self.dt, Cout, Cin, 9, 64, pc.Cin_pad, jtr, stable=stable)
        pc.bias = None if bias is None else self.f32(bias)
        self._keep.append(w)
        return pc

    def static_f32(self, key, value, parts=None, addend=None):
        """fp32 device tensor with a stable address holding ``value`` (a tensor computed on the fly).  For the batched
        refresh the caller says how ``value`` derives from parameters: ``parts`` = the tensors it is the dim-0 concatenation
        of, or ``addend`` = (a, b) with value = a + b."""
        buf = self._pack_cache.get(("f32", key))
        v = self.f32(value)
        if buf is None:
            buf = self._pack_cache[("f32", key)] = v.clone()
        else:
            buf.copy_(v)
        if self.jobs is not None:
            if addend is not None:
                a, b = addend
                ok = a.is_contiguous() and b.is_contiguous() and a.dtype == torch.float32 and b.dtype == torch.float32
                self._job(nat.PACK_COPY, a.data_ptr(), buf.data_ptr(), nat.F32, a.numel(), 1, 1, 1, 1, 0, src2=b.data_ptr(), stable=ok)
            elif parts is not None:
                off = 0
                for t in parts:
                    ok = t.is_contiguous() and t.dtype == torch.float32
                    self._job(nat.PACK_COPY, t.data_ptr(), buf.data_ptr() + 4 * off, nat.F32, t.numel(), 1, 1, 1, 1, 0, stable=ok)
                    off += t.numel()
                assert off == buf.numel()
            else:
                self.jobs_ok = False
        return buf

    def pack_upsample_conv(self, weight, bias=None):
        """Weights of 'nearest x2 upsample + conv3x3' (functional_layers.py:62-67).  In bf16 mode the taps that read the
        same source pixel are pre-summed per output phase (2.25x fewer MACs); the fp32 check mode keeps the 9 exact taps."""
        if self.mode != "bf16":
            return self.pack_conv(weight, bias)
        w = self.f32(weight)
        Cout, Cin, KH, KW = w.shape
        assert KH == 3 and KW == 3
        key = ("upconv", self._src_key(weight))
        pc = self._pack_cache.get(key)
        if pc is None:
            pc = self._pack_cache[key] = PackedConv()
            pc.Cout, pc.Cin, pc.k, pc.Cin_pad, pc.rows, pc.merged_up = Cout, Cin, 3, Cin, Cout, True
            pc.w = self.empty((16, Cout, Cin))
        nat.call("wsr_pack_upsample_weight", w.data_ptr(), Cout, Cin, pc.w.data_ptr(), self.dt, Cout, Cin, self.stream)
        self._job(nat.PACK_UPSAMPLE, w.data_ptr(), pc.w.data_ptr(), self.dt, Cout, Cin, 9, Cout, Cin, stable=w.data_ptr() == weight.data_ptr())
        pc.bias = None if bias is None else self.f32(bias)
        self._keep.append(w)
        return pc

    def pack_rows(self, weight2d):
        """(rows, K) fp32 matrix -> engine dtype, row-major (K-major operand for the GEMM kernels)."""
        w = self.f32(weight2d)
        key = ("rows", self._src_key(weight2d))
        out = self._pack_cache.get(key)
        if out is None:
            out = self._pack_cache[key] = self.empty(tuple(w.shape))
        nat.call("wsr_cast", w.data_ptr(), nat.F32, out.data_ptr(), self.dt, w.numel(), self.stream)
        self._job(nat.PACK_COPY, w.data_ptr(), out.data_ptr(), self.dt, w.numel(), 1, 1, 1, 1, stable=w.data_ptr() == weight2d.data_ptr())
        self._keep.append(w)
        return out

    # ---- ops -------------------------------------------------------------------------------------------------------
    def _tc_conv_ok(self, x, pc, x2, y, bias=None, rowvec=0, rowvec_ld=0):
        if not self.use_tc:
            return False
        if bias is not None and bias.data_ptr() % 16:
            return False
        if rowvec and (rowvec % 16 or rowvec_ld % 4):
            return False
        ok = (x.dt == nat.BF16 and pc.Cin_pad % 64 == 0 and x.C == pc.Cin_pad and x.ld % 8 == 0 and x.ptr % 16 == 0
              and x.W >= 1)
        if x2 is not None:
            ok = ok and x2.C % 64 == 0 and x2.ld % 8 == 0 and x2.ptr % 16 == 0
        return ok

    def conv(self, x, pc, y, stride=1, upsample=False, bias=True, rowvec=None, rowvec_ld=0, act=nat.ACT_NONE,
             out_scale=1.0, res=None, res_scale=1.0, res2=None, res2_scale=1.0, x2=None, w2=None, extra_bias=None,
             force_simt=False, taps=None, gn=None):
        """y = act(conv(x) [+ conv1x1(x2, w2)] + bias + rowvec) * out_scale + res*res_scale + res2*res2_scale.
        taps: a ``nat.TapTable`` -- run the tap-table variant (``pc.k`` / stride / upsample are then ignored).
        gn = (table, act): x is the RAW tensor; GroupNorm (+act) is applied inside the tcgen05 kernel (``conv_can_fuse_gn``)."""
        if taps is not None:
            assert stride == 1 and not upsample and x2 is None
        d = nat.ConvDesc()
        d.x, d.x_dtype, d.N, d.H, d.W, d.Cin, d.x_ld = x.ptr, x.dt, x.N, x.H, x.W, pc.Cin_pad, x.ld
        assert x.C == pc.Cin_pad, (x.C, pc.Cin_pad)
        d.w, d.w_rows = pc.w.data_ptr(), pc.rows
        if pc.w_vm is not None and taps is None and stride == 1 and not upsample:
            d.w_vmerge = pc.w_vm.data_ptr()
        d.ksize, d.stride, d.upsample = (1 if taps is not None else pc.k), stride, (2 if pc.merged_up else 1) if upsample else 0
        assert upsample or not pc.merged_up or taps is not None
        d.Cout = pc.Cout
        assert y.C == pc.Cout, (y.C, pc.Cout)
        if x2 is not None:
            assert w2.rows == pc.rows and w2.Cout == pc.Cout and x2.C == w2.Cin_pad
            d.x2, d.Cin2, d.x2_ld, d.w2 = x2.ptr, x2.C, x2.ld, w2.w.data_ptr()
        b = extra_bias if extra_bias is not None else (pc.bias if bias else None)
        d.bias = _ptr(b)
        d.rowvec, d.rowvec_ld = (rowvec or 0), rowvec_ld
        d.act, d.out_scale = act, out_scale
        if res is not None:
            d.res, d.res_dtype, d.res_ld, d.res_scale = res.ptr, res.dt, res.ld, res_scale
        if res2 is not None:
            d.res2, d.res2_dtype, d.res2_ld, d.res2_scale = res2.ptr, res2.dt, res2.ld, res2_scale
        d.y, d.y_dtype, d.y_ld = y.ptr, y.dt, y.ld
        if y.st is not None:
            d.gn_stats, d.gn_stats_ld = y.stats_ptr, y.st_ld       # GroupNorm statistics of y come out of the epilogue
        if gn is not None:
            assert taps is None and not force_simt
            d.gn_table, d.gn_table_ld, d.gn_act = gn[0].data_ptr(), gn[0].shape[1], gn[1]
        up = 2 if upsample else 1
        opix = x.N * (x.H * up // stride) * (x.W * up // stride)
        flops = 2 * opix * pc.Cout * (pc.k * pc.k * pc.Cin + (x2.C if x2 is not None else 0))
        # nearest-x2 + 3x3 with phase-merged weights: 4 taps per output pixel are executed instead of 9 (SURVEY 8d asks for both)
        xflops = 2 * opix * pc.Cout * 4 * pc.Cin if (upsample and pc.merged_up) else flops
        if taps is not None:
            opix = x.N * taps.GH * taps.GW
            flops = 2 * opix * pc.Cout * taps.ntaps * pc.Cin
        es = 2 if x.dt == nat.BF16 else 4
        nbytes = x.N * x.H * x.W * x.C * es + opix * pc.Cout * (2 if y.dt == nat.BF16 else 4) + pc.w.numel() * es
        if taps is not None:
            tc = (not force_simt and self._tc_conv_ok(x, pc, x2, y, b, rowvec or 0, rowvec_ld)
                  and (taps.in_sub == 1 or (x.H % 2 == 0 and x.W % 2 == 0)) and not (y.st is not None and taps.out_mul != 1))
            if y.st is not None and taps.out_mul != 1:
                d.gn_stats = 0
            if tc:
                self.n_tc += 1
                self.call("wsr_conv_taps_tc", C.byref(d), C.byref(taps), self.stream, flops=flops, nbytes=nbytes, tag="conv_taps_tc")
            else:
                if self.strict_tc and not force_simt:
                    raise nat.WsrError("strict_tc: taps conv Cin=%d Cout=%d not eligible for the tcgen05 kernel" % (pc.Cin_pad, pc.Cout))
                self.n_simt += 1
                self.call("wsr_conv_taps_simt", C.byref(d), C.byref(taps), self.stream, flops=flops, nbytes=nbytes, tag="conv_taps_simt")
            return y
        if not force_simt and self._tc_conv_ok(x, pc, x2, y, b, rowvec or 0, rowvec_ld):
            self.n_tc += 1
            self.call("wsr_conv_tc", C.byref(d), self.stream, flops=flops, nbytes=nbytes, xflops=xflops,
                      tag="conv_tc" if not self.prof_detail else "conv_tc %4d->%4d k%d s%d%s %dx%d" % (
                          pc.Cin_pad + (x2.C if x2 is not None else 0), pc.Cout, pc.k, stride, "u" if upsample else " ", x.H, x.W))
        else:
            if self.strict_tc and not force_simt:
                raise nat.WsrError("strict_tc: conv Cin=%d Cout=%d k=%d not eligible for the tcgen05 kernel" % (pc.Cin_pad, pc.Cout, pc.k))
            self.n_simt += 1
            self.call("wsr_conv_simt", C.byref(d), self.stream, flops=flops, nbytes=nbytes, tag="conv_simt")
        return y

    def conv_can_fuse_gn(self, x, pc, stride=1, upsample=False, x2=None):
        """True when ``conv(x, pc, ..., gn=...)`` is available for this layer (tcgen05 halo mode)."""
        if not self.use_tc or upsample or stride != 1 or not self._tc_conv_ok(x, pc, x2, None):
            return False
        d = nat.ConvDesc()
        d.x, d.x_dtype, d.N, d.H, d.W, d.Cin, d.x_ld = x.ptr, x.dt, x.N, x.H, x.W, pc.Cin_pad, x.ld
        d.ksize, d.stride, d.upsample = pc.k, 1, 0
        if x2 is not None:
            d.x2, d.Cin2 = x2.ptr, x2.C
        return bool(nat.call("wsr_conv_tc_can_fuse_gn", C.byref(d)))

    def gn_finalize(self, x, gamma, beta, groups, table, eps=1e-5):
        """table (N, C, 2) fp32 <- (scale, shift) of GroupNorm(x) from x's statistics slot."""
        assert x.stats_ptr and table.shape[0] == x.N and table.shape[1] >= x.C
        self.call("wsr_gn_finalize", x.stats_ptr, x.st_ld, x.N, x.H * x.W, x.C, groups, eps, gamma.data_ptr(), beta.data_ptr(),
                  table.data_ptr(), table.shape[1], self.stream, tag="wsr_gn_finalize")
        return table

    def gemm(self, a_ptr, a_dt, a_s, b_ptr, b_dt, b_s, d_ptr, d_dt, d_s, batch, M, N, K, alpha=1.0, bias=None,
             force_simt=False, res=None):
        """D[b][m][n] = alpha * sum_k A[b][m][k] B[b][n][k] (+bias[n]) (+res[b][m][n]).  *_s = (batch stride, row stride,
        k/col stride); res = (ptr, dtype, strides) or None."""
        g = nat.GemmDesc()
        if res is not None:
            g.res, g.res_dtype, (g.res_sb, g.res_sm, g.res_sn) = res
        g.a, g.a_dtype, (g.a_sb, g.a_sm, g.a_sk) = a_ptr, a_dt, a_s
        g.b, g.b_dtype, (g.b_sb, g.b_sn, g.b_sk) = b_ptr, b_dt, b_s
        g.d, g.d_dtype, (g.d_sb, g.d_sm, g.d_sn) = d_ptr, d_dt, d_s
        g.bias = _ptr(bias)
        g.batch, g.M, g.N, g.K, g.alpha = batch, M, N, K, alpha
        # each operand is either K-major (unit k stride) or MN-major (unit row stride, i.e. a transposed view): the
        # tcgen05 kernel consumes both directly, the strided dimension must be a multiple of 8 elements
        def _major_ok(st):
            return (st[2] == 1 and st[1] % 8 == 0) or (st[1] == 1 and st[2] % 8 == 0)
        tc_ok = (self.use_tc and not force_simt and a_dt == nat.BF16 and b_dt == nat.BF16 and _major_ok(a_s) and _major_ok(b_s)
                 and K % 64 == 0 and a_s[0] % 8 == 0 and b_s[0] % 8 == 0 and a_ptr % 16 == 0 and b_ptr % 16 == 0)
        flops = 2 * batch * M * N * K
        if tc_ok:
            self.n_tc += 1
            self.call("wsr_gemm_tc", C.byref(g), self.stream, flops=flops,
                      tag="gemm_tc" if not self.prof_detail else "gemm_tc M%d N%d K%d" % (M, N, K))
        else:
            if self.strict_tc and not force_simt:
                raise nat.WsrError("strict_tc: gemm M=%d N=%d K=%d not eligible for the tcgen05 kernel" % (M, N, K))
            self.n_simt += 1
            self.call("wsr_gemm_simt", C.byref(g), self.stream, flops=flops, tag="gemm_simt")

    def gn_stats(self, x, stats=None, stats_ld=None):
        """Stand-alone statistics pass (only needed for tensors that were not produced by a convolution)."""
        sp = x.stats_ptr if stats is None else stats.data_ptr()
        sl = x.st_ld if stats is None else (stats_ld or 2 * x.C)
        self.call("wsr_gn_stats", x.ptr, x.dt, x.N, x.H * x.W, x.C, x.ld, sp, sl, self.stream,
                  nbytes=x.N * x.H * x.W * x.C * (2 if x.dt == nat.BF16 else 4))

    def gn_apply(self, x, gamma, beta, groups, act, y, eps=1e-5, stats=None, stats_ld=None):
        """y = act(GroupNorm(x)); the statistics come from x's arena slot (filled by the producing convolution)."""
        sp = x.stats_ptr if stats is None else stats.data_ptr()
        sl = x.st_ld if stats is None else (stats_ld or 2 * x.C)
        assert sp, "gn_apply: no statistics attached to the input"
        self.call("wsr_gn_apply", x.ptr, x.dt, x.N, x.H * x.W, x.C, x.ld, sp, sl, gamma.data_ptr(), beta.data_ptr(),
                  groups, eps, act, y.ptr, y.dt, y.ld, self.stream,
                  nbytes=2 * x.N * x.H * x.W * x.C * (2 if x.dt == nat.BF16 else 4))
        return y

    # ---- training step ------------------------------------------------------------------------------------------
    def gn_apply_dropout(self, x, gamma, beta, groups, act, y, p, seed, tag, eps=1e-5):
        assert x.stats_ptr
        self.call("wsr_gn_apply_dropout", x.ptr, x.dt, x.N, x.H * x.W, x.C, x.ld, x.stats_ptr, x.st_ld, gamma.data_ptr(),
                  beta.data_ptr(), groups, eps, act, y.ptr, y.dt, y.ld, float(p), seed if isinstance(seed, C.c_uint64) else int(seed),
                  int(tag), self.stream,
                  nbytes=2 * x.N * x.H * x.W * x.C * (2 if x.dt == nat.BF16 else 4))
        return y

    def gn_bwd(self, x, gamma, beta, groups, act, da, dx, red_ptr, dgamma, dbeta, accumulate=True, colsum=0, colsum_ld=0,
               drop=(0.0, 0, 0), eps=1e-5):
        """Backward of y = dropout(act(GroupNorm(x))): da -> dx (accumulated), dgamma / dbeta accumulated;
        red_ptr: zeroed [N][2C] doubles scratch; colsum: optional [N][colsum_ld] fp32 = per-image column sums of dx."""
        assert x.stats_ptr and da.dt == x.dt and dx.dt == x.dt
        common = (x.ptr, x.dt, x.N, x.H * x.W, x.C, x.ld, x.stats_ptr, x.st_ld, gamma.data_ptr(), beta.data_ptr(), groups, eps,
                  act, da.ptr, da.dt, da.ld, float(drop[0]), drop[1] if isinstance(drop[1], C.c_uint64) else int(drop[1]), int(drop[2]),
                  red_ptr, 2 * x.C)
        nb = x.N * x.H * x.W * x.C * (2 if x.dt == nat.BF16 else 4)
        shape = " C%d %dx%d" % (x.C, x.H, x.W) if self.prof_detail else ""
        self.call("wsr_gn_bwd_reduce", *common, self.stream, nbytes=2 * nb, tag="gn_bwd_reduce" + shape)
        self.call("wsr_gn_bwd_apply", *common, dx.ptr, dx.dt, dx.ld, 1 if accumulate else 0, _ptr(dgamma), _ptr(dbeta),
                  colsum, colsum_ld, self.stream, nbytes=(4 if accumulate else 3) * nb, tag="gn_bwd_apply" + shape)

    def wgrad(self, x, dy, taps, dw, dw_strides, dbias=None, up=1, force_simt=False):
        """dw (fp32 tensor view, strides (tap, co, ci) in elements) += weight gradient; dbias += column sums of dy."""
        d = nat.WgradDesc()
        d.x, d.x_dtype, d.N, d.H, d.W, d.Cin, d.x_ld = x.ptr, x.dt, x.N, x.H, x.W, x.C, x.ld
        d.dy, d.dy_dtype, d.Cout, d.dy_ld = dy.ptr, dy.dt, dy.C, dy.ld
        d.dw = dw.data_ptr()
        d.dw_stap, d.dw_sco, d.dw_sci = dw_strides
        d.up = up
        flops = 2 * x.N * taps.GH * taps.GW * dy.C * x.C * taps.ntaps
        if not force_simt and self._tc_wgrad_ok(x, dy, taps, up):
            d.dbias = 0
            self.n_tc += 1
            self.call("wsr_conv_wgrad_tc", C.byref(d), C.byref(taps), self.stream, flops=flops,
                      tag="wgrad_tc" if not self.prof_detail else "wgrad_tc %4d->%4d t%d %dx%d" % (x.C, dy.C, taps.ntaps, x.H, x.W))
            if dbias is not None:
                self.call("wsr_col_sums", dy.ptr, dy.dt, dy.N * dy.H * dy.W, dy.C, dy.ld, dbias.data_ptr(), self.stream,
                          nbytes=dy.N * dy.H * dy.W * dy.C * 2, tag="col_sums")
            return
        if self.strict_tc and not force_simt:
            raise nat.WsrError("strict_tc: wgrad Cin=%d Cout=%d not eligible for the tcgen05 kernel" % (x.C, dy.C))
        d.dbias = _ptr(dbias)
        self.n_simt += 1
        self.call("wsr_conv_wgrad_simt", C.byref(d), C.byref(taps), self.stream, flops=flops, tag="wgrad_simt")

    def _tc_wgrad_ok(self, x, dy, taps, up):
        if not self.use_tc or x.dt != nat.BF16 or dy.dt != nat.BF16:
            return False
        if x.ld % 8 or dy.ld % 8 or x.ptr % 16 or dy.ptr % 16:
            return False
        if taps.out_mul != 1 or taps.GH != taps.OH or taps.GW != taps.OW:
            return False
        if taps.in_sub > 2 or (taps.in_sub == 2 and (x.H % 2 or x.W % 2)):
            return False
        lw, lh = (x.W, x.H) if up == 2 else (taps.GW, taps.GH)
        t1 = min(lw, 64)
        t2 = min(lh, 64 // t1)
        t3 = min(x.N, 64 // (t1 * t2))
        return t1 * t2 * t3 == 64

    def softmax_bwd(self, p, p_dt, dp, dp_dt, rows, cols, scale, ds, ds_dt):
        self.call("wsr_softmax_bwd_rows", p.data_ptr(), p_dt, dp.data_ptr(), dp_dt, rows, cols, cols, scale, ds.data_ptr(), ds_dt,
                  self.stream)

    def softmax(self, s, s_dt, rows, cols, scale, p, p_dt):
        self.call("wsr_softmax_rows", s.data_ptr(), s_dt, rows, cols, cols, scale, p.data_ptr(), p_dt, cols, self.stream,
                  nbytes=rows * cols * ((2 if s_dt == nat.BF16 else 4) + (2 if p_dt == nat.BF16 else 4)))

    def nchw_to_act(self, src, y):
        src = src.contiguous()
        N, Cc, H, W = src.shape
        nat.call("wsr_nchw_to_nhwc", src.data_ptr(), N, Cc, H, W, y.ptr, y.dt, y.ld, self.stream)
        self._keep_tmp = src
        return y

    # ---- attention (single head, dense softmax; nn_modules/resnet.py:81-100, guided_cross_attention.py:24-44) --------
    def small_attention_takes_nhwc_v(self, Nq, Nk, Cc):
        """True when the fused low-resolution attention kernel can consume V as pixels x channels (no V^T GEMM)."""
        return (self.use_tc and not self.no_fused_attention and bool(nat.call("wsr_attention_small_tc_supported", Nq, Nk, Cc))
                and (Cc // ((Cc + 255) // 256)) % 64 == 0)

    def attention(self, q, k, vT, o, scores, probs, v=None):
        """q, k: Act (B, H, W, C) row-major pixels x channels; vT: tensor (B, C, Nk) (V transposed, K-major for P*V);
        o: Act (B, H, W, C).  scores/probs: scratch tensors (B, Nq, Nk).  v: alternatively V as an Act (pixels x channels, e.g. a slice
        of the q | k | v projection) -- only for shapes with ``small_attention_takes_nhwc_v``."""
        B, Nq, Nk, Cc = q.N, q.H * q.W, k.H * k.W, q.C
        if v is not None:
            assert vT is None and self.small_attention_takes_nhwc_v(Nq, Nk, Cc) and v.dt == nat.BF16 and v.ld % 8 == 0 and v.ptr % 16 == 0
            self.n_tc += 1
            self.call("wsr_attention_small_nhwc_tc", q.ptr, q.ld, k.ptr, k.ld, v.ptr, v.ld, o.ptr, o.ld, B, Nq, Nk, Cc,
                      1.0 / math.sqrt(Cc), self.stream, flops=4 * B * Nq * Nk * Cc,
                      tag="attn_small_tc" if not self.prof_detail else "attn_small_tc N%d d%d" % (Nk, Cc))
            return o
        if (self.use_tc and not self.no_fused_attention and Cc in (64, 128) and Nq % 128 == 0 and Nk % 128 == 0
                and q.dt == nat.BF16 and k.dt == nat.BF16 and o.dt == nat.BF16 and q.ld % 8 == 0 and k.ld % 8 == 0
                and o.ld % 8 == 0 and q.ptr % 16 == 0 and k.ptr % 16 == 0 and o.ptr % 16 == 0):
            self.n_tc += 1
            self.call("wsr_attention_tc", q.ptr, q.ld, k.ptr, k.ld, vT.data_ptr(), o.ptr, o.ld, B, Nq, Nk, Cc,
                      1.0 / math.sqrt(Cc), self.stream, flops=4 * B * Nq * Nk * Cc,
                      tag="attn_tc" if not self.prof_detail else "attn_tc N%d d%d" % (Nk, Cc))
            return o
        if (self.use_tc and not self.no_fused_attention and q.dt == nat.BF16 and k.dt == nat.BF16 and o.dt == nat.BF16
                and q.ld % 8 == 0 and k.ld % 8 == 0 and o.ld % 8 == 0 and q.ptr % 16 == 0 and k.ptr % 16 == 0 and o.ptr % 16 == 0
                and vT.dtype == torch.bfloat16 and nat.call("wsr_attention_small_tc_supported", Nq, Nk, Cc)):
            # low-resolution levels (N <= 512, d <= 512): whole score block in tensor memory, one launch, nothing in HBM
            self.n_tc += 1
            self.call("wsr_attention_small_tc", q.ptr, q.ld, k.ptr, k.ld, vT.data_ptr(), o.ptr, o.ld, B, Nq, Nk, Cc,
                      1.0 / math.sqrt(Cc), self.stream, flops=4 * B * Nq * Nk * Cc,
                      tag="attn_small_tc" if not self.prof_detail else "attn_small_tc N%d d%d" % (Nk, Cc))
            return o
        s_dt = nat.BF16 if scores.dtype == torch.bfloat16 else nat.F32
        p_dt = nat.BF16 if probs.dtype == torch.bfloat16 else nat.F32
        self.gemm(q.ptr, q.dt, (Nq * q.ld, q.ld, 1), k.ptr, k.dt, (Nk * k.ld, k.ld, 1),
                  scores.data_ptr(), s_dt, (Nq * Nk, Nk, 1), B, Nq, Nk, Cc)
        self.softmax(scores, s_dt, B * Nq, Nk, 1.0 / math.sqrt(Cc), probs, p_dt)
        self.gemm(probs.data_ptr(), p_dt, (Nq * Nk, Nk, 1), vT.data_ptr(), self.dt, (Cc * Nk, Nk, 1),
                  o.ptr, o.dt, (Nq * o.ld, o.ld, 1), B, Nq, Cc, Nk)
        return o
