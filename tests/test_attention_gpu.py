"""GPU tests of the attention kernels and of the training step's attention backward, against float64 torch on the same
bf16-rounded operands the kernels read (so what remains is the kernel's own error):

  * the fused forward kernels: wsr_attention_small_nhwc_tc and wsr_attention_small_tc (the sampler's low-resolution levels,
    V as pixels x channels or as V^T) and wsr_attention_tc (the long-sequence levels, sampled softmax shift), plus the unfused
    GEMM -> softmax -> GEMM path of the bf16 and the fp32 engine;
  * the row softmax and its backward at the training step's row lengths;
  * UNetTrainPlan._attention_bwd and UNetTrainPlan._v_bwd, called unbound on a small stand-in for the plan, with the buffer layout
    of the train plan, at its configs[2] shapes and at a batch whose fp32 score scratch passes 2^31 bytes;
  * GEMM operand layouts only that backward uses.

Every check reports three numbers: rel-L2 over the whole output, the worst 128-row tile's rel-L2 (rows = queries, keys or
pixels, per image), and the worst row's max-abs error relative to that row's reference norm.  A wrong tile is 1/256 of an
N = 8192, B = 4 output and would hide in the first number alone.  References at N = 8192 are computed one image at a time.
Outputs written with = start as a NaN sentinel and must be fully overwritten; outputs accumulated with += start from a random
prefill and the test checks prefill + result; channels outside a written slice must stay bit-identical.  Each bound is about
2-3x the value measured on a B200 (1000 W power limit), written beside it."""
import math

import pytest
import torch
import torch.nn.functional as F

import wsr
from conftest import rel_l2

pytestmark = pytest.mark.gpu

nat = wsr.pkg.native
Engine = wsr.sub("engine").Engine
UNetTrainPlan = wsr.sub("unet_train").UNetTrainPlan

F64 = torch.float64
NAN = float("nan")


def _dev():
    return torch.device("cuda:0")


def _gen(seed):
    return torch.Generator(device=_dev()).manual_seed(seed)


def _randn(g, *shape, scale=1.0):
    return torch.randn(*shape, generator=g, device=_dev()) * scale


def _bf16(t):
    return t.to(torch.bfloat16).float()


def _act(eng, B, N, ld, dt=None, fill=NAN):
    """Act (B, 1, N, ld): the kernels see only pixels x channels, so one image row of N pixels stands for h x w."""
    a = eng.new_act(B, 1, N, ld, dt=dt)
    a.buf.fill_(fill)
    return a


def _put(a, x):
    """x: (B, N, C) -> the Act's channel slice (rounded to the Act's dtype)."""
    a.buf[..., a.coff:a.coff + a.C] = x.view(a.N, 1, a.H * a.W, a.C).to(a.buf.dtype)


def _get(a):
    return a.buf[..., a.coff:a.coff + a.C].reshape(a.N, a.H * a.W, a.C).to(F64)


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


def _outside(a):
    """Channels of the Act's buffer outside its slice (a copy)."""
    return torch.cat([a.buf[..., :a.coff], a.buf[..., a.coff + a.C:]], -1).clone()


def _assert_outside_unchanged(a, before):
    assert torch.equal(_bits(_outside(a)), _bits(before)), "channels outside the written slice changed"


class _Err:
    """Error of an output against its reference, accumulated image by image: (rows, cols) float64 tensors."""

    def __init__(self):
        self.d2 = self.r2 = 0.0
        self.tile = self.row = 0.0

    def add(self, got, ref):
        got, ref = got.to(F64), ref.to(F64)
        assert bool(torch.isfinite(got).all()), "non-finite output (sentinel not overwritten?)"
        diff = got - ref
        dr, rr = (diff * diff).sum(-1), (ref * ref).sum(-1)
        self.d2 += float(dr.sum())
        self.r2 += float(rr.sum())
        pad = (-dr.numel()) % 128
        td, tr = F.pad(dr, (0, pad)).view(-1, 128).sum(-1), F.pad(rr, (0, pad)).view(-1, 128).sum(-1)
        self.tile = max(self.tile, float((td / tr.clamp_min(1e-300)).sqrt().max()))
        self.row = max(self.row, float((diff.abs().amax(-1) / rr.sqrt().clamp_min(1e-300)).max()))
        return self

    def check(self, tag, bound):
        l2 = math.sqrt(self.d2 / max(self.r2, 1e-300))
        print("\n[attention] %s: rel-L2 %.2e, worst tile %.2e, worst row %.2e" % (tag, l2, self.tile, self.row))
        b_l2, b_tile, b_row = bound
        assert l2 < b_l2 and self.tile < b_tile and self.row < b_row, (tag, (l2, self.tile, self.row), bound)


def _attn_ref(q, k, v, scale):
    """float64, one image: q (Nq, d), k (Nk, d), v (Nk, d) -> softmax(scale q k^T) v."""
    return torch.softmax((q @ k.T) * scale, -1) @ v


# ----------------------------------------------------------------------------------------------------------------
# 1a. wsr_attention_small_nhwc_tc / wsr_attention_small_tc (attn_small_tc.cu)
# ----------------------------------------------------------------------------------------------------------------
# bounds (rel-L2, worst tile, worst row) against float64; the output is bf16
SMALL_BOUND = (5e-3, 5e-3, 4e-3)       # measured worst over the cases: 1.89e-3, 1.97e-3, 1.57e-3
# V as pixels x channels and V^T feed the same MMAs: the two outputs were bit-identical in every case (measured 0)
SMALL_AGREE = 1e-5

SMALL_CASES = [
    # B, Nq, Nk, d, layout ("qkv": q | k | v in one 3d-channel Act, the self-attention projection; "kv": q alone, k | v in one
    # 2d-channel Act, the HF-CA projections)
    pytest.param(4, 512, 512, 256, "kv", id="hfca-512x256"),                   # sampling plan, HF-CA level 2
    pytest.param(4, 128, 128, 512, "kv", id="hfca-128x512"),                   # HF-CA level 3
    pytest.param(4, 512, 512, 512, "qkv", id="self-512x512"),                  # self-attention at 16x32
    pytest.param(4, 128, 128, 512, "qkv", id="mid-128x512"),
    pytest.param(64, 512, 512, 256, "kv", id="hfca-512x256-B64"),              # the headline batch on one GPU: grid.y = 64
    pytest.param(2, 128, 64, 512, "kv", id="Nk64-d512"),                       # one K piece, 4-stage phase-1 ring wraps
    pytest.param(2, 256, 64, 128, "kv", id="Nq256-Nk64-d128"),
    pytest.param(3, 128, 192, 64, "kv", id="Nk192-d64"),
    pytest.param(2, 256, 320, 128, "kv", id="Nk320-d128"),                     # two K pieces of 160
    pytest.param(2, 384, 448, 384, "kv", id="Nk448-d384"),                     # two K pieces of 224, two V pieces of 192
    pytest.param(2, 256, 256, 192, "qkv", id="self-256x192"),                  # three 64-channel V boxes in one piece
    pytest.param(1, 384, 384, 384, "qkv", id="self-384x384"),
    pytest.param(2, 128, 512, 256, "kv", id="Nq128-Nk512-d256"),
]


def _wide_out(eng, B, N, d):
    """Output slice [64, 64 + d) of a (d + 128)-channel bf16 buffer: random outside, NaN inside."""
    o = eng.new_act(B, 1, N, d + 128).slice(64, d)
    o.buf.copy_(torch.randn(o.buf.shape, generator=_gen(7), device=_dev()).to(o.buf.dtype))
    o.buf[..., 64:64 + d] = NAN
    return o


@pytest.mark.parametrize("B,Nq,Nk,d,layout", SMALL_CASES)
def test_attention_small_tc(B, Nq, Nk, d, layout):
    dev = _dev()
    eng = Engine(dev, "bf16")
    assert nat.call("wsr_attention_small_tc_supported", Nq, Nk, d) == 1
    g = _gen(100 + B + Nq + 3 * Nk + 7 * d)
    q, k, v = _randn(g, B, Nq, d, scale=1.5), _randn(g, B, Nk, d, scale=1.5), _randn(g, B, Nk, d)
    if layout == "qkv":
        assert Nq == Nk
        qkv = _act(eng, B, Nq, 3 * d)
        qa, ka, va = qkv.slice(0, d), qkv.slice(d, d), qkv.slice(2 * d, d)
    else:
        qa = _act(eng, B, Nq, d)
        kv = _act(eng, B, Nk, 2 * d)
        ka, va = kv.slice(0, d), kv.slice(d, d)
    for a, x in ((qa, q), (ka, k), (va, v)):
        _put(a, x)
    vT = va.buf[..., va.coff:va.coff + d].reshape(B, Nk, d).transpose(1, 2).contiguous()
    o_mn, o_t = _wide_out(eng, B, Nq, d), _wide_out(eng, B, Nq, d)
    out_mn, out_t = _outside(o_mn), _outside(o_t)
    scale = 1.0 / math.sqrt(d)
    # V as pixels x channels: the sampling plan's route
    assert eng.small_attention_takes_nhwc_v(Nq, Nk, d)
    eng.attention(qa, ka, None, o_mn, None, None, v=va)
    assert eng.n_tc == 1 and eng.n_simt == 0
    # V^T: through the engine where it routes there; at d = 64 / 128 with Nk % 128 == 0 it routes to wsr_attention_tc instead
    if d in (64, 128) and Nk % 128 == 0:
        nat.call("wsr_attention_small_tc", qa.ptr, qa.ld, ka.ptr, ka.ld, vT.data_ptr(), o_t.ptr, o_t.ld, B, Nq, Nk, d, scale, eng.stream)
    else:
        eng.attention(qa, ka, vT, o_t, None, None)
        assert eng.n_tc == 2 and eng.n_simt == 0
    torch.cuda.synchronize()
    _assert_outside_unchanged(o_mn, out_mn)
    _assert_outside_unchanged(o_t, out_t)
    Q, K, V = _get(qa), _get(ka), _get(va)
    got_mn, got_t = _get(o_mn), _get(o_t)
    e_mn, e_t = _Err(), _Err()
    for b in range(B):
        ref = _attn_ref(Q[b], K[b], V[b], scale)
        e_mn.add(got_mn[b], ref)
        e_t.add(got_t[b], ref)
    tag = "small B%d Nq%d Nk%d d%d %s" % (B, Nq, Nk, d, layout)
    e_mn.check(tag + " nhwc-V", SMALL_BOUND)
    e_t.check(tag + " V^T", SMALL_BOUND)
    agree = rel_l2(got_mn, got_t)
    print("[attention] %s: nhwc-V vs V^T rel-L2 %.2e" % (tag, agree))
    assert agree < SMALL_AGREE


# ----------------------------------------------------------------------------------------------------------------
# 1b. wsr_attention_tc (attn_tc.cu): sampled softmax shift
# ----------------------------------------------------------------------------------------------------------------
TC_BOUND = (6e-3, 6e-3, 6e-3)          # measured worst (incl. the B = 64 case): 2.44e-3, 2.65e-3, 2.43e-3
TC_HOT = (1.0, 0.97, 0.94, 0.91)        # planted keys: score = (sampled maximum + gap) * factor


def _sampled_blocks(Nk):
    """Key blocks of pass A in wsr_attention_tc: na = min(nblocks, 4) blocks, block g * (nblocks // na)."""
    nb = Nk // 128
    na = min(nb, 4)
    return [g * (nb // na) for g in range(na)]


def _stress(q, k, scale, max_gap=40.0):
    """Plant keys in UNSAMPLED key blocks whose scores beat the row's sampled maximum by up to ``max_gap`` natural units (q, k:
    (B, N, d) bf16-valued float32, changed in place).  Channel 0 of every other key is zero, so the sampled maximum does not
    depend on channel 0 of q, which then sets each row's gap exactly; four planted keys with scores in the ratios TC_HOT keep
    the result sensitive to the relative size of large exponentials.  Every 16th row is scaled to near-uniform scores instead."""
    B, Nq, d = q.shape
    Nk = k.shape[1]
    nb = Nk // 128
    samp = _sampled_blocks(Nk)
    free = [j for j in range(nb) if j not in samp] or [nb - 1]
    hot = [free[round(m * (len(free) - 1) / 3)] * 128 + (37 * m + 11) % 128 for m in range(4)]
    c = 4.0
    k[:, :, 0] = 0
    for h, f in zip(hot, TC_HOT):
        k[:, h] = 0
        k[:, h, 0] = c * f
    rows = torch.arange(Nq, device=q.device)
    uniform = rows % 16 == 15
    q[:, uniform] *= 0.02
    q[:, :, 0] = 0
    q.copy_(_bf16(q))
    gap = max_gap * ((rows * 37) % 128).to(F64) / 127
    gap[uniform] = 0
    ks = torch.cat([k[:, j * 128:(j + 1) * 128] for j in samp], 1)
    for b in range(B):
        smax = (q[b].to(F64) @ ks[b].to(F64).T).amax(-1) * scale
        a = (smax + gap) / (c * scale)
        a[uniform] = 0
        q[b, :, 0] = a.float()
    q.copy_(_bf16(q))
    k.copy_(_bf16(k))
    return hot


def _gap(Q, K, scale):
    """Largest (row maximum - maximum over the sampled key blocks) of one image, in natural units."""
    s = (Q @ K.T) * scale
    cols = torch.cat([torch.arange(j * 128, (j + 1) * 128, device=Q.device) for j in _sampled_blocks(K.shape[0])])
    return float((s.amax(-1) - s[:, cols].amax(-1)).max())


TC_CASES = [
    # B, Nq, Nk, d, stress
    pytest.param(4, 8192, 8192, 64, True, id="8192x64-B4"),             # configs[2] HF-CA level 0
    pytest.param(2, 8192, 8192, 128, True, id="8192x128-B2"),           # configs[4] HF-CA level 0
    pytest.param(2, 2048, 2048, 128, True, id="2048x128"),
    pytest.param(2, 2048, 2048, 64, False, id="2048x64-plain"),
    pytest.param(2, 128, 128, 64, True, id="N128"),                       # 1-4 key blocks: the shift is the exact maximum
    pytest.param(2, 256, 256, 128, True, id="N256"),
    pytest.param(2, 384, 384, 64, True, id="N384"),
    pytest.param(2, 512, 512, 128, True, id="N512"),
    pytest.param(2, 640, 640, 64, True, id="N640"),                       # 5 blocks: stride_a 1 with a remainder
    pytest.param(2, 1152, 1152, 128, True, id="N1152"),                   # 9 blocks: stride_a 2 with a remainder
    pytest.param(2, 128, 8192, 64, True, id="Nq128-Nk8192"),
    pytest.param(1, 8192, 128, 128, True, id="Nq8192-Nk128"),
]


def _tc_inputs(eng, B, Nq, Nk, d, stress, seed):
    """q, k (Acts: slices of one 2d-channel Act when Nq == Nk, as the self-attention's q | k; else separate), vT (B, d, Nk)."""
    g = _gen(seed)
    q, k, v = _randn(g, B, Nq, d, scale=1.5), _randn(g, B, Nk, d, scale=1.5), _randn(g, B, Nk, d)
    q, k = _bf16(q), _bf16(k)
    scale = 1.0 / math.sqrt(d)
    if stress:
        _stress(q, k, scale)
    if Nq == Nk:
        qk = _act(eng, B, Nq, 2 * d)
        qa, ka = qk.slice(0, d), qk.slice(d, d)
    else:
        qa, ka = _act(eng, B, Nq, d), _act(eng, B, Nk, d)
    _put(qa, q)
    _put(ka, k)
    vT = v.transpose(1, 2).contiguous().to(torch.bfloat16)
    return qa, ka, vT


def _check_tc(qa, ka, vT, o, images, tag, stress):
    d = qa.C
    scale = 1.0 / math.sqrt(d)
    Q, K, V, got = _get(qa), _get(ka), vT.to(F64).transpose(1, 2), _get(o)
    err, gap = _Err(), 0.0
    for b in images:
        err.add(got[b], _attn_ref(Q[b], K[b], V[b], scale))
        gap = max(gap, _gap(Q[b], K[b], scale))
    print("\n[attention] %s: largest gap between the row maximum and the sampled maximum %.1f" % (tag, gap))
    # the +64 exponent clamp (log2 units) is exact up to a 44-unit gap; the stress cases use the domain up to 40
    assert gap < 44.0
    if stress and K.shape[1] // 128 > 4:
        assert gap > 35.0
    err.check(tag, TC_BOUND)


@pytest.mark.parametrize("B,Nq,Nk,d,stress", TC_CASES)
def test_attention_tc(B, Nq, Nk, d, stress):
    eng = Engine(_dev(), "bf16")
    qa, ka, vT = _tc_inputs(eng, B, Nq, Nk, d, stress, 200 + B + Nq + 3 * Nk + d)
    o = _wide_out(eng, B, Nq, d)
    out = _outside(o)
    eng.attention(qa, ka, vT, o, None, None)
    assert eng.n_tc == 1 and eng.n_simt == 0
    torch.cuda.synchronize()
    _assert_outside_unchanged(o, out)
    _check_tc(qa, ka, vT, o, range(B), "tc B%d Nq%d Nk%d d%d%s" % (B, Nq, Nk, d, " stress" if stress else ""), stress)


def test_attention_tc_headline_batch():
    """B = 64 at N = 8192 (grid.y = 64): images 0, 1, 63 and a seeded sample are checked."""
    B, N, d = 64, 8192, 64
    eng = Engine(_dev(), "bf16")
    qa, ka, vT = _tc_inputs(eng, B, N, N, d, True, 300)
    o = _wide_out(eng, B, N, d)
    eng.attention(qa, ka, vT, o, None, None)
    assert eng.n_tc == 1
    torch.cuda.synchronize()
    assert bool(torch.isfinite(o.buf[..., 64:64 + d]).all())
    sample = torch.randperm(B - 3, generator=torch.Generator().manual_seed(5))[:2] + 2
    _check_tc(qa, ka, vT, o, [0, 1, 63] + sample.tolist(), "tc B64 N8192 d64 stress", True)


# ----------------------------------------------------------------------------------------------------------------
# 1c. unfused GEMM -> softmax -> GEMM (Engine.attention's last route)
# ----------------------------------------------------------------------------------------------------------------
UNFUSED_BOUND = {"bf16": (6e-3, 6e-3, 4e-3),      # measured worst: 2.37e-3, 2.52e-3, 1.58e-3
                 "fp32": (6e-6, 7e-6, 3e-6)}      # measured worst: 2.45e-6, 2.88e-6, 1.27e-6


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
@pytest.mark.parametrize("N,d,no_fused", [(2048, 256, False), (128, 1024, False), (512, 1024, False), (512, 256, True)],
                         ids=["2048x256", "128x1024", "512x1024", "512x256-no-fused"])
def test_attention_unfused(mode, N, d, no_fused):
    """configs[4]'s (2048, 256), (128, 1024) and (512, 1024), which no fused kernel takes, and one shape that would be fused."""
    B = 2
    eng = Engine(_dev(), mode)
    eng.no_fused_attention = no_fused
    g = _gen(400 + N + d)
    qa, ka = _act(eng, B, N, d), _act(eng, B, N, d)
    _put(qa, _randn(g, B, N, d, scale=1.5))
    _put(ka, _randn(g, B, N, d, scale=1.5))
    vT = _randn(g, B, d, N).to(eng.tdt)
    o = _act(eng, B, N, d)
    scores = torch.full((B * N * N,), NAN, device=_dev())
    probs = torch.full((B * N * N,), NAN, device=_dev(), dtype=eng.tdt)
    eng.attention(qa, ka, vT, o, scores, probs)
    assert (eng.n_tc, eng.n_simt) == ((2, 0) if mode == "bf16" else (0, 2))
    torch.cuda.synchronize()
    Q, K, V, got = _get(qa), _get(ka), vT.to(F64).transpose(1, 2), _get(o)
    err = _Err()
    for b in range(B):
        err.add(got[b], _attn_ref(Q[b], K[b], V[b], 1.0 / math.sqrt(d)))
    err.check("unfused %s B%d N%d d%d%s" % (mode, B, N, d, " no_fused_attention" if no_fused else ""), UNFUSED_BOUND[mode])


# ----------------------------------------------------------------------------------------------------------------
# 2. wsr_softmax_rows (block kernel) and wsr_softmax_bwd_rows at the training widths
# ----------------------------------------------------------------------------------------------------------------
SOFTMAX_BOUND = {nat.F32: (6e-8, 6e-8, 1.2e-7),      # measured worst: 2.54e-8, 2.54e-8, 5.23e-8
                 nat.BF16: (1.2e-3, 1.2e-3, 2.5e-3)}   # measured worst: 4.83e-4, 4.83e-4, 1.09e-3


@pytest.mark.parametrize("p_dt", [nat.F32, nat.BF16], ids=["P-fp32", "P-bf16"])
@pytest.mark.parametrize("cols", [1000, 2048, 8192])
def test_softmax_rows_block_kernel(cols, p_dt):
    """Row lengths that are not multiples of 128 or exceed 1024 take the block-per-row kernel; 37 rows (not a multiple of 8),
    row 3 dominated by one logit, row 4 constant."""
    rows, scale = 37, 0.125
    eng = Engine(_dev(), "fp32")
    s = _randn(_gen(500 + cols), rows, cols, scale=8.0)
    s[3, 5] = 400.0
    s[4] = 1.5
    p = torch.full((rows, cols), NAN, device=_dev(), dtype=torch.float32 if p_dt == nat.F32 else torch.bfloat16)
    eng.softmax(s, nat.F32, rows, cols, scale, p, p_dt)
    torch.cuda.synchronize()
    ref = torch.softmax(s.to(F64) * scale, -1)
    assert float(p[3, 5]) == pytest.approx(1.0, abs=1e-6)
    _Err().add(p, ref).check("softmax cols %d P %s" % (cols, "fp32" if p_dt == nat.F32 else "bf16"), SOFTMAX_BOUND[p_dt])


SOFTMAX_BWD_BOUND = {"bf16": (4.5e-3, 4.5e-3, 6e-3),   # measured worst: 1.82e-3, 1.82e-3, 2.58e-3
                     "fp32": (1.2e-7, 1.2e-7, 6e-7)}    # measured worst: 4.62e-8, 4.62e-8, 2.43e-7


@pytest.mark.parametrize("dts", ["bf16", "fp32"], ids=["P-bf16-dP-fp32-dS-bf16", "all-fp32"])
@pytest.mark.parametrize("cols", [128, 512, 2048, 8192])
def test_softmax_bwd_rows(cols, dts):
    """dS = scale * P * (dP - rowsum(P * dP)); (P, dP, dS) = (bf16, fp32, bf16) is what the bf16 training step uses.
    Row 0 is one-hot, where dS is exactly 0."""
    rows, scale = 37, 0.125
    eng = Engine(_dev(), "fp32")
    g = _gen(600 + cols)
    tdt = torch.bfloat16 if dts == "bf16" else torch.float32
    pdt = nat.BF16 if dts == "bf16" else nat.F32
    P = torch.softmax(_randn(g, rows, cols, scale=2.0), -1).to(tdt)
    P[0] = 0
    P[0, cols // 3] = 1
    dP = _randn(g, rows, cols)
    dS = torch.full((rows, cols), NAN, device=_dev(), dtype=tdt)
    eng.softmax_bwd(P, pdt, dP, nat.F32, rows, cols, scale, dS, pdt)
    torch.cuda.synchronize()
    p64, dp64 = P.to(F64), dP.to(F64)
    ref = scale * p64 * (dp64 - (p64 * dp64).sum(-1, keepdim=True))
    assert float(dS[0].float().abs().max()) == 0.0
    _Err().add(dS[1:], ref[1:]).check("softmax_bwd cols %d %s" % (cols, dts), SOFTMAX_BWD_BOUND[dts])


# ----------------------------------------------------------------------------------------------------------------
# 3. the training step's attention backward: UNetTrainPlan._attention_bwd / _v_bwd
# ----------------------------------------------------------------------------------------------------------------
class _PlanStub:
    """What _attention_bwd / _v_bwd read from the plan: the engine, the batch, the shared attention scratch, _on_side."""

    def __init__(self, eng, B, scratch):
        self.eng, self.B = eng, B
        self.scores, self.probs, self.dP, self.dS = scratch

    def _on_side(self, launch):
        launch()


def _scratch(eng, n):
    """S and dP fp32, P and dS in the engine dtype, as the train plan allocates them; NaN, so stale reads show."""
    dev = _dev()
    return tuple(torch.full((n,), NAN, device=dev, dtype=t) for t in (torch.float32, eng.tdt, torch.float32, eng.tdt))


# measured worst over the cases beside each bound.  dn is bf16 in the bf16 engine and holds prefill + gradient: its rows are
# rounded relative to the prefill, which is why its worst row is further from its rel-L2 than the others'.
BWD_BOUND = {
    "bf16": {"dq": (7e-3, 9e-3, 1.2e-2),        # 2.86e-3, 3.63e-3, 4.96e-3
             "dk": (7e-3, 8.5e-3, 8e-3),        # 2.79e-3, 3.40e-3, 3.27e-3
             "dvT": (6e-3, 7e-3, 6.5e-3),       # 2.35e-3, 2.82e-3, 2.68e-3
             "dn": (6e-3, 7e-3, 4.5e-2),        # 2.35e-3, 2.93e-3, 1.90e-2
             "dWv": (2.5e-5, 2.5e-5, 1.2e-5)},  # 9.63e-6, 9.63e-6, 4.94e-6
    "fp32": {"dq": (5e-6, 5.5e-6, 8e-6),        # 2.03e-6, 2.28e-6, 3.31e-6
             "dk": (5e-6, 5.5e-6, 1e-5),        # 2.02e-6, 2.29e-6, 4.15e-6
             "dvT": (5e-6, 6e-6, 8e-6),         # 2.06e-6, 2.36e-6, 3.29e-6
             "dn": (1e-6, 1e-6, 7e-7),          # 4.09e-7, 4.15e-7, 2.79e-7
             "dWv": (4e-6, 4e-6, 3e-6)},        # 1.64e-6, 1.64e-6, 1.26e-6
}

BWD_CASES = [
    # B, N, C, kind ("hfca": separate q and k Acts; "self": q | k in one 2C-channel Act), scratch ("shared": the plan's; "private":
    # the HF-CA branch stream's own tuple, passed as scratch=)
    pytest.param(4, 8192, 64, "hfca", "shared", id="hfca-8192x64"),            # configs[2], B = 4 train plan
    pytest.param(4, 2048, 128, "hfca", "shared", id="hfca-2048x128"),
    pytest.param(4, 512, 256, "hfca", "shared", id="hfca-512x256"),
    pytest.param(4, 128, 512, "hfca", "shared", id="hfca-128x512"),
    pytest.param(4, 512, 512, "self", "shared", id="self-512x512"),
    pytest.param(4, 128, 512, "self", "shared", id="mid-128x512"),
    pytest.param(2, 8192, 128, "hfca", "shared", id="hfca-8192x128-B2"),       # inner 128
    pytest.param(4, 2048, 128, "hfca", "private", id="hfca-2048x128-private"),
    pytest.param(9, 8192, 64, "hfca", "shared", id="hfca-8192x64-B9"),         # fp32 scores: 2.4 GB, offsets past 2^31 bytes
]


def _bwd_ref(q, k, vT, do, scale):
    """float64 autograd, one image: o = softmax(scale q k^T) v with v = vT^T -> (dq, dk, dvT)."""
    q, k, vT = (t.detach().clone().requires_grad_(True) for t in (q, k, vT))
    o = torch.softmax((q @ k.T) * scale, -1) @ vT.T
    return torch.autograd.grad(o, (q, k, vT), do)


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
@pytest.mark.parametrize("B,N,C,kind,scratch", BWD_CASES)
def test_attention_backward(mode, B, N, C, kind, scratch):
    dev = _dev()
    eng = Engine(dev, mode)
    g = _gen(700 + B + N + C + (1 if kind == "self" else 0))
    n = B * N * N
    shared = _scratch(eng, n + 4096)                 # the plan's scratch is sized for its largest attention
    stub = _PlanStub(eng, B, shared)
    private = _scratch(eng, n) if scratch == "private" else None
    if kind == "self":
        qk, d_qk = _act(eng, B, N, 2 * C), _act(eng, B, N, 2 * C)
        qa, ka, dq, dk = qk.slice(0, C), qk.slice(C, C), d_qk.slice(0, C), d_qk.slice(C, C)
    else:
        qa, ka, dq, dk = _act(eng, B, N, C), _act(eng, B, N, C), _act(eng, B, N, C), _act(eng, B, N, C)
    _put(qa, _randn(g, B, N, C, scale=1.5))
    _put(ka, _randn(g, B, N, C, scale=1.5))
    vT = _randn(g, B, C, N).to(eng.tdt)
    do = _act(eng, B, N, C)
    _put(do, _randn(g, B, N, C))
    dvT = torch.full((B, C, N), NAN, device=dev, dtype=eng.tdt)
    UNetTrainPlan._attention_bwd(stub, qa, ka, vT, do, dq, dk, dvT, scratch=private)
    assert (eng.n_tc, eng.n_simt) == ((5, 0) if mode == "bf16" else (0, 5))
    torch.cuda.synchronize()
    for t in shared:                                  # beyond n, and entirely when a private tuple is passed, nothing is written
        tail = t[n:] if private is None else t
        assert bool(torch.isnan(tail.float()).all())
    images = range(B) if B <= 4 else [0, B // 2, B - 1]
    scale = 1.0 / math.sqrt(C)
    Q, K, V, DO = _get(qa), _get(ka), vT.to(F64), _get(do)
    DQ, DK, DV = _get(dq), _get(dk), dvT.to(F64)
    errs = {"dq": _Err(), "dk": _Err(), "dvT": _Err()}
    for b in images:
        rq, rk, rv = _bwd_ref(Q[b], K[b], V[b], DO[b], scale)
        errs["dq"].add(DQ[b], rq)
        errs["dk"].add(DK[b], rk)
        errs["dvT"].add(DV[b].T, rv.T)
        del rq, rk, rv
    tag = "bwd %s %s B%d N%d C%d %s" % (mode, kind, B, N, C, scratch)
    for name in ("dq", "dk", "dvT"):
        errs[name].check(tag + " " + name, BWD_BOUND[mode][name])

    # _v_bwd with the dvT the step just produced: vT = Wv n^T  ->  dn += dvT^T Wv (in place through res), dWv += sum_b dvT n
    wv = _randn(g, C, C, scale=1.0 / math.sqrt(C))
    wv_packed = eng.pack_rows(wv)
    nact = _act(eng, B, N, C)
    _put(nact, _randn(g, B, N, C))
    W64, N64 = wv_packed.to(F64).requires_grad_(True), _get(nact).requires_grad_(True)
    rw, rn = torch.autograd.grad(W64 @ N64.transpose(1, 2), (W64, N64), DV)
    dn = _act(eng, B, N, C)
    _put(dn, _randn(g, B, N, C, scale=float(rn.std())))
    dn0 = _get(dn)
    dwbuf = _randn(g, 2 * C, C, scale=float(rw.std()))
    dw0 = dwbuf.clone()
    n_tc, n_simt = eng.n_tc, eng.n_simt
    UNetTrainPlan._v_bwd(stub, wv_packed, nact, dvT, dn, dwbuf[C:])
    assert (eng.n_tc - n_tc, eng.n_simt - n_simt) == ((1 + B, 0) if mode == "bf16" else (0, 1 + B))
    torch.cuda.synchronize()
    assert torch.equal(dwbuf[:C], dw0[:C])
    err_n = _Err()
    got_n = _get(dn) - dn0
    for b in range(B):
        err_n.add(got_n[b], rn[b])
    err_n.check(tag + " dn", BWD_BOUND[mode]["dn"])
    _Err().add(dwbuf[C:].to(F64) - dw0[C:].to(F64), rw).check(tag + " dWv", BWD_BOUND[mode]["dWv"])


# ----------------------------------------------------------------------------------------------------------------
# 4. GEMM operand layouts only the attention backward uses (bf16 operands, tcgen05)
# ----------------------------------------------------------------------------------------------------------------
GEMM_BOUND = {nat.F32: (2.5e-6, 2.5e-6, 1e-6),     # measured worst: 9.91e-7, 9.91e-7, 3.87e-7
              nat.BF16: (6e-3, 6e-3, 4e-3)}       # measured: 2.35e-3, 2.37e-3, 1.63e-3 (bf16 output rounding)


def _gemm_case(case, g):
    """Stored bf16 operands, their strides and the logical (batch, M, K) / (batch, N, K) float64 views."""
    bf = torch.bfloat16
    if case == "b-mn-shared":
        batch, M, N, K = 3, 512, 128, 128
        a, a_s = _randn(g, batch, K, M).to(bf), (K * M, 1, M)             # A[b][m][k] = a[b][k][m]
        b, b_s = _randn(g, K, N).to(bf), (0, 1, N)                        # B[n][k] = b[k][n], the same for every image
    elif case == "a-mn-m64-wide-pitch":
        batch, M, N, K, lda = 2, 64, 256, 512, 200
        a, a_s = _randn(g, batch, K, lda).to(bf), (K * lda, 1, lda)
        b, b_s = _randn(g, batch, N, K).to(bf), (N * K, K, 1)
    else:
        batch, M, N, K = 2, 256, 128, 128
        a, a_s = _randn(g, batch, M, K).to(bf), (M * K, K, 1)
        b, b_s = _randn(g, batch, N, K).to(bf), (N * K, K, 1)
    A = torch.as_strided(a, (batch, M, K), a_s).to(F64)
    Bm = torch.as_strided(b, (batch, N, K), b_s).to(F64)
    return (batch, M, N, K), (a, a_s), (b, b_s), A, Bm


@pytest.mark.parametrize("case", ["b-mn-shared", "a-mn-m64-wide-pitch", "res-is-d-bf16", "res-is-d-fp32"])
def test_gemm_backward_layouts(case):
    """b-mn-shared: B MN-major with b_sb = 0 and batch 3 (the dn GEMM of _v_bwd); a-mn-m64-wide-pitch: A MN-major, M = 64, row
    pitch 200 > M; res-is-d-*: D += A B^T in place (res aliases D), bf16 and fp32 D."""
    dev = _dev()
    eng = Engine(dev, "bf16")
    g = _gen(800 + len(case))
    (batch, M, N, K), (a, a_s), (b, b_s), A, Bm = _gemm_case(case, g)
    ref = torch.einsum("bmk,bnk->bmn", A, Bm)
    d_dt = nat.BF16 if case == "res-is-d-bf16" else nat.F32
    dt = torch.bfloat16 if d_dt == nat.BF16 else torch.float32
    inplace = case.startswith("res-is-d")
    d = _randn(g, batch, M, N, scale=float(ref.std())).to(dt) if inplace else torch.full((batch, M, N), NAN, device=dev, dtype=dt)
    d0 = d.to(F64) if inplace else 0
    d_s = (M * N, N, 1)
    eng.gemm(a.data_ptr(), nat.BF16, a_s, b.data_ptr(), nat.BF16, b_s, d.data_ptr(), d_dt, d_s, batch, M, N, K,
             res=(d.data_ptr(), d_dt, d_s) if inplace else None)
    assert eng.n_tc == 1 and eng.n_simt == 0
    torch.cuda.synchronize()
    got = d.to(F64) - d0
    err = _Err()
    for i in range(batch):
        err.add(got[i], ref[i])
    err.check("gemm " + case, GEMM_BOUND[d_dt])


def test_gemm_per_image_accumulation():
    """dw_launches of _v_bwd: one launch per image into the same fp32 D (d_sb = 0, res = D), A K-major, B MN-major with a pixel
    pitch wider than N."""
    dev = _dev()
    eng = Engine(dev, "bf16")
    g = _gen(900)
    batch, M, N, K, ldb = 3, 128, 128, 1024, 136
    a = _randn(g, batch, M, K).to(torch.bfloat16)                       # A_i = dvT[i] (channels x pixels)
    b = _randn(g, batch, K, ldb).to(torch.bfloat16)                     # B_i[n][k] = nbuf[i][k][n]
    ref = torch.einsum("bmk,bkn->mn", a.to(F64), b[..., :N].to(F64))
    d = _randn(g, M, N, scale=float(ref.std()))
    d0 = d.to(F64)
    for i in range(batch):
        eng.gemm(a[i].data_ptr(), nat.BF16, (0, K, 1), b[i].data_ptr(), nat.BF16, (0, 1, ldb), d.data_ptr(), nat.F32, (0, N, 1),
                 1, M, N, K, res=(d.data_ptr(), nat.F32, (0, N, 1)))
    assert eng.n_tc == batch and eng.n_simt == 0
    torch.cuda.synchronize()
    _Err().add(d.to(F64) - d0, ref).check("gemm per-image accumulation", GEMM_BOUND[nat.F32])
