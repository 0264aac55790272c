"""GPU unit tests of the individual kernels, called through the C ABI (ctypes), against plain PyTorch fp32 on the same
device.  Tolerances: fp32 SIMT kernels 2e-5 rel-L2 (summation order); bf16 tcgen05 kernels are compared with the SIMT
kernel on the SAME bf16 inputs (both accumulate in fp32) at 2e-3 rel-L2 after bf16 output rounding."""
import math

import pytest
import torch
import torch.nn.functional as F

import wsr
from conftest import rel_l2

pytestmark = pytest.mark.gpu

# the PyTorch side must be a true fp32 reference: no TF32 in cuDNN / cuBLAS
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False

nat = wsr.pkg.native
engine_mod = wsr.sub("engine")
Engine, Act = engine_mod.Engine, engine_mod.Act
T = wsr.sub("taps")


def _dev():
    return torch.device("cuda:0")


def _nhwc(x, eng, ld=None, coff=0, dt=None):
    """NCHW fp32 tensor -> Act (optionally embedded at channel offset coff of a wider buffer)."""
    N, C, H, W = x.shape
    full = eng.new_act(N, H, W, ld or C, dt=dt, zero=True)
    a = full.slice(coff, C)
    eng.nchw_to_act(x, a)
    return a


def _ref_conv(x, w, b, stride=1, upsample=False):
    if upsample:
        x = F.interpolate(x, scale_factor=2, mode="nearest")
    return F.conv2d(x, w, b, stride=stride, padding=(w.shape[-1] - 1) // 2)


CONV_CASES = [
    # N, Cin, Cout, H, W, k, stride, upsample
    (2, 64, 64, 16, 32, 3, 1, False),
    (1, 128, 64, 8, 16, 3, 1, False),
    (2, 64, 128, 16, 32, 1, 1, False),
    (2, 64, 64, 16, 32, 3, 2, False),
    (1, 64, 64, 8, 16, 3, 1, True),
    (3, 192, 256, 4, 8, 3, 1, False),
    (2, 64, 64, 2, 4, 3, 1, False),
    (1, 64, 128, 32, 256, 3, 1, False),
    # tiles that are segments of one image row -> "halo" mode of the tcgen05 kernel (one activation fetch per 9 taps)
    (2, 128, 64, 5, 128, 3, 1, False),
    (1, 192, 256, 3, 256, 3, 1, False),
    (1, 64, 64, 3, 128, 3, 1, True),
    # even row counts -> two output rows per tile (two TMEM accumulators share each weight tile)
    (2, 64, 64, 4, 256, 3, 1, False),
    (1, 128, 128, 6, 128, 3, 1, False),
    (1, 64, 64, 4, 128, 3, 1, True),
]


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_simt_fp32_vs_torch(case):
    N, Cin, Cout, H, W, k, stride, up = case
    torch.manual_seed(0)
    dev = _dev()
    eng = Engine(dev, "fp32")
    x = torch.randn(N, Cin, H, W, device=dev)
    w = torch.randn(Cout, Cin, k, k, device=dev) / math.sqrt(Cin * k * k)
    b = torch.randn(Cout, device=dev)
    ref = _ref_conv(x, w, b, stride, up)
    pc = eng.pack_conv(w, b)
    y = eng.new_act(N, ref.shape[2], ref.shape[3], Cout)
    eng.conv(_nhwc(x, eng), pc, y, stride=stride, upsample=up)
    assert rel_l2(y.to_nchw(eng), ref) < 2e-5


def test_conv_simt_odd_channels_and_epilogue():
    torch.manual_seed(1)
    dev = _dev()
    eng = Engine(dev, "fp32")
    N, Cin, Cout, H, W = 2, 5, 7, 8, 16
    x = torch.randn(N, Cin, H, W, device=dev)
    w = torch.randn(Cout, Cin, 3, 3, device=dev) * 0.2
    b = torch.randn(Cout, device=dev)
    rv = torch.randn(N, 11, device=dev)
    res = torch.randn(N, Cout, H, W, device=dev)
    x2 = torch.randn(N, 3, H, W, device=dev)
    w2 = torch.randn(Cout, 3, 1, 1, device=dev)
    ref = F.leaky_relu(F.conv2d(x, w, b, padding=1) + F.conv2d(x2, w2) + rv[:, 2:2 + Cout, None, None], 0.2) * 0.5 + 0.25 * res
    y = eng.new_act(N, H, W, 16).slice(4, Cout)
    eng.conv(_nhwc(x, eng, ld=8, coff=1), eng.pack_conv(w, b), y, rowvec=rv.data_ptr() + 8, rowvec_ld=11,
             act=nat.ACT_LRELU02, out_scale=0.5, res=_nhwc(res, eng), res_scale=0.25, x2=_nhwc(x2, eng), w2=eng.pack_conv(w2, None))
    assert rel_l2(y.to_nchw(eng), ref) < 2e-5


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_tc_vs_simt(case):
    N, Cin, Cout, H, W, k, stride, up = case
    torch.manual_seed(2)
    dev = _dev()
    eng = Engine(dev, "bf16")
    assert eng.use_tc, "tcgen05 path needs an sm_100 device"
    x = torch.randn(N, Cin, H, W, device=dev)
    w = torch.randn(Cout, Cin, k, k, device=dev) / math.sqrt(Cin * k * k)
    b = torch.randn(Cout, device=dev)
    rv = torch.randn(N, Cout, device=dev)
    OH, OW = (H * (2 if up else 1)) // stride, (W * (2 if up else 1)) // stride
    res = torch.randn(N, Cout, OH, OW, device=dev)
    pc = eng.pack_conv(w, b)
    xa, ra = _nhwc(x, eng), _nhwc(res, eng)
    y_tc = eng.new_act(N, OH, OW, Cout, zero=True)
    y_si = eng.new_act(N, OH, OW, Cout, dt=nat.F32, zero=True)
    kw = dict(stride=stride, upsample=up, rowvec=rv.data_ptr(), rowvec_ld=Cout, res=ra)
    eng.conv(xa, pc, y_tc, **kw)
    eng.conv(xa, pc, y_si, force_simt=True, **kw)
    assert eng.n_tc == 1 and eng.n_simt == 1
    torch.cuda.synchronize()
    err = rel_l2(y_tc.to_nchw(eng), y_si.to_nchw(eng))
    assert err < 4e-3, err
    # and against fp32 torch on the bf16-rounded operands
    ref = _ref_conv(x.bfloat16().float(), w.bfloat16().float(), b, stride, up) + rv[:, :, None, None] + res.bfloat16().float()
    assert rel_l2(y_si.to_nchw(eng), ref) < 1e-4


SPLITK_CASES = [
    # N, Cin, Cout, H, W, k, stride, up, Cin2 (fused 1x1 segment), expect a split.  Every split case has 64-column tiles.
    pytest.param(8, 512, 512, 8, 16, 3, 1, False, 0, True, id="3x3-8x16"),           # 64 tiles, 72 K blocks: halved over 2-CTA clusters
    pytest.param(8, 512, 512, 8, 16, 3, 1, False, 1024, True, id="3x3-res_conv"),    # ... + the 1x1 res_conv as a second K segment (88)
    pytest.param(8, 640, 512, 8, 16, 3, 1, True, 0, True, id="merged-upsample"),     # phase-merged nearest-x2 + 3x3, 4 launches of 40
    pytest.param(8, 512, 512, 16, 32, 3, 2, False, 0, True, id="stride2"),           # phase-subsampled tensor maps
    pytest.param(3, 576, 256, 4, 8, 3, 1, False, 0, True, id="uneven-partial"),      # 81 K blocks split 41 / 40, partial 96-row tile
    pytest.param(4, 256, 512, 8, 16, 4, 1, "dgrad", 0, True, id="taps-dgrad"),       # tap table: dgrad of nearest-x2 + 3x3, 16 taps, 64 K blocks
    pytest.param(64, 256, 512, 8, 16, 4, 1, "dgrad", 0, False, id="taps-dgrad-b64"), # ... at 64 images: 128 tiles of 256 columns
    pytest.param(8, 512, 512, 8, 16, 1, 1, False, 0, False, id="1x1"),               # 1x1: the K loop is too short to pay for the exchange
    pytest.param(8, 512, 512, 16, 32, 3, 1, False, 0, False, id="3x3-16x32"),        # 128 tiles of 128 columns: no room for a second CTA
    pytest.param(8, 1024, 512, 16, 32, 3, 1, False, 0, False, id="3x3-16x32-1024"),  # ... with a longer K loop
    pytest.param(64, 512, 512, 8, 16, 3, 1, False, 0, False, id="3x3-8x16-b64"),     # enough tiles: no split
]


@pytest.mark.parametrize("N, Cin, Cout, H, W, k, stride, up, Cin2, expect", SPLITK_CASES)
def test_conv_tc_split_k_vs_simt(N, Cin, Cout, H, W, k, stride, up, Cin2, expect):
    """Split-K of the classic-mode tcgen05 convolution: only the cut that measured faster on B200 -- the unsplit tile shape with its K
    loop halved over a 2-CTA cluster, for 3x3 convolutions whose tiles fill at most half of the SMs.  The two CTAs each accumulate half
    of the K blocks and exchange fp32 partial tiles through distributed shared memory; distributed fix-up with bias / time-embedding
    row / residual / GroupNorm statistics in the epilogue; compared with the SIMT kernel on the same bf16 operands, run twice, and the
    split (or its absence) checked through wsr_debug_last_tc_config."""
    _split_k_case(N, Cin, Cout, H, W, k, stride, up, Cin2, expect)


PAIR_CASES = [
    # N, Cin, Cout, H, W, k, stride, up, Cin2: classic-mode launches with 256-column tiles and an even number of row tiles
    (64, 512, 512, 8, 16, 3, 1, False, 0),
    (64, 512, 512, 8, 16, 3, 1, False, 1024),          # fused 1x1 res_conv segment (second weight map)
    (64, 256, 512, 16, 32, 3, 2, False, 0),            # stride 2 (phase-subsampled activation maps)
    (64, 512, 512, 8, 16, 3, 1, True, 0),              # nearest-x2 + 3x3, four phase launches
    (64, 512, 1536, 8, 16, 1, 1, False, 0),            # 1x1 q | k | v projection, 6 column tiles
    (64, 256, 768, 8, 16, 3, 1, False, 0),             # odd number of column tiles
    (16, 768, 256, 32, 64, 3, 1, False, 0),            # 64-pixel rows (two image rows per tile), several tiles per pair
]


@pytest.mark.parametrize("case", PAIR_CASES)
def test_conv_tc_cta_pair_vs_simt(case):
    """CTA pairs (tcgen05 cta_group::2) of the classic-mode 256-column convolution tiles: two CTAs of a 2-wide cluster share one
    256 x 256 tile, each stages its own 128 rows of activations and HALF of the weight columns, the leader issues the MMAs for both and
    commits to the barriers of both, both run the epilogue on their own TMEM rows.  By default only launches of more than one wave take
    this path; the test forces it (wsr_debug_set_pair(2)) and checks that it really ran (bit 20 of wsr_debug_last_tc_config)."""
    prev = nat.call("wsr_debug_set_pair", 2)
    try:
        _split_k_case(*case, expect=False, expect_pair=True)
    finally:
        nat.call("wsr_debug_set_pair", prev)


def _split_k_case(N, Cin, Cout, H, W, k, stride, up, Cin2, expect, expect_pair=None):
    # up == "dgrad": the tap-table data gradient of nearest-x2 + 3x3 with input (H, W) -- a 4x4 convolution reading dY at (2H, 2W)
    dgrad, up = up == "dgrad", up is True
    torch.manual_seed(12)
    dev = _dev()
    eng = Engine(dev, "bf16")
    x = torch.randn(N, Cin, 2 * H, 2 * W, device=dev) if dgrad else torch.randn(N, Cin, H, W, device=dev)
    if dgrad:
        w = T.upsample_dgrad_weight(torch.randn(Cin, Cout, 3, 3, device=dev) / math.sqrt(Cout * 9))
    else:
        w = torch.randn(Cout, Cin, k, k, device=dev) / math.sqrt(Cin * k * k)
    b = torch.randn(Cout, device=dev)
    rv = torch.randn(N, Cout, device=dev)
    OH, OW = (H * (2 if up else 1)) // stride, (W * (2 if up else 1)) // stride
    res = torch.randn(N, Cout, OH, OW, device=dev)
    pc = eng.pack_upsample_conv(w, b) if up else eng.pack_conv(w, b)
    pc_ref = eng.pack_conv(w, b)
    xa, ra = _nhwc(x, eng), _nhwc(res, eng)
    kw = dict(stride=stride, upsample=up, rowvec=rv.data_ptr(), rowvec_ld=Cout, res=ra)
    if dgrad:
        kw["taps"] = T.dgrad_upsample_taps(H, W)
    kw_ref = dict(kw)
    if Cin2:
        x2 = torch.randn(N, Cin2, H, W, device=dev)
        w2 = torch.randn(Cout, Cin2, 1, 1, device=dev) / math.sqrt(Cin2)
        kw.update(x2=_nhwc(x2, eng), w2=eng.pack_conv(w2, None))
        kw_ref.update(x2=kw["x2"], w2=kw["w2"])
    arena = engine_mod.StatsArena()
    y_tc = eng.new_act(N, OH, OW, Cout, zero=True, stats=arena)
    arena.finalize(dev)
    y_si = eng.new_act(N, OH, OW, Cout, dt=nat.F32, zero=True)
    eng.conv(xa, pc_ref, y_si, force_simt=True, **kw_ref)
    ref = y_si.to_nchw(eng)
    for rep in range(2):
        arena.tensor.zero_()
        y_tc.buf.zero_()
        eng.conv(xa, pc, y_tc, **kw)
        cfg = nat.call("wsr_debug_last_tc_config")
        assert ((cfg & 0xff) > 1) == expect, (cfg >> 8, cfg & 0xff)
        if expect_pair is not None:
            assert bool(cfg >> 20) == expect_pair, ((cfg >> 8) & 0xfff, cfg >> 20)
        got = y_tc.to_nchw(eng)
        err = rel_l2(got, ref)
        assert err < (8e-3 if up else 4e-3), (rep, err)          # merged upsample taps are summed before the bf16 rounding
        # GroupNorm statistics of the output came out of the (distributed) epilogue
        st = arena.tensor.view(N, Cout, 2)
        assert rel_l2(st[..., 0].float(), got.double().sum((2, 3)).float()) < 2e-3
        assert rel_l2(st[..., 1].float(), (got.double() ** 2).sum((2, 3)).float()) < 2e-3


@pytest.mark.parametrize("hw", [(16, 32), (4, 128)])
def test_conv_tc_second_segment_slices_and_f32_out(hw):
    """fused 1x1 res_conv segment, channel-slice input/output pitches, fp32 output, Cout=1 with padded weight rows
    (classic and halo tiles)."""
    torch.manual_seed(3)
    dev = _dev()
    eng = Engine(dev, "bf16")
    N, Cin, Cout = 2, 128, 128
    H, W = hw
    x = torch.randn(N, Cin, H, W, device=dev)
    x2 = torch.randn(N, 192, H, W, device=dev)
    w = torch.randn(Cout, Cin, 3, 3, device=dev) / math.sqrt(Cin * 9)
    w2 = torch.randn(Cout, 192, 1, 1, device=dev) / math.sqrt(192)
    b = torch.randn(Cout, device=dev)
    xa = _nhwc(x, eng, ld=Cin + 64, coff=64)
    x2a = _nhwc(x2, eng)
    y_tc = eng.new_act(N, H, W, Cout + 64, zero=True).slice(64, Cout)
    y_si = eng.new_act(N, H, W, Cout, dt=nat.F32)
    pc, pc2 = eng.pack_conv(w, b), eng.pack_conv(w2, None)
    eng.conv(xa, pc, y_tc, x2=x2a, w2=pc2)
    eng.conv(xa, pc, y_si, x2=x2a, w2=pc2, force_simt=True)
    assert eng.n_tc == 1
    assert rel_l2(y_tc.to_nchw(eng), y_si.to_nchw(eng)) < 4e-3
    # Cout = 1, fp32 output (the UNet head)
    wf = torch.randn(1, Cin, 3, 3, device=dev) / math.sqrt(Cin * 9)
    bfin = torch.randn(1, device=dev)
    pcf = eng.pack_conv(wf, bfin, rows=64)
    o_tc = eng.new_act(N, H, W, 1, dt=nat.F32)
    o_si = eng.new_act(N, H, W, 1, dt=nat.F32)
    eng.conv(xa, pcf, o_tc)
    eng.conv(xa, pcf, o_si, force_simt=True)
    assert eng.n_tc == 2
    assert rel_l2(o_tc.to_nchw(eng), o_si.to_nchw(eng)) < 1e-4


@pytest.mark.parametrize("shape", [(2, 512, 512, 64), (3, 128, 128, 512), (1, 256, 64, 128), (2, 100, 72, 64)])
def test_gemm_tc_vs_simt(shape):
    batch, M, N, K = shape
    torch.manual_seed(4)
    dev = _dev()
    eng = Engine(dev, "bf16")
    a = (torch.randn(batch, M, K, device=dev) / math.sqrt(K)).bfloat16()
    b = torch.randn(batch, N, K, device=dev).bfloat16()
    d_tc = torch.zeros(batch, M, N, device=dev, dtype=torch.float32)
    d_si = torch.zeros(batch, M, N, device=dev, dtype=torch.float32)
    for d, force in ((d_tc, False), (d_si, True)):
        eng.gemm(a.data_ptr(), nat.BF16, (M * K, K, 1), b.data_ptr(), nat.BF16, (N * K, K, 1), d.data_ptr(), nat.F32,
                 (M * N, N, 1), batch, M, N, K, alpha=0.5, force_simt=force)
    assert eng.n_tc == 1 and eng.n_simt == 1
    ref = 0.5 * torch.einsum("bmk,bnk->bmn", a.float(), b.float())
    assert rel_l2(d_si, ref) < 2e-5
    assert rel_l2(d_tc, ref) < 2e-5


def test_gemm_tc_shared_a_transposed_out():
    """V^T = Wv * n^T: A shared across the batch (a_sb = 0), output (B, C, pixels)."""
    torch.manual_seed(5)
    dev = _dev()
    eng = Engine(dev, "bf16")
    B, Cc, n = 2, 128, 512
    wv = (torch.randn(Cc, Cc, device=dev) / math.sqrt(Cc)).bfloat16()
    act = torch.randn(B, n, Cc, device=dev).bfloat16()
    vT = torch.zeros(B, Cc, n, device=dev, dtype=torch.bfloat16)
    eng.gemm(wv.data_ptr(), nat.BF16, (0, Cc, 1), act.data_ptr(), nat.BF16, (n * Cc, Cc, 1), vT.data_ptr(), nat.BF16,
             (Cc * n, n, 1), B, Cc, n, Cc)
    assert eng.n_tc == 1
    ref = torch.einsum("ck,bpk->bcp", wv.float(), act.float())
    assert rel_l2(vT.float(), ref) < 4e-3


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("shape", [(2, 64, 16, 32), (2, 768, 4, 8), (1, 192, 8, 16)])
def test_group_norm(mode, shape):
    N, Cc, H, W = shape
    torch.manual_seed(6)
    dev = _dev()
    eng = Engine(dev, mode)
    x = torch.randn(N, Cc, H, W, device=dev) * 2 + 0.5
    g, b = torch.randn(Cc, device=dev), torch.randn(Cc, device=dev)
    xa = _nhwc(x, eng)
    xr = xa.to_nchw(eng)
    ref = F.group_norm(xr, 32, g, b, eps=1e-5)
    ref = ref * torch.sigmoid(ref)
    stats = torch.zeros(N * Cc * 2, device=dev, dtype=torch.float64)
    eng.gn_stats(xa, stats)
    y = eng.gn_apply(xa, g, b, 32, nat.ACT_SWISH, eng.new_act(N, H, W, Cc), stats=stats)
    assert rel_l2(y.to_nchw(eng), ref) < (2e-5 if mode == "fp32" else 4e-3)


def test_softmax_rows():
    torch.manual_seed(7)
    dev = _dev()
    eng = Engine(dev, "fp32")
    s = torch.randn(37, 513, device=dev) * 4
    p = torch.empty_like(s)
    eng.softmax(s, nat.F32, 37, 513, 0.3, p, nat.F32)
    assert rel_l2(p, torch.softmax(s * 0.3, -1)) < 1e-5


@pytest.mark.parametrize("cols", [128, 512, 1024])
def test_softmax_rows_warp_per_row_path(cols):
    """Row lengths that are multiples of 128 up to 1024 (the sampler's attention shapes) take the one-warp-per-row kernel: fp32 and packed
    bf16 outputs, a row count that is not a multiple of the 8 rows per block, large logits."""
    torch.manual_seed(8)
    dev = _dev()
    eng = Engine(dev, "fp32")
    s = torch.randn(37, cols, device=dev) * 6
    s[3, 5] = 80.0
    ref = torch.softmax(s * 0.25, -1)
    p = torch.empty_like(s)
    eng.softmax(s, nat.F32, 37, cols, 0.25, p, nat.F32)
    assert rel_l2(p, ref) < 1e-6 and float((p.sum(-1) - 1).abs().max()) < 1e-5
    pb = torch.empty(37, cols, device=dev, dtype=torch.bfloat16)
    eng.softmax(s, nat.F32, 37, cols, 0.25, pb, nat.BF16)
    assert rel_l2(pb.float(), ref) < 4e-3


def test_sampler_step_and_randn():
    from oracle.schedule import ddpm_tables
    from oracle.cases import LINEAR_1000
    dev = _dev()
    tabs, _ = ddpm_tables(LINEAR_1000)
    order = ("sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod", "posterior_mean_coef1", "posterior_mean_coef2",
             "posterior_log_variance_clipped")
    tab = torch.stack([torch.from_numpy(tabs[k]) for k in order]).to(dev).contiguous()
    torch.manual_seed(8)
    n = 4096 + 3
    x, eps, z = torch.randn(n, device=dev), torch.randn(n, device=dev), torch.randn(n, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    for t in (999, 500, 1, 0):
        t_dev = torch.tensor([t], dtype=torch.int32, device=dev)
        out = torch.empty_like(x)
        nat.call("wsr_sampler_step", x.data_ptr(), eps.data_ptr(), nat.F32, z.data_ptr(), 0, 0, tab.data_ptr(), 1000,
                 t_dev.data_ptr(), 1, out.data_ptr(), n, st)
        x0 = (tab[0, t] * x - tab[1, t] * eps).clamp(-1, 1)
        ref = tab[2, t] * x0 + tab[3, t] * x + (z * (0.5 * tab[4, t]).exp() if t > 0 else 0)
        assert rel_l2(out, ref) < 1e-6
    r = torch.empty(1 << 20, device=dev)
    nat.call("wsr_randn", r.data_ptr(), r.numel(), 1234, 7, st)
    assert abs(float(r.mean())) < 5e-3 and abs(float(r.std()) - 1) < 5e-3
    r2 = torch.empty_like(r)
    nat.call("wsr_randn", r2.data_ptr(), r2.numel(), 1234, 8, st)
    assert abs(float((r * r2).mean())) < 5e-3


@pytest.mark.parametrize("case", [(2, 64, 1, 12, 160), (1, 128, 3, 8, 256), (3, 64, 1, 7, 128), (1, 64, 4, 5, 40)])
def test_final_conv_sampler_step_fused_vs_torch(case):
    """wsr_final_conv_sampler_step: GroupNorm + Swish + conv3x3 to <= 4 channels (final_conv, resdiff/unet.py:119,177) fused with the
    reverse-step update, against fp32 torch (GroupNorm -> x*sigmoid(x) -> conv2d -> the update formula) and against the stand-alone
    wsr_sampler_step fed with the fused kernel's own eps_hat (injected noise AND the in-kernel Philox stream must match exactly).
    Sizes exercise partial tiles (H % 4 != 0, W % 128 != 0)."""
    from oracle.schedule import ddpm_tables
    from oracle.cases import LINEAR_1000
    B, Cin, Cout, H, W = case
    dev = _dev()
    torch.manual_seed(21)
    eng = Engine(dev, "bf16")
    tabs, _ = ddpm_tables(LINEAR_1000)
    order = ("sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod", "posterior_mean_coef1", "posterior_mean_coef2",
             "posterior_log_variance_clipped")
    tab = torch.stack([torch.from_numpy(tabs[k]) for k in order]).to(dev).contiguous()
    x = torch.randn(B, Cin, H, W, device=dev) * 1.7 + 0.3
    xa = _nhwc(x, eng)
    xq = xa.to_nchw(eng)                                    # the bf16-rounded tensor the kernel reads
    gamma, beta = 1 + 0.2 * torch.randn(Cin, device=dev), 0.1 * torch.randn(Cin, device=dev)
    w, bias = torch.randn(Cout, Cin, 3, 3, device=dev) / math.sqrt(9 * Cin), 0.1 * torch.randn(Cout, device=dev)
    wp = torch.empty(9, Cout, Cin, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    nat.call("wsr_pack_conv_weight", w.contiguous().data_ptr(), Cout, Cin, 3, 3, wp.data_ptr(), nat.F32, Cout, Cin, st)
    wp32 = wp
    wp = torch.empty((Cin // 64) * 9 * 4 * 2 * 64, device=dev, dtype=torch.bfloat16)
    nat.call("wsr_pack_head_weight", wp32.data_ptr(), Cout, Cin, wp.data_ptr(), st)
    stats = torch.zeros(B, 2 * Cin, device=dev, dtype=torch.float64)
    nat.call("wsr_gn_stats", xa.ptr, xa.dt, B, H * W, Cin, xa.ld, stats.data_ptr(), 2 * Cin, st)
    ref_eps = F.conv2d(F.silu(F.group_norm(xq, 32, gamma, beta, 1e-5)), w, bias, padding=1)
    state0 = torch.randn(B, Cout, H, W, device=dev)
    z = torch.randn(B, Cout, H, W, device=dev)
    for t in (999, 1, 0):
        t_dev = torch.tensor([t], dtype=torch.int32, device=dev)
        for use_z in (True, False):
            eps = torch.zeros(B, Cout, H, W, device=dev)
            state = state0.clone()
            nat.call("wsr_final_conv_sampler_step", xa.ptr, xa.ld, B, H, W, Cin, stats.data_ptr(), 2 * Cin, gamma.data_ptr(), beta.data_ptr(),
                     32, 1e-5, wp.data_ptr(), bias.data_ptr(), Cout, eps.data_ptr(), state.data_ptr(), z.data_ptr() if use_z else 0, 0,
                     4242, tab.data_ptr(), 1000, t_dev.data_ptr(), 1, st)
            e_eps = rel_l2(eps, ref_eps)
            assert e_eps < 6e-3, e_eps                       # bf16 rounding of the normalised activation, fp32 weights and sums
            # the update itself: exact against the stand-alone kernel on the same eps_hat (same injected noise / same Philox words)
            out2 = torch.empty_like(state0)
            nat.call("wsr_sampler_step", state0.data_ptr(), eps.data_ptr(), nat.F32, z.data_ptr() if use_z else 0, 0, 4242, tab.data_ptr(),
                     1000, t_dev.data_ptr(), 1, out2.data_ptr(), state0.numel(), st)
            assert torch.equal(state, out2) or rel_l2(state, out2) < 1e-6
            if use_z:
                x0 = (tab[0, t] * state0 - tab[1, t] * ref_eps).clamp(-1, 1)
                ref = tab[2, t] * x0 + tab[3, t] * state0 + (z * (0.5 * tab[4, t]).exp() if t > 0 else 0)
                assert rel_l2(state, ref) < 6e-3
    # convolution-only mode (no state)
    eps = torch.zeros(B, Cout, H, W, device=dev)
    nat.call("wsr_final_conv_sampler_step", xa.ptr, xa.ld, B, H, W, Cin, stats.data_ptr(), 2 * Cin, gamma.data_ptr(), beta.data_ptr(), 32, 1e-5,
             wp.data_ptr(), 0, Cout, eps.data_ptr(), 0, 0, 0, 0, 0, 0, 0, 0, st)
    assert rel_l2(eps, ref_eps - bias.view(1, -1, 1, 1)) < 6e-3


def test_noise_embed_and_fd_and_haar_vs_oracle():
    """level embedding, FD splitter precompute (4-D FFT over B,C,H,W) and Haar queries against the CPU oracle."""
    from oracle import nets
    from oracle.weights import seeded_randn
    dev = _dev()
    U = wsr.sub("models.diffusion_models.resdiff.unet").UNet
    from oracle.cases import unet_cfg
    from oracle.weights import fill_module
    for c_img, B in ((1, 3), (3, 2)):
        cfg = unet_cfg(32, 64, attn_res=(4,), c_img=c_img)
        net = fill_module(U(in_channel=cfg["in_channel"], out_channel=c_img, norm_groups=32, inner_channel=64,
                            channel_mults=cfg["channel_mults"], attn_res=cfg["attn_res"], res_blocks=2, dropout=0,
                            image_height=32, image_width=64, image_channels=c_img, precision="fp32"), 5).to(dev)
        sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
        cond = seeded_randn("c", (B, c_img, 32, 64), 1)
        x_t = seeded_randn("x", (B, c_img, 32, 64), 2)
        level = torch.linspace(0.2, 0.9, B).view(B, 1)
        pl = net.plan(B, dev)
        pl.set_condition(cond.to(dev))
        pl.set_levels(level.view(B).to(dev))
        t_ref = nets.noise_level_mlp(sd, level, 64)
        assert rel_l2(pl.cur_temb.cpu(), t_ref.view(B, 64)) < 1e-5
        ref = nets.fd_info_spliter(sd, "fd_spliter.", torch.cat([cond, x_t], 1), t_ref, c_img, 32, 64)
        # channels: [x, cnn_x, denoise_x, lf, hf]
        assert rel_l2(pl.lf.cpu(), ref[:, 3 * c_img:4 * c_img]) < 2e-5
        assert rel_l2(pl.hf.cpu(), ref[:, 4 * c_img:5 * c_img]) < 2e-5
        qs = nets.haar_detail_sums(cond, 4)
        off = 0
        for q in qs:
            got = pl.haar_out[off:off + q.numel()].view(q.shape).cpu()
            assert rel_l2(got, q) < 1e-6
            off += q.numel()


@pytest.mark.parametrize("shape", [(2, 16, 32, 64), (1, 32, 64, 128), (3, 8, 16, 64), (1, 64, 128, 64)])
def test_attention_tc_fused_vs_torch(shape):
    """fused tcgen05 attention (scores stay on chip) against fp32 torch on the same bf16 operands."""
    B, H, W, d = shape
    n = H * W
    torch.manual_seed(9)
    dev = _dev()
    eng = Engine(dev, "bf16")
    q = torch.randn(B, d, H, W, device=dev) * 1.5
    k = torch.randn(B, d, H, W, device=dev) * 1.5
    v = torch.randn(B, d, H, W, device=dev)
    qa, ka = _nhwc(q, eng), _nhwc(k, eng, ld=2 * d, coff=d)
    vT = v.reshape(B, d, n).bfloat16().contiguous()
    o = eng.new_act(B, H, W, d, zero=True)
    scores = torch.empty(B * n * n, device=dev, dtype=torch.float32)
    probs = torch.empty(B * n * n, device=dev, dtype=torch.bfloat16)
    eng.attention(qa, ka, vT, o, scores, probs)
    assert eng.n_tc == 1 and eng.n_simt == 0          # one fused launch
    qf = qa.to_nchw(eng).reshape(B, d, n)
    kf = ka.to_nchw(eng).reshape(B, d, n)
    s = torch.einsum("bcq,bck->bqk", qf, kf) / math.sqrt(d)
    ref = torch.einsum("bqk,bck->bcq", torch.softmax(s, -1), vT.float()).reshape(B, d, H, W)
    err = rel_l2(o.to_nchw(eng), ref)
    assert err < 1e-2, err
    # and the unfused path (GEMM -> softmax -> GEMM) agrees as well
    eng.no_fused_attention = True
    o2 = eng.new_act(B, H, W, d, zero=True)
    eng.attention(qa, ka, vT, o2, scores, probs)
    assert rel_l2(o2.to_nchw(eng), ref) < 1e-2


@pytest.mark.parametrize("shape", [(2, 16, 32, 512), (2, 16, 32, 256), (3, 8, 16, 512), (1, 12, 32, 192), (5, 16, 16, 320)])
def test_attention_small_tc_fused_vs_torch(shape):
    """fused low-resolution attention (N <= 512 keys, head dimension up to 512: nn_modules/resnet.py:81-100 at 16x32 / 8x16,
    guided_cross_attention.py levels 2-3): ONE launch, whole score block in tensor memory, against fp32 torch on the same bf16
    operands; the operands are channel slices of wider buffers as in the UNet plan (q | k in one 2C-channel tensor)."""
    B, H, W, d = shape
    n = H * W
    torch.manual_seed(10)
    dev = _dev()
    eng = Engine(dev, "bf16")
    # scores with a realistic spread: |s| / sqrt(d) of a few units, so the softmax is far from uniform
    q = torch.randn(B, d, H, W, device=dev) * 2.0
    k = torch.randn(B, d, H, W, device=dev) * 2.0
    v = torch.randn(B, d, H, W, device=dev)
    qk = eng.new_act(B, H, W, 2 * d, zero=True)
    qa, ka = qk.slice(0, d), qk.slice(d, d)
    eng.nchw_to_act(q, qa)
    eng.nchw_to_act(k, ka)
    vT = v.reshape(B, d, n).bfloat16().contiguous()
    o = eng.new_act(B, H, W, d, zero=True)
    scores = torch.empty(B * n * n, device=dev, dtype=torch.float32)
    probs = torch.empty(B * n * n, device=dev, dtype=torch.bfloat16)
    assert nat.call("wsr_attention_small_tc_supported", n, n, d) == 1
    eng.attention(qa, ka, vT, o, scores, probs)
    assert eng.n_tc == 1 and eng.n_simt == 0          # one fused launch
    qf = qa.to_nchw(eng).reshape(B, d, n)
    kf = ka.to_nchw(eng).reshape(B, d, n)
    s = torch.einsum("bcq,bck->bqk", qf, kf) / math.sqrt(d)
    ref = torch.einsum("bqk,bck->bcq", torch.softmax(s, -1), vT.float()).reshape(B, d, H, W)
    got = o.to_nchw(eng)
    err = rel_l2(got, ref)
    assert torch.isfinite(got).all()
    assert err < 1e-2, err
    # per image as well (a wrong batch coordinate would hide in the average)
    for b in range(B):
        assert rel_l2(got[b], ref[b]) < 1.5e-2
    # and the unfused path (GEMM -> softmax -> GEMM) agrees
    eng.no_fused_attention = True
    o2 = eng.new_act(B, H, W, d, zero=True)
    eng.attention(qa, ka, vT, o2, scores, probs)
    assert rel_l2(o2.to_nchw(eng), ref) < 1e-2


def test_attention_small_tc_shape_gate():
    ok = lambda nq, nk, d: nat.call("wsr_attention_small_tc_supported", nq, nk, d)
    assert ok(512, 512, 512) and ok(128, 128, 512) and ok(512, 512, 256) and ok(256, 64, 64)
    assert not ok(32, 32, 64) and not ok(512, 1024, 64) and not ok(512, 512, 1024) and not ok(128, 96, 64) and not ok(128, 128, 96)


@pytest.mark.parametrize("case", [(2, 64, 64, 16, 32, 3, 1, False), (2, 64, 128, 16, 32, 3, 2, False), (1, 64, 64, 8, 16, 3, 1, True),
                                  (3, 128, 64, 2, 4, 1, 1, False), (2, 64, 64, 6, 256, 3, 1, False), (2, 64, 128, 4, 128, 3, 1, True)])
def test_conv_tc_fused_gn_stats(case):
    """GroupNorm statistics produced by the conv epilogue == statistics of the stored output (into a concat slot)."""
    N, Cin, Cout, H, W, k, stride, up = case
    torch.manual_seed(10)
    dev = _dev()
    eng = Engine(dev, "bf16")
    arena = engine_mod.StatsArena()
    OH, OW = (H * (2 if up else 1)) // stride, (W * (2 if up else 1)) // stride
    cat = eng.new_act(N, OH, OW, Cout + 64, zero=True, stats=arena)
    arena.finalize(dev)
    y = cat.slice(64, Cout)
    x = torch.randn(N, Cin, H, W, device=dev)
    w = torch.randn(Cout, Cin, k, k, device=dev) / math.sqrt(Cin * k * k)
    b = torch.randn(Cout, device=dev)
    eng.conv(_nhwc(x, eng), eng.pack_conv(w, b), y, stride=stride, upsample=up)
    assert eng.n_tc == 1
    got = arena.tensor.view(N, Cout + 64, 2)[:, 64:, :]
    yv = y.to_nchw(eng).double()
    ref = torch.stack([yv.sum(dim=(2, 3)), (yv * yv).sum(dim=(2, 3))], dim=-1)
    assert rel_l2(got, ref) < 1e-3      # statistics are taken from the fp32 accumulators, before the bf16 store rounding
    assert float(arena.tensor.view(N, Cout + 64, 2)[:, :64, :].abs().max()) == 0.0


@pytest.mark.parametrize("case", [(2, 64, 64, 8, 16), (1, 128, 128, 4, 128), (1, 64, 128, 16, 32)])
def test_upsample_conv_merged_taps(case):
    """phase-merged 2x2 taps (2.25x fewer MACs) == nearest-x2 upsample + conv3x3, on the tcgen05 and the SIMT kernel."""
    N, Cin, Cout, H, W = case
    torch.manual_seed(11)
    dev = _dev()
    eng = Engine(dev, "bf16")
    x = torch.randn(N, Cin, H, W, device=dev)
    w = torch.randn(Cout, Cin, 3, 3, device=dev) / math.sqrt(Cin * 9)
    b = torch.randn(Cout, device=dev)
    xa = _nhwc(x, eng)
    ref = _ref_conv(xa.to_nchw(eng), w, b, 1, True)
    pm = eng.pack_upsample_conv(w, b)
    assert pm.merged_up
    y_tc = eng.new_act(N, 2 * H, 2 * W, Cout)
    y_si = eng.new_act(N, 2 * H, 2 * W, Cout, dt=nat.F32)
    eng.conv(xa, pm, y_tc, upsample=True)
    eng.conv(xa, pm, y_si, upsample=True, force_simt=True)
    assert eng.n_tc == 1 and eng.n_simt == 1
    assert rel_l2(y_si.to_nchw(eng), ref) < 5e-3          # weights pre-summed in fp32, then rounded to bf16
    assert rel_l2(y_tc.to_nchw(eng), y_si.to_nchw(eng)) < 4e-3


FUSE_GN_CASES = [
    # N, Cin, Cout, H, W, Cin2 (fused 1x1 segment; 0 = none)
    (2, 64, 64, 8, 256, 0),          # N = 64 tile, four output rows per tile
    (1, 192, 64, 6, 128, 192),       # two rows per tile fallback (6 % 4 != 0), res_conv segment
    (2, 128, 128, 4, 128, 0),        # N = 128 tile, two rows per tile
    (1, 384, 128, 4, 128, 384),
    (1, 128, 256, 3, 256, 0),        # N = 256 tile, one row per tile, odd row count
    (2, 64, 1, 4, 256, 0),           # final conv: one output channel
]


@pytest.mark.parametrize("out_bf16", [False, True])
@pytest.mark.parametrize("case", FUSE_GN_CASES + [(2, 64, 64, 7, 256, 0), (1, 128, 64, 5, 128, 128), (3, 192, 128, 6, 256, 0)])
def test_conv_tc_fused_groupnorm_input(case, out_bf16):
    """GroupNorm + Swish applied inside the tcgen05 convolution (transform warps rewrite the operand tile in shared memory)
    against the two-kernel path (wsr_gn_apply, then wsr_conv_tc) on the same raw tensor."""
    N, Cin, Cout, H, W, Cin2 = case
    torch.manual_seed(11)
    dev = _dev()
    eng = Engine(dev, "bf16")
    x = torch.randn(N, Cin, H, W, device=dev) * 1.3 + 0.2
    w = torch.randn(Cout, Cin, 3, 3, device=dev) / math.sqrt(Cin * 9)
    b = torch.randn(Cout, device=dev)
    gamma, beta = 1 + 0.1 * torch.randn(Cin, device=dev), 0.1 * torch.randn(Cin, device=dev)
    arena = engine_mod.StatsArena()
    xa = eng.new_act(N, H, W, Cin, stats=arena)
    arena.finalize(dev)
    eng.nchw_to_act(x, xa)
    eng.gn_stats(xa)
    pc = eng.pack_conv(w, b, rows=64 if Cout < 16 else None)
    kw = {}
    if Cin2:
        x2 = torch.randn(N, Cin2, H, W, device=dev)
        w2 = torch.randn(Cout, Cin2, 1, 1, device=dev) / math.sqrt(Cin2)
        kw = dict(x2=_nhwc(x2, eng), w2=eng.pack_conv(w2, None))
    assert eng.conv_can_fuse_gn(xa, pc, x2=kw.get("x2"))
    a = eng.new_act(N, H, W, Cin)
    eng.gn_apply(xa, gamma, beta, 32, nat.ACT_SWISH, a)
    # out_bf16: bf16 output with fused output statistics and a residual = the staged-epilogue kernels the UNet plan launches
    # (vertical tap merge for Cout <= 64, two-row tiles for 128); fp32 output = the plain epilogue
    odt = nat.BF16 if out_bf16 else nat.F32
    if out_bf16 and Cout < 16:
        pytest.skip("the one-channel head writes fp32")
    res = _nhwc(torch.randn(N, Cout, H, W, device=dev), eng) if out_bf16 else None
    arena2 = engine_mod.StatsArena()
    y_ref = eng.new_act(N, H, W, Cout, dt=odt, zero=True)
    y = eng.new_act(N, H, W, Cout, dt=odt, zero=True, stats=arena2 if out_bf16 else None)
    arena2.finalize(dev)
    eng.conv(a, pc, y_ref, res=res, **kw)
    tab = eng.empty((N, Cin, 2), torch.float32)
    eng.gn_finalize(xa, gamma, beta, 32, tab)
    for rep in range(2):
        eng.conv(xa, pc, y, gn=(tab, nat.ACT_SWISH), res=res, **kw)
    torch.cuda.synchronize()
    got, ref = y.to_nchw(eng), y_ref.to_nchw(eng)
    err = rel_l2(got, ref)
    # the fused transform works in packed bf16x2 arithmetic (scale / shift and the pre-activation are rounded to bf16; see gemm_tc.cu):
    # about one extra bf16 rounding per activation relative to the two-kernel path
    assert err < (8e-3 if out_bf16 else 5e-3), err
    if out_bf16:
        st = arena2.tensor.view(N, Cout, 2) / 2              # two launches accumulated into the same slot
        assert rel_l2(st[..., 0].float(), got.double().sum((2, 3)).float()) < 3e-3


@pytest.mark.parametrize("case", [(2, 64, 64, 7, 256, 0), (1, 192, 64, 6, 128, 128), (2, 128, 64, 3, 128, 64), (1, 64, 1, 5, 256, 0)])
def test_conv_tc_vertical_tap_merge_vs_simt(case):
    """N = 64 layers on rows of >= 128 pixels run the vertically merged schedule (one MMA per halo row feeds three output
    rows; register-accumulated GroupNorm statistics): against the SIMT kernel on the same bf16 inputs, incl. the fused 1x1
    segment, partial last tiles (H % 3 != 0) and the statistics."""
    N, Cin, Cout, H, W, Cin2 = case
    torch.manual_seed(12)
    dev = _dev()
    eng = Engine(dev, "bf16")
    x = torch.randn(N, Cin, H, W, device=dev)
    w = torch.randn(Cout, Cin, 3, 3, device=dev) / math.sqrt(Cin * 9)
    b = torch.randn(Cout, device=dev)
    pc = eng.pack_conv(w, b, rows=64 if Cout < 16 else None)
    assert pc.w_vm is not None
    kw = {}
    if Cin2:
        x2 = torch.randn(N, Cin2, H, W, device=dev)
        w2 = torch.randn(Cout, Cin2, 1, 1, device=dev) / math.sqrt(Cin2)
        kw = dict(x2=_nhwc(x2, eng), w2=eng.pack_conv(w2, None))
    res = torch.randn(N, Cout, H, W, device=dev)
    xa, ra = _nhwc(x, eng), _nhwc(res, eng)
    arena = engine_mod.StatsArena()
    y_tc = eng.new_act(N, H, W, Cout, dt=nat.F32, stats=arena)
    y_si = eng.new_act(N, H, W, Cout, dt=nat.F32, stats=arena)
    st = arena.finalize(dev)
    eng.conv(xa, pc, y_tc, res=ra, **kw)
    eng.conv(xa, pc, y_si, res=ra, force_simt=True, **kw)
    assert eng.n_tc == 1 and eng.n_simt == 1
    torch.cuda.synchronize()
    assert rel_l2(y_tc.to_nchw(eng), y_si.to_nchw(eng)) < 2e-5
    half = st.numel() // 2
    assert rel_l2(st[:half], st[half:]) < 1e-5


def test_attention_tc_sampled_shift_is_exact_when_the_maximum_is_not_sampled():
    """The fused attention takes its softmax shift from 4 sampled key blocks.  Softmax is shift-invariant, so rows whose
    true maximum lies in an UNSAMPLED block (probabilities > 1 before normalisation, here by up to e^25) must still match
    torch, as must rows dominated by a sampled key."""
    B, H, W, d = 1, 16, 64, 64           # 1024 keys = 8 blocks; blocks 0, 2, 4, 6 are sampled
    n = H * W
    torch.manual_seed(10)
    dev = _dev()
    eng = Engine(dev, "bf16")
    q = torch.randn(B, d, H, W, device=dev)
    k = torch.randn(B, d, H, W, device=dev) * 0.5
    v = torch.randn(B, d, H, W, device=dev)
    kf0 = k.reshape(B, d, n)
    qf0 = q.reshape(B, d, n)
    # key 200 (block 1, unsampled) is strongly aligned with queries 0..255; key 700 (block 5) with queries 256..511
    kf0[:, :, 200] = 6.0 * qf0[:, :, :256].mean(-1) / qf0[:, :, :256].mean(-1).norm() * math.sqrt(d) / 2
    kf0[:, :, 700] = 12.0 * qf0[:, :, 256:512].mean(-1) / qf0[:, :, 256:512].mean(-1).norm() * math.sqrt(d) / 2
    qa, ka = _nhwc(q, eng), _nhwc(k, eng)
    vT = v.reshape(B, d, n).bfloat16().contiguous()
    o = eng.new_act(B, H, W, d, zero=True)
    eng.attention(qa, ka, vT, o, None, None)
    assert eng.n_tc == 1
    qf = qa.to_nchw(eng).reshape(B, d, n)
    kf = ka.to_nchw(eng).reshape(B, d, n)
    s = torch.einsum("bcq,bck->bqk", qf, kf) / math.sqrt(d)
    spread = float((s.max(-1).values - s[:, :, torch.arange(n, device=dev) // 128 % 2 == 0].max(-1).values).max())
    assert spread > 5.0, spread            # the case really exercises P > 1
    ref = torch.einsum("bqk,bck->bcq", torch.softmax(s, -1), vT.float()).reshape(B, d, H, W)
    out = o.to_nchw(eng)
    assert torch.isfinite(out).all()
    assert rel_l2(out, ref) < 1e-2, rel_l2(out, ref)
