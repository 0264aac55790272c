"""GPU tests of the training step (SURVEY.md 8 a.7 / a.8: p_losses -> loss / numel -> backward -> Adam).

Kernel level: every backward kernel is called through the C ABI and compared with torch.autograd (fp32, no TF32) on
the same inputs.  End to end: the reference-facing classes (ResDiffDiffusion.p_losses -> .backward()) against the
gradients of the REAL reference (tests/golden/resdiff_grad_small.npz) and of the CPU oracle's autograd, per parameter.
Tolerances: fp32 check mode rel-L2 <= 2e-4 per tensor (atomics / summation order; measured 1.2e-6 over the whole
gradient).  bf16 mode: 2x the REAL reference's own bf16-autocast drift on this case (oracle/bf16_drift.py: whole gradient
7.6e-2, median tensor 3.2e-2, worst 0.53 on a 2-element tensor) -> per tensor <= 1.6e-1; whole gradient <= 1.5 x the value this
path measures on B200 (ResDiff 6.8e-2 -> 1.0e-1, PhyDiff 3.0e-2 -> 5e-2, SR3 8.9e-3 -> 2e-2, SRDiff 2.7e-2 -> 5e-2; round 1 used a
flat 1.5e-1, which a 2x regression would have passed)
(tensors with fewer than 16 elements: <= 1.0); measured on B200: 6.8e-2 whole gradient."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import wsr
from conftest import load_golden, rel_l2
from oracle import process
from oracle.cases import CASES, LINEAR_1000
from oracle.weights import fill_module

pytestmark = pytest.mark.gpu

torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False

nat = wsr.pkg.native
engine_mod = wsr.sub("engine")
Engine, Act = engine_mod.Engine, engine_mod.Act
T = wsr.sub("taps")


def _dev():
    return torch.device("cuda:0")


def _nhwc(x, eng, ld=None, coff=0, dt=None):
    N, C, H, W = x.shape
    full = eng.new_act(N, H, W, ld or C, dt=dt, zero=True)
    a = full.slice(coff, C)
    eng.nchw_to_act(x, a)
    return a


# ----------------------------------------------------------------------------------------------------------------
# convolution gradients
# ----------------------------------------------------------------------------------------------------------------
BWD_CASES = [
    # N, Cin, Cout, H, W, k, stride, upsample
    (2, 64, 64, 8, 16, 3, 1, False),
    (2, 64, 128, 8, 16, 1, 1, False),
    (2, 64, 64, 8, 16, 3, 2, False),
    (1, 64, 64, 4, 8, 3, 1, True),
    (2, 5, 64, 8, 16, 3, 1, False),
    (2, 64, 1, 8, 16, 3, 1, False),
    (1, 128, 64, 4, 128, 3, 1, False),
]


def _autograd_case(case, dev, seed=0):
    N, Cin, Cout, H, W, k, stride, up = case
    torch.manual_seed(seed)
    x = torch.randn(N, Cin, H, W, device=dev, requires_grad=True)
    w = (torch.randn(Cout, Cin, k, k, device=dev) / math.sqrt(Cin * k * k)).requires_grad_(True)
    b = torch.randn(Cout, device=dev, requires_grad=True)
    xin = F.interpolate(x, scale_factor=2, mode="nearest") if up else x
    y = F.conv2d(xin, w, b, stride=stride, padding=(k - 1) // 2)
    dy = torch.randn_like(y)
    y.backward(dy)
    return x.detach(), w.detach(), dy, x.grad, w.grad, b.grad


def _dgrad(eng, case, w, dy_act, dx_act, force_simt=False):
    N, Cin, Cout, H, W, k, stride, up = case
    if up:
        pc = eng.pack_conv(T.upsample_dgrad_weight(w), None)
        eng.conv(dy_act, pc, dx_act, taps=T.dgrad_upsample_taps(H, W), bias=False, res=dx_act, force_simt=force_simt)
    elif stride == 2:
        pc = eng.pack_conv(T.dgrad_weight(w), None)
        for tp in T.dgrad_down_taps(H, W):
            eng.conv(dy_act, pc, dx_act, taps=tp, bias=False, res=dx_act, force_simt=force_simt)
    else:
        pc = eng.pack_conv(T.dgrad_weight(w), None)
        eng.conv(dy_act, pc, dx_act, bias=False, res=dx_act, force_simt=force_simt)


@pytest.mark.parametrize("case", BWD_CASES)
def test_conv_backward_fp32_vs_autograd(case):
    N, Cin, Cout, H, W, k, stride, up = case
    dev = _dev()
    eng = Engine(dev, "fp32")
    x, w, dy, dx_ref, dw_ref, db_ref = _autograd_case(case, dev)
    dy_act = _nhwc(dy, eng)
    dx_act = eng.new_act(N, H, W, Cin, zero=True)
    _dgrad(eng, case, w, dy_act, dx_act)
    assert rel_l2(dx_act.to_nchw(eng), dx_ref) < 2e-5
    dw = torch.zeros_like(w)
    db = torch.zeros(Cout, device=dev)
    taps = T.forward_upsample_taps(H, W) if up else T.forward_taps(k, stride, H, W)
    eng.wgrad(_nhwc(x, eng), dy_act, taps, dw, (1, Cin * k * k, k * k), db, 2 if up else 1)
    assert rel_l2(dw, dw_ref) < 2e-5
    assert rel_l2(db, db_ref) < 2e-5


@pytest.mark.parametrize("case", [c for c in BWD_CASES if c[2] % 64 == 0])
def test_conv_dgrad_tc_vs_simt(case):
    """bf16 mode: the data gradient runs on the tcgen05 kernel (tap-table variant for stride 2 / upsample)."""
    N, Cin, Cout, H, W, k, stride, up = case
    dev = _dev()
    eng = Engine(dev, "bf16")
    assert eng.use_tc
    x, w, dy, dx_ref, _, _ = _autograd_case(case, dev, seed=1)
    dy_act = _nhwc(dy, eng)
    dx_tc = eng.new_act(N, H, W, Cin, zero=True)
    dx_si = eng.new_act(N, H, W, Cin, dt=nat.F32, zero=True)
    _dgrad(eng, case, w, dy_act, dx_tc)
    n_tc = eng.n_tc
    _dgrad(eng, case, w, dy_act, dx_si, force_simt=True)
    assert n_tc >= 1 and eng.n_tc == n_tc
    assert rel_l2(dx_tc.to_nchw(eng), dx_si.to_nchw(eng)) < 4e-3
    assert rel_l2(dx_tc.to_nchw(eng), dx_ref) < 1.5e-2


WGRAD_TC_CASES = [
    # N, Cin, Cout, H, W, k, stride, upsample, x_ld (0 = Cin)
    (2, 64, 64, 8, 16, 3, 1, False, 0),
    (1, 128, 64, 4, 128, 3, 1, False, 0),
    (2, 192, 128, 8, 16, 3, 1, False, 0),        # partial Cin tile (192 in a 256-wide tile)
    (2, 64, 320, 8, 16, 1, 1, False, 0),         # three Cout tiles, the last one half full
    (2, 64, 64, 16, 32, 3, 2, False, 0),         # Downsample: phase-subsampled X views
    (2, 64, 64, 8, 16, 3, 1, True, 0),           # Upsample: four dY phase segments per tap
    (2, 5, 64, 8, 16, 3, 1, False, 64),          # stem: 5 channels inside a 64-channel buffer
    (8, 512, 512, 2, 4, 3, 1, False, 0),         # deepest level: one 64-pixel tile spans all eight images
]


@pytest.mark.parametrize("case", WGRAD_TC_CASES)
def test_conv_wgrad_tc_vs_simt(case):
    """bf16 mode: the weight gradient on tcgen05 (MN-major operands, split-K) against the SIMT kernel on the same bf16
    inputs, and against autograd."""
    N, Cin, Cout, H, W, k, stride, up, x_ld = case
    dev = _dev()
    eng = Engine(dev, "bf16")
    assert eng.use_tc
    x, w, dy, _, dw_ref, db_ref = _autograd_case(case[:8], dev, seed=2)
    xa = _nhwc(x, eng, ld=x_ld or None)
    dya = _nhwc(dy, eng)
    taps = T.forward_upsample_taps(H, W) if up else T.forward_taps(k, stride, H, W)
    outs = []
    for force in (False, True):
        dw = torch.zeros_like(w)
        db = torch.zeros(Cout, device=dev)
        n_tc = eng.n_tc
        eng.wgrad(xa, dya, taps, dw, (1, Cin * k * k, k * k), db, 2 if up else 1, force_simt=force)
        assert (eng.n_tc == n_tc + 1) == (not force)
        outs.append((dw, db))
    assert rel_l2(outs[0][0], outs[1][0]) < 2e-5, rel_l2(outs[0][0], outs[1][0])
    assert rel_l2(outs[0][1], outs[1][1]) < 2e-5
    assert rel_l2(outs[0][0], dw_ref) < 8e-3 and rel_l2(outs[0][1], db_ref) < 8e-3


@pytest.mark.parametrize("a_mn,b_mn", [(False, True), (True, False), (True, True)])
@pytest.mark.parametrize("M,N,K,batch", [(128, 128, 64, 2), (256, 64, 128, 3), (64, 192, 256, 1), (512, 512, 64, 2),
                                     (64, 128, 8192, 2)])
def test_gemm_tc_transposed_operands(a_mn, b_mn, M, N, K, batch):
    """Attention backward needs A^T / B^T operands: the tcgen05 GEMM consumes MN-major (transposed) operands directly."""
    dev = _dev()
    eng = Engine(dev, "bf16")
    torch.manual_seed(7)
    a = torch.randn(batch, M, K, device=dev).to(torch.bfloat16)
    b = torch.randn(batch, N, K, device=dev).to(torch.bfloat16)
    ref = torch.matmul(a.float(), b.float().transpose(1, 2))
    a_st = a.transpose(1, 2).contiguous() if a_mn else a          # stored (batch, K, M): unit stride along m
    b_st = b.transpose(1, 2).contiguous() if b_mn else b
    a_s = (M * K, 1, M) if a_mn else (M * K, K, 1)
    b_s = (N * K, 1, N) if b_mn else (N * K, K, 1)
    d = torch.zeros(batch, M, N, device=dev, dtype=torch.float32)
    eng.gemm(a_st.data_ptr(), nat.BF16, a_s, b_st.data_ptr(), nat.BF16, b_s, d.data_ptr(), nat.F32, (M * N, N, 1), batch, M, N, K)
    assert eng.n_tc == 1 and eng.n_simt == 0
    assert rel_l2(d, ref) < 1e-5


# ----------------------------------------------------------------------------------------------------------------
# GroupNorm + Swish (+ dropout) backward
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C,groups,act", [(64, 32, "swish"), (96, 32, "swish"), (64, 32, "none")])
def test_gn_backward_vs_autograd(C, groups, act):
    dev = _dev()
    eng = Engine(dev, "fp32")
    torch.manual_seed(3)
    N, H, W = 2, 8, 16
    x = (torch.randn(N, C, H, W, device=dev) * 1.5 + 0.3).requires_grad_(True)
    gamma = (1 + 0.1 * torch.randn(C, device=dev)).requires_grad_(True)
    beta = (0.1 * torch.randn(C, device=dev)).requires_grad_(True)
    z = F.group_norm(x, groups, gamma, beta, eps=1e-5)
    y = z * torch.sigmoid(z) if act == "swish" else z
    da = torch.randn_like(y)
    y.backward(da)
    arena = engine_mod.StatsArena()
    xa = eng.new_act(N, H, W, C, stats=arena)
    arena.finalize(dev)
    eng.nchw_to_act(x.detach(), xa)
    eng.gn_stats(xa)
    dx = eng.new_act(N, H, W, C, zero=True)
    red = torch.zeros(N * 2 * C, device=dev, dtype=torch.float64)
    dg, db = torch.zeros(C, device=dev), torch.zeros(C, device=dev)
    colsum = torch.zeros(N, C, device=dev)
    eng.gn_bwd(xa, gamma.detach(), beta.detach(), groups, nat.ACT_SWISH if act == "swish" else nat.ACT_NONE, _nhwc(da, eng), dx,
               red.data_ptr(), dg, db, True, colsum.data_ptr(), C)
    dxn = dx.to_nchw(eng)
    assert rel_l2(dxn, x.grad) < 2e-5
    assert rel_l2(dg, gamma.grad) < 2e-5 and rel_l2(db, beta.grad) < 2e-5
    assert rel_l2(colsum, x.grad.sum(dim=(2, 3))) < 1e-4


def test_gn_dropout_forward_backward_consistent():
    """The backward regenerates the forward's Philox mask: d/dx of sum(y * g) must match a finite-difference-free check --
    y_drop = y_nodrop * m with m in {0, 1/(1-p)}, and the dx of the dropout path equals the no-dropout dx fed with da * m."""
    dev = _dev()
    eng = Engine(dev, "fp32")
    torch.manual_seed(4)
    N, C, H, W, p = 2, 64, 8, 16, 0.2
    x = torch.randn(N, C, H, W, device=dev)
    gamma, beta = 1 + 0.1 * torch.randn(C, device=dev), 0.1 * torch.randn(C, device=dev)
    arena = engine_mod.StatsArena()
    xa = eng.new_act(N, H, W, C, stats=arena)
    arena.finalize(dev)
    eng.nchw_to_act(x, xa)
    eng.gn_stats(xa)
    y0, y1 = eng.new_act(N, H, W, C), eng.new_act(N, H, W, C)
    eng.gn_apply(xa, gamma, beta, 32, nat.ACT_SWISH, y0)
    eng.gn_apply_dropout(xa, gamma, beta, 32, nat.ACT_SWISH, y1, p, 1234, 7)
    a0, a1 = y0.to_nchw(eng), y1.to_nchw(eng)
    m = torch.where(a0.abs() > 1e-6, a1 / a0, torch.full_like(a0, float("nan")))
    valid = ~torch.isnan(m)
    keep = (m[valid] - 1 / (1 - p)).abs() < 1e-4
    drop = m[valid].abs() < 1e-6
    assert bool((keep | drop).all())
    frac = float(drop.float().mean())
    assert abs(frac - p) < 0.02, frac
    mask = torch.where(a1 != 0, torch.full_like(a0, 1 / (1 - p)), torch.zeros_like(a0))
    da = torch.randn_like(x)
    outs = []
    for da_in, drop_arg in ((da, (p, 1234, 7)), (da * mask, (0.0, 0, 0))):
        dx = eng.new_act(N, H, W, C, zero=True)
        red = torch.zeros(N * 2 * C, device=dev, dtype=torch.float64)
        dg, db = torch.zeros(C, device=dev), torch.zeros(C, device=dev)
        eng.gn_bwd(xa, gamma, beta, 32, nat.ACT_SWISH, _nhwc(da_in, eng), dx, red.data_ptr(), dg, db, True, 0, 0, drop_arg)
        outs.append((dx.to_nchw(eng), dg.clone()))
    assert rel_l2(outs[0][0], outs[1][0]) < 1e-5 and rel_l2(outs[0][1], outs[1][1]) < 1e-5


# ----------------------------------------------------------------------------------------------------------------
# softmax backward, Adam
# ----------------------------------------------------------------------------------------------------------------
def test_softmax_backward_vs_autograd():
    dev = _dev()
    eng = Engine(dev, "fp32")
    torch.manual_seed(5)
    rows, cols, scale = 96, 200, 0.125
    s = torch.randn(rows, cols, device=dev, requires_grad=True)
    p = torch.softmax(s * scale, dim=-1)
    dp = torch.randn_like(p)
    p.backward(dp)
    ds = torch.empty_like(s)
    eng.softmax_bwd(p.detach().contiguous(), nat.F32, dp, nat.F32, rows, cols, scale, ds, nat.F32)
    assert rel_l2(ds, s.grad) < 1e-5


def test_fused_adam_matches_torch_adam():
    dev = _dev()
    FusedAdam = wsr.sub("autograd_glue").FusedAdam
    torch.manual_seed(6)
    p0 = [torch.randn(257, 33, device=dev), torch.randn(64, device=dev)]
    a = [torch.nn.Parameter(t.clone()) for t in p0]
    b = [torch.nn.Parameter(t.clone()) for t in p0]
    oa, ob = FusedAdam(a, lr=1e-3), torch.optim.Adam(b, lr=1e-3)
    for step in range(5):
        gs = [torch.randn_like(t) for t in p0]
        for pa, pb, g in zip(a, b, gs):
            pa.grad, pb.grad = g.clone(), g.clone()
        oa.step(); ob.step()
    for pa, pb in zip(a, b):
        assert rel_l2(pa.data, pb.data) < 1e-6
    sa, sb = oa.state_dict(), ob.state_dict()
    assert sa["state"].keys() == sb["state"].keys()
    assert rel_l2(sa["state"][0]["exp_avg_sq"], sb["state"][0]["exp_avg_sq"]) < 1e-6
    assert float(sa["state"][0]["step"]) == float(sb["state"][0]["step"]) == 5.0


# ----------------------------------------------------------------------------------------------------------------
# the whole training step against the reference
# ----------------------------------------------------------------------------------------------------------------
def _build(cfg, seed, precision, arch="resdiff"):
    U = wsr.sub("models.diffusion_models.%s.unet" % arch).UNet
    D = getattr(wsr.sub("models.diffusion_models.%s.%s_diffusion" % (arch, arch)),
                {"resdiff": "ResDiffDiffusion", "phydiff": "PhyDiffDiffusion", "sr3": "SR3Diffusion"}[arch])
    net = U(in_channel=cfg["in_channel"], out_channel=cfg["out_channel"], norm_groups=cfg["norm_groups"],
            inner_channel=cfg["inner_channel"], channel_mults=cfg["channel_mults"], attn_res=cfg["attn_res"],
            res_blocks=cfg["res_blocks"], dropout=cfg["dropout"], image_height=cfg["image_height"],
            image_width=cfg["image_width"], image_channels=cfg["image_channels"], precision=precision)
    net = fill_module(net, seed).to("cuda:0").train()
    diff = D(net, image_height=cfg["image_height"], image_width=cfg["image_width"], channels=1, conditional=True).cuda()
    diff.set_new_noise_schedule(LINEAR_1000, "cuda:0")
    diff.set_loss("cuda:0")
    return net, diff


def _train_backward(diff, g, spec):
    u = g["level"].numpy().astype(np.float64)
    ri, un = np.random.randint, np.random.uniform
    np.random.randint = lambda *a, **k: spec["t"]
    np.random.uniform = lambda *a, **k: u
    try:
        loss = diff.p_losses({"HR": g["hr"].cuda(), "SR": g["sr"].cuda()}, noise=g["noise"].cuda())
    finally:
        np.random.randint, np.random.uniform = ri, un
    l_pix = loss.sum() / int(g["hr"].numel())
    l_pix.backward()
    return float(loss)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_training_step_gradients_with_dropout_on_vs_oracle(precision):
    """The REAL training configuration has dropout 0.2 in every block2 (nn_modules/resnet.py:23).  The CUDA path draws its masks from
    Philox (seed, tag = res-block index, element); the masks are exported (wsr_dropout_mask) and the oracle -- pinned to the reference
    on the dropout-free fixtures -- applies the SAME masks where the reference applies nn.Dropout, so all 396 parameter gradients can be
    compared exactly (fp32: 2e-4 per tensor) instead of statistically."""
    from conftest import manifest
    from oracle import nets
    from oracle.weights import seeded_state_dict
    g, spec = load_golden("resdiff_grad_small"), CASES["resdiff_grad_small"]
    cfg = dict(spec["cfg"])
    cfg["dropout"] = 0.2
    net, diff = _build(cfg, spec["seed"], precision)
    assert net.training
    B = g["hr"].shape[0]
    dev = torch.device("cuda:0")
    torch.manual_seed(77)
    loss = _train_backward(diff, g, spec)
    plan = net.train_plan(B, dev)
    assert plan.drop_p == 0.2 and plan.drop_seed != 0
    masks = []
    frac = []
    for r in plan._res_records():
        m = torch.empty(B, r.h * r.w, r.cout, device=dev)
        nat.call("wsr_dropout_mask", m.data_ptr(), B, r.h * r.w, r.cout, 0.2, plan.drop_seed, r.drop_tag, torch.cuda.current_stream().cuda_stream)
        masks.append(m.view(B, r.h, r.w, r.cout).permute(0, 3, 1, 2).contiguous().cpu())
        frac.append(float((masks[-1] == 0).float().mean()))
    assert len(masks) == 27 or len(masks) == len(plan._res_records())
    assert abs(sum(frac) / len(frac) - 0.2) < 0.01
    sd = seeded_state_dict(manifest("resdiff", cfg), spec["seed"])
    nets.DROP_MASKS = iter(masks)
    try:
        ref_loss, oracle_grads = process.arch_param_grads("resdiff", sd, cfg, g["hr"], g["sr"], g["level"], g["noise"])
        assert next(nets.DROP_MASKS, None) is None                 # every mask consumed, in order
    finally:
        nets.DROP_MASKS = None
    rel_loss = abs(loss - float(ref_loss)) / float(ref_loss)
    # the masks really changed the problem: the dropout-free reference loss differs
    assert abs(float(ref_loss) - float(g["loss"])) / float(g["loss"]) > 1e-3
    named = dict(net.named_parameters())
    tol_t, tol_all = (2e-4, 1e-4) if precision == "fp32" else (1.6e-1, 1.0e-1)
    num = den = 0.0
    bad = []
    for n, p in named.items():
        got, ref = p.grad.detach().cpu().double(), oracle_grads[n].double()
        err, rn = float((got - ref).norm()), float(ref.norm())
        num += err ** 2
        den += rn ** 2
    for n, p in named.items():
        got, ref = p.grad.detach().cpu().double(), oracle_grads[n].double()
        err, rn = float((got - ref).norm()), float(ref.norm())
        tol_n = tol_t if (precision == "fp32" or ref.numel() >= 16) else 1.0
        if err / max(rn, 1e-30) > tol_n and err > tol_t * 1e-3 * math.sqrt(den):
            bad.append("%s rel %.3e" % (n, err / max(rn, 1e-30)))
    total = math.sqrt(num / den)
    print("\n[parity] training step with dropout 0.2 (exported Philox masks) %s: loss rel err %.3e, whole-gradient rel-L2 %.3e, %d / %d tensors out"
          % (precision, rel_loss, total, len(bad), len(named)))
    assert rel_loss < (1e-4 if precision == "fp32" else 2e-2)
    assert not bad, bad[:10]
    assert total < tol_all


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("arch", ["resdiff", "phydiff", "sr3"])
def test_training_step_gradients_vs_reference(arch, precision):
    from oracle.cases import grad_summary
    from conftest import manifest
    from oracle.weights import seeded_state_dict
    g, spec = load_golden(arch + "_grad_small"), CASES[arch + "_grad_small"]
    cfg = spec["cfg"]
    net, diff = _build(cfg, spec["seed"], precision, arch)
    loss = _train_backward(diff, g, spec)
    rel_loss = abs(loss - float(g["loss"])) / float(g["loss"])
    sd = seeded_state_dict(manifest(arch, cfg), spec["seed"])
    _, oracle_grads = process.arch_param_grads(arch, sd, cfg, g["hr"], g["sr"], g["level"], g["noise"])
    tol_t, tol_all = (2e-4, 1e-4) if precision == "fp32" else (1.6e-1, {"resdiff": 1.0e-1, "phydiff": 5e-2, "sr3": 2e-2}[arch])
    named = dict(net.named_parameters())
    assert sorted(named) == sorted(str(n) for n in g["names"])
    plan = net.train_plan(g["hr"].shape[0], torch.device("cuda:0"))
    name_of = {id(p): n for n, p in named.items()}
    bad, num, den = [], 0.0, 0.0
    lines = []
    for p in plan.param_order:                      # completion order of the backward pass: first failure localises a bug
        n = name_of[id(p)]
        assert p.grad is not None, n
        got, ref = p.grad.detach().cpu().double(), oracle_grads[n].double()
        err = float((got - ref).norm())
        rn = float(ref.norm())
        num += err ** 2
        den += rn ** 2
        ref_norm = float(g["norm/" + n])
        assert abs(rn - ref_norm) <= 1e-3 * ref_norm + 1e-12, n          # oracle == reference (pinned on CPU as well)
        rel = err / max(rn, 1e-30)
        lines.append("%-60s |g| %.3e  rel %.3e" % (n, rn, rel))
        # tiny tensors (e.g. squeeze-excite scalars) are judged against the global gradient scale
        tol_n = tol_t if (precision == "fp32" or ref.numel() >= 16) else 1.0
        if rel > tol_n and err > tol_t * 1e-3 * math.sqrt(den):
            bad.append(lines[-1])
    total = math.sqrt(num / den)
    print("\n[parity] training step " + arch + " %s: loss rel err %.3e, whole-gradient rel-L2 %.3e, %d / %d tensors above %.0e"
          % (precision, rel_loss, total, len(bad), len(lines), tol_t))
    if bad:
        print("\n".join(bad[:40]))
    assert rel_loss < (1e-4 if precision == "fp32" else 2e-2)
    assert not bad, "%d parameter gradients out of tolerance; first (backward order): %s" % (len(bad), bad[0])
    assert total < tol_all
    # summaries of the REAL reference's gradients
    summ = grad_summary([(n, named[n].grad) for n in named], spec["seed"])
    for n in named:
        ref_norm = float(g["norm/" + n])
        tol = 1e-3 if precision == "fp32" else (1.6e-1 if named[n].numel() >= 16 else 1.0)
        if ref_norm > 1e-6 * math.sqrt(den):
            assert abs(float(summ["norm/" + n]) - ref_norm) <= tol * ref_norm, n


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_training_step_at_benchmark_shape_vs_reference(precision):
    """BASELINE configs[2] ITSELF -- ResDiff Cfg-A at 128x256, batch 4, HF_guided_CA over 8192 keys at level 0 -- one p_losses +
    backward against the REAL reference's gradients (tests/golden/resdiff_grad_full_b4.npz, made by oracle/make_golden.py from the
    reference's own modules on CPU): per parameter tensor the L2 norm, the dot product with a seeded normal probe (a random projection
    of the error) and, for tensors below 4096 elements (every bias / GroupNorm / squeeze-excite parameter), the whole gradient.  The
    tile choices of the backward kernels (row-tile shapes, split of the weight-gradient K loop, images per tile) depend on the batch and
    the resolution, so the 32x64 fixtures do not cover what bench.py --workload train launches.  Tolerances: fp32 check mode 2e-4 per
    tensor, bf16 1.6e-1 per tensor and 1e-1 on the projected whole-gradient error."""
    from oracle.cases import grad_inputs, grad_summary
    g, spec = grad_inputs("resdiff_grad_full_b4", load_golden("resdiff_grad_full_b4")), CASES["resdiff_grad_full_b4"]
    cfg = spec["cfg"]
    net, diff = _build(cfg, spec["seed"], precision, "resdiff")
    loss = _train_backward(diff, g, spec)
    rel_loss = abs(loss - float(g["loss"])) / float(g["loss"])
    named = dict(net.named_parameters())
    assert sorted(named) == sorted(str(n) for n in g["names"])
    summ = grad_summary([(n, named[n].grad) for n in named], spec["seed"])
    tol_t, tol_all = (2e-4, 2e-5) if precision == "fp32" else (1.6e-1, 4.0e-2)      # measured on B200: 1.5e-6 / 1.06e-2
    gscale = math.sqrt(sum(float(g["norm/" + n]) ** 2 for n in named))
    bad, num = [], 0.0
    for n in named:
        ref_norm, got_norm = float(g["norm/" + n]), float(summ["norm/" + n])
        # the probe is standard normal, so (dot_got - dot_ref) is a one-dimensional random projection of the error vector: its
        # magnitude estimates |error|
        proj = abs(float(summ["dot/" + n]) - float(g["dot/" + n]))
        num += proj ** 2
        floor = tol_t * 1e-3 * gscale                       # tensors far below the global gradient scale are judged against it
        small = named[n].numel() < 16 and precision != "fp32"
        if abs(got_norm - ref_norm) > (1.0 if small else tol_t) * ref_norm + floor:
            bad.append("%s: |g| %.4e vs %.4e" % (n, got_norm, ref_norm))
        elif proj > 4.0 * (1.0 if small else tol_t) * ref_norm + 4.0 * floor:
            bad.append("%s: probe projection of the error %.3e vs |g| %.3e" % (n, proj, ref_norm))
        if ("full/" + n) in g:
            ref_full = torch.as_tensor(g["full/" + n]).double().flatten()
            err = float((named[n].grad.detach().cpu().double().flatten() - ref_full).norm())
            if err > (1.0 if small else tol_t) * ref_norm + floor:
                bad.append("%s: full-tensor error %.3e vs |g| %.3e" % (n, err, ref_norm))
    total = math.sqrt(num) / gscale
    print("\n[parity] training step at the configs[2] shape (B=4, 128x256) %s: loss rel err %.3e, projected whole-gradient rel error %.3e, "
          "%d / %d tensors out" % (precision, rel_loss, total, len(bad), len(named)))
    assert rel_loss < (1e-4 if precision == "fp32" else 2e-2)
    assert not bad, bad[:10]
    assert total < tol_all


def test_optimize_parameters_decreases_loss_and_flat_adam():
    """Three optimizer steps on a fixed batch through the flat-buffer path: the loss goes down, the parameters move, and
    the one-launch flat Adam equals per-parameter torch.optim.Adam driven by the same gradients."""
    g, spec = load_golden("resdiff_grad_small"), CASES["resdiff_grad_small"]
    cfg = spec["cfg"]
    FusedAdam = wsr.sub("autograd_glue").FusedAdam
    net, diff = _build(cfg, spec["seed"], "fp32")
    plan = net.train_plan(g["hr"].shape[0], torch.device("cuda:0"))
    opt = FusedAdam(list(diff.parameters()), lr=1e-4)
    opt.attach_flat(plan)
    assert plan.parameters_are_flat()
    shadow = [torch.nn.Parameter(p.detach().clone()) for p in diff.parameters()]
    ref_opt = torch.optim.Adam(shadow, lr=1e-4)
    losses = []
    for it in range(3):
        opt.zero_grad()
        losses.append(_train_backward(diff, g, spec))
        for s, p in zip(shadow, diff.parameters()):
            s.grad = None if p.grad is None else p.grad.detach().clone()
        opt.step()
        ref_opt.step()
    assert losses[2] < losses[0], losses
    worst = max(rel_l2(p.detach(), s.detach()) for s, p in zip(shadow, diff.parameters()))
    print("\n[train] losses %s, flat Adam vs torch Adam worst rel-L2 %.2e" % (losses, worst))
    assert worst < 1e-5
    sd = opt.state_dict()
    assert len(sd["state"]) == len(list(diff.parameters()))


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_recorded_launch_lists_reproduce_the_eager_step(precision):
    """The forward / backward launch lists are recorded on the second call and replayed from the third: the same batch must
    give the same loss and gradients in all three modes, and the lists must really be used.  Tolerance: the GroupNorm /
    bias reductions use atomics, so the summation order differs from run to run: 1e-5 in fp32; in bf16 a last-bit change
    of a reduced statistic flips bf16 roundings of whole activation-gradient tensors downstream (measured 1.4e-3 on the whole
    gradient between two runs of the SAME mode; bf16 eps = 3.9e-3) -> 5e-3."""
    g, spec = load_golden("resdiff_grad_small"), CASES["resdiff_grad_small"]
    net, diff = _build(spec["cfg"], spec["seed"], precision)
    plan = net.train_plan(g["hr"].shape[0], torch.device("cuda:0"))
    outs = []
    for it in range(4):
        for p in diff.parameters():
            p.grad = None
        loss = _train_backward(diff, g, spec)
        outs.append((loss, plan.gflat.clone()))
    assert "fwd" in plan._lists and "bwd" in plan._lists and len(plan._lists["bwd"]) > 300
    for loss, gf in outs[1:]:
        assert abs(loss - outs[0][0]) <= 1e-6 * abs(outs[0][0])
        assert rel_l2(gf, outs[0][1]) < (1e-5 if precision == "fp32" else 5e-3)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_batched_weight_refresh_is_bit_identical_to_the_per_tensor_packs(precision):
    """After an optimizer step the plan re-packs all forward and data-gradient weights with ONE wsr_repack_batch launch
    (job table recorded on the first refresh).  Every destination buffer must equal, bit for bit, what the per-tensor pack
    entry points produce from the same parameters."""
    g, spec = load_golden("resdiff_grad_small"), CASES["resdiff_grad_small"]
    net, diff = _build(spec["cfg"], spec["seed"], precision)
    plan = net.train_plan(g["hr"].shape[0], torch.device("cuda:0"))
    opt = wsr.sub("autograd_glue").FusedAdam(list(diff.parameters()), lr=1e-4)
    opt.attach_flat(plan)
    plan.refresh_weights()
    assert plan._jobtab is not None and plan._jobtab[1] > 100
    cache = plan.eng._pack_cache

    def snapshot():
        torch.cuda.synchronize()
        out = {}
        for k, v in cache.items():
            if isinstance(v, torch.Tensor):
                out[k] = v.clone()
            else:
                out[(k, "w")] = v.w.clone()
                if v.w_vm is not None:
                    out[(k, "vm")] = v.w_vm.clone()
        return out

    torch.manual_seed(5)
    with torch.no_grad():
        for p in diff.parameters():
            p.add_(0.05 * torch.randn_like(p))
    before = nat.launches
    plan.refresh_weights()                       # batched
    assert nat.launches - before == 1
    batched = snapshot()
    for v in cache.values():                     # poison, then redo through the per-tensor path
        (v if isinstance(v, torch.Tensor) else v.w).fill_(7.0)
    plan.batched_refresh = False
    plan._wver = None
    plan.refresh_weights()
    eager = snapshot()
    assert batched.keys() == eager.keys() and len(eager) > 100
    for k in eager:
        assert torch.equal(batched[k], eager[k]), k
    # and the poisoned buffers are rewritten completely by the batched path too
    for v in cache.values():
        (v if isinstance(v, torch.Tensor) else v.w).fill_(7.0)
        if not isinstance(v, torch.Tensor) and v.w_vm is not None:
            v.w_vm.fill_(7.0)
    plan.batched_refresh = True
    plan._wver = None
    plan.refresh_weights()
    again = snapshot()
    for k in eager:
        assert torch.equal(again[k], eager[k]), k


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_srdiff_training_step_gradients_vs_reference(precision):
    """SRDiff (RRDB-conditioned) training step: frozen encoder forward, UNet forward + hand-written backward including the
    cond_proj transposed-convolution weight gradient (expressed as a stride-4 tap-table weight gradient with the operand
    roles swapped).  Every UNet parameter gradient against the oracle's autograd, which is pinned to the REAL reference's
    gradient summaries (tests/golden/srdiff_grad_small.npz)."""
    from conftest import manifest
    from oracle.weights import seeded_state_dict
    g, spec = load_golden("srdiff_grad_small"), CASES["srdiff_grad_small"]
    cfg = spec["cfg"]
    U = wsr.sub("models.diffusion_models.srdiff.unet").UNet
    D = wsr.sub("models.diffusion_models.srdiff.srdiff_diffusion").SRDiffDiffusion
    R = wsr.sub("models.rrdb_encoder.RRDBNet").RRDBNet
    net = U(in_channel=cfg["in_channel"], out_channel=cfg["out_channel"], norm_groups=32, inner_channel=64,
            channel_mults=cfg["channel_mults"], attn_res=cfg["attn_res"], res_blocks=2, dropout=0, image_height=32,
            image_width=64, image_channels=1, precision=precision)
    net = fill_module(net, spec["seed"]).cuda().train()
    diff = D(net, image_height=32, image_width=64, channels=1, conditional=True).cuda()
    diff.rrdb_encoder = fill_module(R(1, 1, 64, 17, 32, precision=precision), spec["seed"] + 1).cuda().eval()
    for p in diff.rrdb_encoder.parameters():
        p.requires_grad_(False)
    diff.set_new_noise_schedule(LINEAR_1000, "cuda:0")
    diff.set_loss("cuda:0")
    u = g["level"].numpy().astype(np.float64)
    ri, un = np.random.randint, np.random.uniform
    np.random.randint = lambda *a, **k: spec["t"]
    np.random.uniform = lambda *a, **k: u
    try:
        loss = diff.p_losses({"HR": g["hr"].cuda(), "SR": g["sr"].cuda(), "LR": g["lr"].cuda()}, noise=g["noise"].cuda())
    finally:
        np.random.randint, np.random.uniform = ri, un
    (loss.sum() / int(g["hr"].numel())).backward()
    rel_loss = abs(float(loss) - float(g["loss"])) / float(g["loss"])
    _, oracle_grads = process.srdiff_param_grads(seeded_state_dict(manifest("srdiff", cfg), spec["seed"]),
                                                 seeded_state_dict(manifest("rrdb"), spec["seed"] + 1), cfg, g["lr"], g["hr"], g["sr"],
                                                 g["level"], g["noise"])
    num = den = 0.0
    worst = (0.0, "")
    for n, p in net.named_parameters():
        assert p.grad is not None, n
        ref = oracle_grads[n].double()
        err = float((p.grad.detach().cpu().double() - ref).norm())
        num += err ** 2
        den += float(ref.norm()) ** 2
        ref_norm = float(g["norm/" + n])
        assert abs(float(ref.norm()) - ref_norm) <= 1e-3 * ref_norm + 1e-12, n
        if ref.numel() >= 16 and float(ref.norm()) > 0:
            worst = max(worst, (err / float(ref.norm()), n))
    total = math.sqrt(num / den)
    cp = rel_l2(net.cond_proj.weight.grad.cpu(), oracle_grads["cond_proj.weight"])
    print("\n[parity] srdiff training step %s: loss rel err %.3e, whole-gradient rel-L2 %.3e, cond_proj.weight %.3e, worst tensor %.3e (%s)"
          % (precision, rel_loss, total, cp, worst[0], worst[1]))
    assert rel_loss < (1e-4 if precision == "fp32" else 2e-2)
    assert total < (1e-4 if precision == "fp32" else 5e-2)
    assert cp < (2e-4 if precision == "fp32" else 1.6e-1)
    assert worst[0] < (2e-4 if precision == "fp32" else 2.5e-1), worst


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_srdiff_joint_training_step_vs_reference(precision):
    """SRDiff with a TRAINABLE RRDB-17 encoder (``lock_weights=False``, srdiff_diffusion.py:176-214): loss = noise loss + l1(rrdb_sr, HR);
    the encoder receives gradients through its SR image and through the six condition features (UNetTrainPlan.cond_grad ->
    _RRDBPlan.backward).  UNet and encoder gradients against the oracle's autograd, which is pinned to the REAL reference's summaries
    (tests/golden/srdiff_joint_grad_small.npz); then one optimizer step moves both parameter sets."""
    from conftest import manifest
    from oracle.cases import calibrate_rrdb_head
    from oracle.weights import seeded_state_dict
    g, spec = load_golden("srdiff_joint_grad_small"), CASES["srdiff_joint_grad_small"]
    cfg = spec["cfg"]
    U = wsr.sub("models.diffusion_models.srdiff.unet").UNet
    D = wsr.sub("models.diffusion_models.srdiff.srdiff_diffusion").SRDiffDiffusion
    R = wsr.sub("models.rrdb_encoder.RRDBNet").RRDBNet
    net = U(in_channel=cfg["in_channel"], out_channel=cfg["out_channel"], norm_groups=32, inner_channel=64,
            channel_mults=cfg["channel_mults"], attn_res=cfg["attn_res"], res_blocks=2, dropout=0, image_height=32,
            image_width=64, image_channels=1, precision=precision)
    net = fill_module(net, spec["seed"]).cuda().train()
    diff = D(net, image_height=32, image_width=64, channels=1, conditional=True, lock_weights=False).cuda()
    diff.rrdb_encoder = calibrate_rrdb_head(fill_module(R(1, 1, 64, 17, 32, precision=precision), spec["seed"] + 1)).cuda().train()
    diff.set_new_noise_schedule(LINEAR_1000, "cuda:0")
    diff.set_loss("cuda:0")
    u = g["level"].numpy().astype(np.float64)
    ri, un = np.random.randint, np.random.uniform
    np.random.randint = lambda *a, **k: spec["t"]
    np.random.uniform = lambda *a, **k: u
    try:
        loss = diff.p_losses({"HR": g["hr"].cuda(), "SR": g["sr"].cuda(), "LR": g["lr"].cuda()}, noise=g["noise"].cuda())
    finally:
        np.random.randint, np.random.uniform = ri, un
    (loss.sum() / int(g["hr"].numel())).backward()
    rel_loss = abs(float(loss.detach()) - float(g["loss"])) / float(g["loss"])
    rrdb_sd = seeded_state_dict(manifest("rrdb"), spec["seed"] + 1)
    rrdb_sd["conv_last.bias"] = torch.full_like(rrdb_sd["conv_last.bias"], 0.5)           # calibrate_rrdb_head
    _, og_unet, og_rrdb = process.srdiff_joint_param_grads(seeded_state_dict(manifest("srdiff", cfg), spec["seed"]), rrdb_sd, cfg,
                                                           g["lr"], g["hr"], g["sr"], g["level"], g["noise"])
    report = {}
    for tag, mod, oracle, prefix in (("unet", net, og_unet, ""), ("rrdb", diff.rrdb_encoder, og_rrdb, "rrdb_encoder.")):
        num = den = 0.0
        worst = (0.0, "")
        gscale = math.sqrt(sum(float(v.double().pow(2).sum()) for v in oracle.values()))
        for n, p in mod.named_parameters():
            assert p.grad is not None, n
            ref = oracle[n].double()
            err = float((p.grad.detach().cpu().double() - ref).norm())
            num += err ** 2
            den += float(ref.norm()) ** 2
            ref_norm = float(g["norm/" + prefix + n])
            assert abs(float(ref.norm()) - ref_norm) <= 2e-3 * ref_norm + 1e-6 * gscale, prefix + n      # oracle == real reference
            if ref.numel() >= 16 and err > 1e-4 * gscale:
                worst = max(worst, (err / max(float(ref.norm()), 1e-30), n))
        report[tag] = (math.sqrt(num / den), worst)
    print("\n[parity] srdiff JOINT training step %s: loss rel err %.3e, whole-gradient rel-L2 unet %.3e / encoder %.3e, worst %s / %s"
          % (precision, rel_loss, report["unet"][0], report["rrdb"][0], report["unet"][1], report["rrdb"][1]))
    assert rel_loss < (1e-4 if precision == "fp32" else 2e-2)
    for tag in ("unet", "rrdb"):
        assert report[tag][0] < (2e-4 if precision == "fp32" else 8e-2), tag          # measured 3.9e-2 / 4.8e-2
        assert report[tag][1][0] < (1e-3 if precision == "fp32" else 3e-1), (tag, report[tag][1])
    # one optimizer step over BOTH parameter sets (the encoder's parameters are outside the UNet's flat buffer)
    FusedAdam = wsr.sub("autograd_glue").FusedAdam
    before_u, before_r = net.cond_proj.weight.detach().clone(), diff.rrdb_encoder.trunk_conv.weight.detach().clone()
    opt = FusedAdam(list(diff.parameters()), lr=1e-4)
    opt.step()
    assert not torch.equal(before_u, net.cond_proj.weight.detach()) and not torch.equal(before_r, diff.rrdb_encoder.trunk_conv.weight.detach())
