"""GPU tests of the training step's second group of kernels (csrc/fd.cu, csrc/backward.cu, the k8/s4 transposed convolution),
each called through the C ABI with the arguments its caller in the training step passes, against float64 torch.autograd of
the same operation written out plainly here, on the same inputs (rounded to bf16 first where the kernel reads bf16):

  * FD_Info_Spliter condition branch: wsr_fd_precompute (lf, hf) + wsr_fd_backward (six parameter gradients), including the
    sigma clamp (both branches, both signs of the pre-abs mean), B = 1, C = 3 and pixel counts that are not multiples of 128;
  * FD noise gate: wsr_fd_gate (with and without a device row index) + wsr_fd_gate_bwd;
  * level embedding: wsr_noise_embed / wsr_noise_embed_bwd (Swish and Mish) and wsr_linear_rows / wsr_linear_rows_bwd at the
    projection width of a built plan;
  * GroupNorm (+ activation, + dropout) backward, vector and scalar kernels, fp32 and bf16;
  * SRDiff's cond_proj = ConvTranspose2d(k 8, s 4, p 2): forward, and the weight / bias / condition gradients the training step
    builds from the same tap tables;
  * wsr_stem_assemble: exact channel layout, zero padding and untouched pad channels.

Buffers a kernel accumulates into (+=) are prefilled with a known non-zero value and the test checks prefill + gradient; outputs
written with = are prefilled with a sentinel that must be overwritten.  Tolerances are rel-L2 per tensor, about 1.5-3x the value
measured on a B200 (written beside each bound)."""
import functools
import math

import pytest
import torch
import torch.nn.functional as F

import wsr
from conftest import rel_l2
from oracle.cases import unet_cfg

pytestmark = pytest.mark.gpu

nat = wsr.pkg.native
engine_mod = wsr.sub("engine")
Engine = engine_mod.Engine
T = wsr.sub("taps")

F64 = torch.float64
NAN = float("nan")


def _dev():
    return torch.device("cuda:0")


def _st():
    return torch.cuda.current_stream(_dev()).cuda_stream


def _nhwc(x, eng, ld=None, coff=0, dt=None):
    N, C, H, W = x.shape
    full = eng.new_act(N, H, W, ld or C, dt=dt, zero=True)
    a = full.slice(coff, C)
    eng.nchw_to_act(x, a)
    return a


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _prefill(ref):
    """fp32 buffer for a += output: a power of two near the reference's magnitude, so that out - prefill loses nothing."""
    s = float(ref.abs().max())
    v = 2.0 ** math.floor(math.log2(s)) if s > 0 else 1.0
    return torch.full(tuple(ref.shape), v, device=ref.device, dtype=torch.float32)


def _bf16(t):
    return t.to(torch.bfloat16).float()


def _report(tag, errs):
    print("\n[train-kernels] %s: %s" % (tag, ", ".join("%s %.2e" % kv for kv in errs.items())))


# ----------------------------------------------------------------------------------------------------------------
# 1. FD_Info_Spliter, condition-only branch (fd_info_spliter.py:61-117)
# ----------------------------------------------------------------------------------------------------------------
def _squeeze(spec):
    """ResSE squeeze of cat([Re, Im]) of a spectrum: (B, 2C) means over (h, w)."""
    return torch.cat([spec.real, spec.imag], 1).mean(dim=(2, 3))


def _highpass(sig, H, W):
    """Gaussian high-pass on the unshifted spectrum, (B, H, W)."""
    u = torch.arange(H, dtype=F64, device=sig.device)[:, None] - H / 2
    v = torch.arange(W, dtype=F64, device=sig.device)[None, :] - W / 2
    return 1 - torch.exp(-(u ** 2 + v ** 2) / (2 * sig[:, None, None] ** 2))


def _fd_sigma(cond, s0, s2):
    """float64: the 4-D spectrum, sigma per sample and the pre-abs channel mean a; sigma = min(|a| + l/2, l - 10), l = min(H, W)."""
    H, W = cond.shape[-2:]
    spec = torch.fft.fftn(cond.to(torch.complex128))
    m = _squeeze(spec)
    se = torch.sigmoid(F.linear(torch.relu(F.linear(m, s0)), s2))
    a = (m * (1 + se)).mean(dim=1)
    ell = min(H, W)
    return spec, torch.minimum(a.abs() + ell / 2, torch.full_like(a, ell - 10.0)), a


def _fd_branch(a, H, W):
    ell = min(H, W)
    if abs(a) + ell / 2 >= ell - 10:
        return "clamped"
    return "unclamped, a > 0" if a > 0 else "unclamped, a < 0"


def _fd_reference(cond, p):
    """float64 lf and hf of the condition branch; p: the six parameters."""
    B, C, H, W = cond.shape
    spec, sig, _ = _fd_sigma(cond, p["sigma_fc0"], p["sigma_fc2"])
    spec_f = spec * _highpass(sig, H, W)[:, None]
    xf = torch.cat([spec_f.real, spec_f.imag], 1)
    se = torch.sigmoid(F.linear(torch.relu(F.linear(_squeeze(spec_f), p["hf_fc0"])), p["hf_fc2"]))
    gate = xf * (1 + se[:, :, None, None])
    lf = cond * (torch.einsum("oc,bchw->bohw", p["ct_w"], gate) + p["ct_b"][None, :, None, None])
    hf = torch.fft.ifftn(spec_f).abs()
    return lf, hf


FD_PARAMS = ("sigma_fc0", "sigma_fc2", "hf_fc0", "hf_fc2", "ct_w", "ct_b")
FD_CASES = [
    pytest.param((2, 1, 32, 64), "", id="B2C1-32x64"),                 # gradient-fixture shape
    pytest.param((4, 1, 128, 256), "", id="B4C1-128x256"),             # configs[2] training shape
    pytest.param((8, 3, 128, 256), "", id="B8C3-128x256"),             # configs[4] shape
    pytest.param((1, 3, 24, 40), "", id="B1C3-24x40"),                 # B-axis DFT pass skipped; HW = 960 = 7.5 x 128
    pytest.param((3, 2, 16, 48), "", id="B3C2-16x48-clamped"),         # l = 16: sigma is always clamped
    pytest.param((2, 1, 32, 64), "signs", id="B2C1-32x64-signs"),      # a > 0 for sample 0, a < 0 for sample 1
]


@functools.lru_cache(maxsize=None)
def _fd_inputs(shape, kind):
    """CPU fp32 inputs: condition, parameters, output gradients."""
    B, C, H, W = shape
    g = _gen(1000 + 97 * B + 31 * C + H + W + (7 if kind else 0))
    cond = torch.randn(B, C, H, W, generator=g)
    if kind == "signs":
        # the mean of the 4-D spectrum over (h, w) is the (B, C)-DFT of pixel (0, 0): at B = 2, C = 1 it is x0 + x1 for sample 0 and
        # x0 - x1 for sample 1, so these values make a > 0 for sample 0 and a < 0 for sample 1, both well inside l/2 - 10 = 6
        cond[0, 0, 0, 0], cond[1, 0, 0, 0] = 0.5, 2.0
    C2 = 2 * C
    p = {"sigma_fc0": torch.randn(C, C2, generator=g) / math.sqrt(C2), "sigma_fc2": torch.randn(C2, C, generator=g) / math.sqrt(C),
         "hf_fc0": torch.randn(C, C2, generator=g) / math.sqrt(C2), "hf_fc2": torch.randn(C2, C, generator=g) / math.sqrt(C),
         "ct_w": torch.randn(C, C2, generator=g) / math.sqrt(C2), "ct_b": 0.1 * torch.randn(C, generator=g)}
    # a ResSE hidden unit that is inactive for the whole batch leaves its block's gradients exactly zero and that part of the
    # backward untested (C = 1 has a single unit): flip the sign of such fc0 rows, sigma_resSE first since HF_guided_resSE's input
    # depends on sigma
    spec = torch.fft.fftn(cond.to(torch.complex128))
    for key, m in (("sigma_fc0", lambda: _squeeze(spec)),
                   ("hf_fc0", lambda: _squeeze(spec * _highpass(_fd_sigma(cond.double(), p["sigma_fc0"].double(),
                                                                           p["sigma_fc2"].double())[1], H, W)[:, None]))):
        dead = (F.linear(m(), p[key].double()) <= 0).all(dim=0)
        p[key][dead] = -p[key][dead]
    return cond, p, torch.randn(B, C, H, W, generator=g), torch.randn(B, C, H, W, generator=g)


def _fd_branches_covered():
    seen = set()
    for case in FD_CASES:
        shape, kind = case.values
        cond, p, _, _ = _fd_inputs(shape, kind)
        _, _, a = _fd_sigma(cond.double(), p["sigma_fc0"].double(), p["sigma_fc2"].double())
        seen.update(_fd_branch(float(v), shape[2], shape[3]) for v in a)
    return seen


# the cases must run both branches of the sigma clamp in the backward (fd_bwd_sigma_kernel), and both signs of |a|'s derivative
_FD_SEEN = _fd_branches_covered()
assert _FD_SEEN == {"clamped", "unclamped, a > 0", "unclamped, a < 0"}, _FD_SEEN


@pytest.mark.parametrize("shape,kind", FD_CASES)
def test_fd_splitter_vs_float64_autograd(shape, kind):
    dev, st = _dev(), _st()
    B, C, H, W = shape
    cond_c, p_c, glf_c, ghf_c = _fd_inputs(shape, kind)
    cond, g_lf, g_hf = cond_c.to(dev), glf_c.to(dev), ghf_c.to(dev)
    p = {k: v.to(dev).contiguous() for k, v in p_c.items()}
    lf = torch.full_like(cond, NAN)
    hf = torch.full_like(cond, NAN)
    work = torch.empty(nat.call("wsr_fd_precompute_workspace_bytes", B, C, H, W), device=dev, dtype=torch.uint8)
    nat.call("wsr_fd_precompute", cond.data_ptr(), B, C, H, W, *[p[k].data_ptr() for k in FD_PARAMS], C, lf.data_ptr(),
             hf.data_ptr(), work.data_ptr(), st)

    p64 = {k: v.double().requires_grad_(True) for k, v in p.items()}
    lf_r, hf_r = _fd_reference(cond.double(), p64)
    (lf_r * g_lf.double() + hf_r * g_hf.double()).sum().backward()
    ref = {k: p64[k].grad for k in FD_PARAMS}
    all_clamped = {_fd_branch(float(v), H, W) for v in _fd_sigma(cond.double(), p64["sigma_fc0"], p64["sigma_fc2"])[2]} == {"clamped"}
    for k in FD_PARAMS:                      # every gradient path runs, except sigma_resSE's when every sample is clamped
        assert bool((ref[k] != 0).any()) != (all_clamped and k.startswith("sigma")), k
    pre = {k: _prefill(ref[k]) for k in FD_PARAMS}
    d = {k: pre[k].clone() for k in FD_PARAMS}
    bwork = torch.empty(nat.call("wsr_fd_backward_workspace_bytes", B, C, H, W), device=dev, dtype=torch.uint8)
    nat.call("wsr_fd_backward", cond.data_ptr(), B, C, H, W, *[p[k].data_ptr() for k in FD_PARAMS[:5]], g_lf.data_ptr(),
             g_hf.data_ptr(), work.data_ptr(), bwork.data_ptr(), *[d[k].data_ptr() for k in FD_PARAMS], st)
    torch.cuda.synchronize()

    errs = {"lf": rel_l2(lf, lf_r.detach()), "hf": rel_l2(hf, hf_r.detach())}
    errs.update({k: rel_l2(d[k] - pre[k], ref[k]) for k in FD_PARAMS})
    _report("fd %s%s" % (shape, " " + kind if kind else ""), errs)
    assert torch.isfinite(lf).all() and torch.isfinite(hf).all()
    assert errs["lf"] < 3e-7 and errs["hf"] < 3e-7, errs                  # measured <= 1.1e-7
    for k in FD_PARAMS:
        assert errs[k] < 6e-6, (k, errs)                                   # measured <= 2.6e-6 (hf_fc0, signs case)
    # where the reference's sigma_resSE gradient is exactly zero (clamped samples, inactive ReLU units) the kernel adds nothing
    for k in ("sigma_fc0", "sigma_fc2"):
        z = ref[k] == 0
        assert torch.equal(d[k][z], pre[k][z]), k


# ----------------------------------------------------------------------------------------------------------------
# 2. FD noise gate (fd_info_spliter.py:43-47): gate[b, c, w] = ne[w] * (1 + sigmoid(fc2 relu(fc0 * mean_w ne)))
# ----------------------------------------------------------------------------------------------------------------
def _gate_reference(ne, fc0, fc2):
    """ne (B, W) float64.  The ResSE input is ne tiled over C and H, so its mean over (H, W) is mean_w ne for every channel."""
    m = ne.mean(dim=1, keepdim=True).expand(-1, fc0.shape[1])
    se = torch.sigmoid(F.linear(torch.relu(F.linear(m, fc0)), fc2))
    return ne[:, None, :] * (1 + se[:, :, None])


GATE_CASES = [
    # B, C, H, W, hidden, dxin dtype, extra channels of dxin (d_ld = 5C + extra)
    pytest.param(4, 1, 128, 256, 1, "f32", 0, id="B4C1-128x256-h1-f32-ld5C"),
    pytest.param(4, 1, 128, 256, 1, "bf16", 3, id="B4C1-128x256-h1-bf16-ld5C+3"),
    pytest.param(4, 3, 128, 256, 1, "bf16", 0, id="B4C3-128x256-h1-bf16-ld5C"),
    pytest.param(1, 3, 5, 72, 1, "f32", 3, id="B1C3-5x72-h1-f32-ld5C+3"),
    pytest.param(1, 1, 5, 72, 4, "bf16", 0, id="B1C1-5x72-h4-bf16-ld5C"),
    pytest.param(4, 3, 5, 256, 5, "f32", 3, id="B4C3-5x256-h5-f32-ld5C+3"),
    pytest.param(1, 3, 128, 72, 2, "bf16", 3, id="B1C3-128x72-h2-bf16-ld5C+3"),
]


@pytest.mark.parametrize("B,C,H,W,hidden,ddt,extra", GATE_CASES)
def test_fd_gate_forward_and_backward_vs_float64_autograd(B, C, H, W, hidden, ddt, extra):
    dev, st = _dev(), _st()
    g = _gen(2000 + 13 * B + 7 * C + H + W + hidden)
    rows, ne_ld, dne_ld, d_ld = B + 2, W + 37, W + 21, 5 * C + extra
    ne_rows = (0.5 + 0.5 * torch.randn(rows, ne_ld, generator=g)).to(dev)        # rows of the level projection; ne at the front
    fc0 = torch.randn(hidden, C, generator=g)
    fc0[0] = fc0[0].abs()                     # mean_w ne > 0: hidden unit 0 is active, so the term through mean_w ne is exercised
    fc0 = fc0.to(dev)
    fc2 = (torch.randn(C, hidden, generator=g) / math.sqrt(hidden)).to(dev)
    x = torch.randn(B, C, H, W, generator=g).to(dev)
    dxin = torch.randn(B, H, W, d_ld, generator=g).to(dev, torch.bfloat16 if ddt == "bf16" else torch.float32)
    row_index = torch.tensor([rows - 1], dtype=torch.int32, device=dev)

    # forward: per-sample rows, then every sample reading the row named by the device index (the sampler's level table)
    gate = torch.full((B, C, W), NAN, device=dev)
    gate_ix = torch.full((B, C, W), NAN, device=dev)
    nat.call("wsr_fd_gate", ne_rows.data_ptr(), ne_ld, 0, B, C, W, fc0.data_ptr(), fc2.data_ptr(), hidden, gate.data_ptr(), st)
    nat.call("wsr_fd_gate", ne_rows.data_ptr(), ne_ld, row_index.data_ptr(), B, C, W, fc0.data_ptr(), fc2.data_ptr(), hidden,
             gate_ix.data_ptr(), st)

    ne64 = ne_rows[:B, :W].double().requires_grad_(True)
    fc0_64, fc2_64 = fc0.double().requires_grad_(True), fc2.double().requires_grad_(True)
    gate_r = _gate_reference(ne64, fc0_64, fc2_64)
    gate_ix_r = _gate_reference(ne_rows[rows - 1:, :W].double(), fc0.double(), fc2.double()).expand(B, -1, -1)
    D = dxin[..., 2 * C:3 * C].permute(0, 3, 1, 2).double()          # d denoise_x: channels [2C, 3C) of the stem's input gradient
    (D * x.double() * gate_r[:, :, None, :]).sum().backward()

    dne = torch.full((B, dne_ld), 7.0, device=dev)
    pre0, pre2 = _prefill(fc0_64.grad), _prefill(fc2_64.grad)
    dfc0, dfc2 = pre0.clone(), pre2.clone()
    nat.call("wsr_fd_gate_bwd", dxin.data_ptr(), nat.BF16 if ddt == "bf16" else nat.F32, d_ld, 2 * C, x.data_ptr(), ne_rows.data_ptr(),
             ne_ld, B, C, H, W, fc0.data_ptr(), fc2.data_ptr(), hidden, dne.data_ptr(), dne_ld, dfc0.data_ptr(), dfc2.data_ptr(), st)
    torch.cuda.synchronize()

    errs = {"gate": rel_l2(gate, gate_r.detach()), "gate[row_index]": rel_l2(gate_ix, gate_ix_r), "dne": rel_l2(dne[:, :W], ne64.grad),
            "dfc0": rel_l2(dfc0 - pre0, fc0_64.grad), "dfc2": rel_l2(dfc2 - pre2, fc2_64.grad)}
    _report("fd_gate B%d C%d %dx%d h%d %s ld%d" % (B, C, H, W, hidden, ddt, d_ld), errs)
    assert torch.isfinite(gate).all() and torch.isfinite(gate_ix).all() and torch.isfinite(dne[:, :W]).all()
    assert bool((dne[:, W:] == 7.0).all())                  # dne is written with =, and only its W leading entries per row
    assert errs["gate"] < 2e-7 and errs["gate[row_index]"] < 2e-7, errs    # measured <= 7.2e-8
    assert errs["dne"] < 6e-7, errs                                         # measured <= 2.4e-7
    # dfc0 / dfc2 sum ~1e5 products whose total nearly cancels for some inputs: measured <= 1.6e-5 (B4C1-128x256-bf16), else <= 6e-7
    assert errs["dfc0"] < 4e-5 and errs["dfc2"] < 4e-5, errs


# ----------------------------------------------------------------------------------------------------------------
# 3. level embedding: temb = W2 act(W1 enc(level) + b1) + b2 (resdiff/unet.py:46-53 Swish, srdiff/unet.py:49-54 Mish), then the
#    concatenated FeatureWiseAffine projections proj = temb Wp^T + bp
# ----------------------------------------------------------------------------------------------------------------
def _embed_reference(level, inner, w1, b1, w2, b2, act):
    half = inner // 2
    k = torch.arange(half, dtype=F64, device=level.device) / half
    arg = level[:, None] * torch.exp(-math.log(1e4) * k[None, :])
    enc = torch.cat([torch.sin(arg), torch.cos(arg)], dim=1)
    pre = F.linear(enc, w1, b1)
    hid = pre * torch.sigmoid(pre) if act == "swish" else pre * torch.tanh(F.softplus(pre))
    return F.linear(hid, w2, b2)


@pytest.mark.parametrize("inner,act,R", [
    pytest.param(64, "swish", 3, id="inner64-swish-R3"), pytest.param(64, "mish", 64, id="inner64-mish-R64"),
    pytest.param(128, "swish", 1, id="inner128-swish-R1"), pytest.param(128, "mish", 3, id="inner128-mish-R3"),
    pytest.param(64, "mish", 1, id="inner64-mish-R1"), pytest.param(128, "swish", 64, id="inner128-swish-R64")])
def test_noise_embed_forward_and_backward_vs_float64_autograd(inner, act, R):
    dev, st = _dev(), _st()
    g = _gen(3000 + inner + R + (1 if act == "mish" else 0))
    level = torch.cat([torch.tensor([1.0, 5e-3]), torch.rand(max(R - 2, 0), generator=g)])[:R].to(dev)
    w1 = (torch.randn(4 * inner, inner, generator=g) / math.sqrt(inner)).to(dev)
    b1 = (0.1 * torch.randn(4 * inner, generator=g)).to(dev)
    w2 = (torch.randn(inner, 4 * inner, generator=g) / math.sqrt(4 * inner)).to(dev)
    b2 = (0.1 * torch.randn(inner, generator=g)).to(dev)
    dtemb = torch.randn(R, inner, generator=g).to(dev)
    code = nat.ACT_SWISH if act == "swish" else nat.ACT_MISH

    temb = torch.full((R, inner), NAN, device=dev)
    nat.call("wsr_noise_embed", level.data_ptr(), R, inner, w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(), code,
             temb.data_ptr(), st)
    prm = [t.double().requires_grad_(True) for t in (w1, b1, w2, b2)]
    temb_r = _embed_reference(level.double(), inner, *prm, act)
    (temb_r * dtemb.double()).sum().backward()
    pre = [_prefill(t.grad) for t in prm]
    out = [t.clone() for t in pre]
    nat.call("wsr_noise_embed_bwd", level.data_ptr(), R, inner, w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), code, dtemb.data_ptr(),
             *[t.data_ptr() for t in out], st)
    torch.cuda.synchronize()
    errs = {"temb": rel_l2(temb, temb_r.detach())}
    errs.update({n: rel_l2(o - p_, t.grad) for n, o, p_, t in zip(("dw1", "db1", "dw2", "db2"), out, pre, prm)})
    _report("noise_embed inner%d %s R%d" % (inner, act, R), errs)
    assert torch.isfinite(temb).all()
    for k, e in errs.items():
        assert e < 1e-5, (k, errs)          # measured <= 4.9e-6 (Mish: fast-math log1p / exp / tanh), <= 2.3e-6 (Swish)


@pytest.fixture(scope="module")
def plan_widths():
    """Width P of the concatenated level projection of built ResDiff plans: configs[2] (Cfg-A, inner 64) and configs[4]
    (3 variables, inner 128), both 128x256."""
    U = wsr.sub("models.diffusion_models.resdiff.unet").UNet
    out = {}
    for tag, c_img, inner in (("cfg2", 1, 64), ("cfg4", 3, 128)):
        cfg = unet_cfg(128, 256, inner=inner, c_img=c_img)
        net = U(in_channel=cfg["in_channel"], out_channel=cfg["out_channel"], norm_groups=cfg["norm_groups"], inner_channel=inner,
                channel_mults=cfg["channel_mults"], attn_res=cfg["attn_res"], res_blocks=cfg["res_blocks"], dropout=cfg["dropout"],
                image_height=128, image_width=256, image_channels=c_img, precision="fp32").to(_dev())
        pl = net.plan(1, _dev(), "fp32")
        out[tag] = (inner, pl.P)
        del net, pl
    torch.cuda.empty_cache()
    return out


# P + 13: P * K is a multiple of 256 for both plans, so only the odd width gives linear_rows_bwd's weight kernel a partial block
@pytest.mark.parametrize("cfg,extra,R,null", [
    pytest.param("cfg2", 0, 4, "", id="cfg2-K64-P-R4"), pytest.param("cfg2", 13, 1, "db", id="cfg2-K64-P+13-R1-db=NULL"),
    pytest.param("cfg2", 0, 64, "dw", id="cfg2-K64-P-R64-dw=db=NULL"), pytest.param("cfg4", 0, 64, "", id="cfg4-K128-P-R64"),
    pytest.param("cfg4", 13, 4, "", id="cfg4-K128-P+13-R4"), pytest.param("cfg4", 0, 1, "db", id="cfg4-K128-P-R1-db=NULL")])
def test_linear_rows_forward_and_backward_vs_float64_autograd(plan_widths, cfg, extra, R, null):
    dev, st = _dev(), _st()
    K, P = plan_widths[cfg]
    P += extra
    g = _gen(4000 + P + R)
    x = torch.randn(R, K, generator=g).to(dev)
    w = (torch.randn(P, K, generator=g) / math.sqrt(K)).to(dev)
    b = (0.1 * torch.randn(P, generator=g)).to(dev)
    dy = torch.randn(R, P, generator=g).to(dev)
    y = torch.full((R, P), NAN, device=dev)
    nat.call("wsr_linear_rows", x.data_ptr(), R, K, w.data_ptr(), b.data_ptr(), P, y.data_ptr(), st)
    x64, w64, b64 = (t.double().requires_grad_(True) for t in (x, w, b))
    y_r = F.linear(x64, w64, b64)
    (y_r * dy.double()).sum().backward()
    pre_w, pre_b = _prefill(w64.grad), _prefill(b64.grad)
    dx = torch.full((R, K), NAN, device=dev)
    dw, db = pre_w.clone(), pre_b.clone()
    nat.call("wsr_linear_rows_bwd", x.data_ptr(), R, K, w.data_ptr(), dy.data_ptr(), P, dx.data_ptr(),
             0 if null == "dw" else dw.data_ptr(), 0 if null in ("dw", "db") else db.data_ptr(), st)
    torch.cuda.synchronize()
    errs = {"y": rel_l2(y, y_r.detach()), "dx": rel_l2(dx, x64.grad)}
    if null != "dw":
        errs["dw"] = rel_l2(dw - pre_w, w64.grad)
    if not null:
        errs["db"] = rel_l2(db - pre_b, b64.grad)
    _report("linear_rows K%d P%d R%d null=%s" % (K, P, R, null or "-"), errs)
    assert torch.isfinite(y).all() and torch.isfinite(dx).all()
    if null == "dw":
        assert torch.equal(dw, pre_w)
    if null:
        assert torch.equal(db, pre_b)
    for k, e in errs.items():
        assert e < 6e-7, (k, errs)          # measured <= 2.4e-7


# ----------------------------------------------------------------------------------------------------------------
# 4. GroupNorm (+ Swish) (+ dropout) backward: Engine.gn_bwd -> wsr_gn_bwd_reduce + wsr_gn_bwd_apply
# ----------------------------------------------------------------------------------------------------------------
GN_GROUPS = 32
SENT = 3.0                   # sentinel of channels outside the slice (exact in bf16)


def _gn_bwd_path(x, da, dx):
    """Which kernel pair wsr_gn_bwd_reduce / wsr_gn_bwd_apply run: mirror of gn_bwd_vec and the launchers' shared-memory test."""
    want = 8 if x.dt == nat.BF16 else 4
    ok = (x.C % want == 0 and all(a.ld % want == 0 and a.ptr % 16 == 0 for a in (x, da, dx)) and x.C // want <= 1024
          and 4 * x.C * 4 <= 48 * 1024)
    return "vec" if ok else "scalar"


def _gn_cases():
    shapes = [(2, 64, 8, 16), (3, 96, 5, 7), (1, 512, 16, 32), (2, 1024, 8, 16), (4, 64, 128, 256)]
    combos = [("f32", "vec"), ("f32", "scalar"), ("bf16", "vec"), ("bf16", "scalar")]
    out = []
    for i, shape in enumerate(shapes):
        for j, (dt, path) in enumerate(combos):
            p = 0.2 if (i + j) % 2 else 0.0
            act = ("swish", "none")[(i + j // 2) % 2]
            acc = (i + j + j // 2) % 2
            out.append(pytest.param(dt, path, shape, act, acc, p, id="%s-%s-N%dC%d-%dx%d-%s-acc%d-p%g" % (
                (dt, path) + shape + (act, acc, p))))
    return out


GN_CASES = _gn_cases()
assert {(c.values[0], c.values[1], c.values[5]) for c in GN_CASES} == {(d, q, p) for d in ("f32", "bf16") for q in ("vec", "scalar")
                                                                        for p in (0.0, 0.2)}
assert {c.values[3] for c in GN_CASES} == {"swish", "none"} and {c.values[4] for c in GN_CASES} == {0, 1}


def _gn_inputs(shape, dt, seed):
    N, C, H, W = shape
    g = _gen(seed)
    x = torch.randn(N, C, H, W, generator=g) * 1.5 + 0.3
    da = torch.randn(N, C, H, W, generator=g)
    gamma = 1 + 0.1 * torch.randn(C, generator=g)
    beta = 0.1 * torch.randn(C, generator=g)
    pre = torch.randn(N, C, H, W, generator=g)
    if dt == "bf16":
        x, da = _bf16(x), _bf16(da)
    return [t.to(_dev()) for t in (x, da, gamma, beta, pre)]


def _gn_bwd_run(dt, path, shape, act, acc, p, seed=5):
    """Runs Engine.gn_bwd on a channel slice laid out for ``path``; returns kernel outputs, the float64 autograd reference and
    the prefills.  Channels outside the slice must keep their sentinel."""
    dev, st = _dev(), _st()
    eng = Engine(dev, "bf16" if dt == "bf16" else "fp32")
    N, C, H, W = shape
    x, da, gamma, beta, pre = _gn_inputs(shape, dt, seed)
    # scalar path: a slice of a wider buffer whose first channel is not 16-byte aligned
    coff, ld = (0, C) if path == "vec" else ((4, C + 8) if dt == "bf16" else (1, C + 4))
    arena = engine_mod.StatsArena()
    xs = eng.new_act(N, H, W, ld, stats=arena).slice(coff, C)
    arena.finalize(dev)
    eng.nchw_to_act(x, xs)
    eng.gn_stats(xs)
    das = _nhwc(da, eng, ld=ld, coff=coff)
    dxf = eng.new_act(N, H, W, ld)
    dxf.buf.fill_(SENT)
    dxs = dxf.slice(coff, C)
    assert _gn_bwd_path(xs, das, dxs) == path
    seed_d, tag_d = 1234 + seed, 7
    mask = torch.ones(N, C, H, W, device=dev, dtype=F64)
    if p > 0:
        m = torch.empty(N * H * W * C, device=dev)
        nat.call("wsr_dropout_mask", m.data_ptr(), N, H * W, C, p, seed_d, tag_d, st)
        mask = m.view(N, H, W, C).permute(0, 3, 1, 2).double()

    x64, g64, b64 = (t.double().requires_grad_(True) for t in (x, gamma, beta))
    z = F.group_norm(x64, GN_GROUPS, g64, b64, eps=1e-5)
    y = z * torch.sigmoid(z) if act == "swish" else z
    (y * mask * da.double()).sum().backward()
    ref = {"dx": x64.grad, "dgamma": g64.grad, "dbeta": b64.grad, "colsum": x64.grad.sum(dim=(2, 3))}

    if acc:
        eng.nchw_to_act(pre * ref["dx"].float().pow(2).mean().sqrt(), dxs)
        before = dxs.to_nchw(eng)
    else:
        dxf.buf[..., coff:coff + C] = NAN
        before = torch.zeros(N, C, H, W, device=dev)
    pre_g, pre_b = _prefill(ref["dgamma"]), _prefill(ref["dbeta"])
    dg, db = pre_g.clone(), pre_b.clone()
    colsum = torch.full((N, C + 3), SENT, device=dev)
    colsum[:, :C] = NAN
    red = torch.zeros(N * 2 * C, device=dev, dtype=F64)
    eng.gn_bwd(xs, gamma, beta, GN_GROUPS, nat.ACT_SWISH if act == "swish" else nat.ACT_NONE, das, dxs, red.data_ptr(), dg, db,
               bool(acc), colsum.data_ptr(), C + 3, (p, seed_d, tag_d))
    torch.cuda.synchronize()
    full = dxf.buf.float()
    assert bool((full[..., :coff] == SENT).all()) and bool((full[..., coff + C:] == SENT).all())
    assert bool((colsum[:, C:] == SENT).all())
    out = {"dx": dxs.to_nchw(eng) - before, "dgamma": dg - pre_g, "dbeta": db - pre_b, "colsum": colsum[:, :C], "red": red}
    return out, ref


@pytest.mark.parametrize("dt,path,shape,act,acc,p", GN_CASES)
def test_gn_backward_vs_float64_autograd(dt, path, shape, act, acc, p):
    out, ref = _gn_bwd_run(dt, path, shape, act, acc, p)
    assert torch.isfinite(out["dx"]).all() and torch.isfinite(out["colsum"]).all()
    errs = {k: rel_l2(out[k], ref[k]) for k in ("dx", "dgamma", "dbeta", "colsum")}
    _report("gn_bwd %s %s %s %s acc%d p%g" % (dt, path, shape, act, acc, p), errs)
    # bf16 dx: the output-rounding floor, measured 1.7e-3 (overwrite) / 2.4e-3 (accumulate: the prefill + gradient is rounded too);
    # fp32 dx measured <= 9.5e-8; fp32 reductions (also from bf16 inputs) measured <= 2.1e-7
    assert errs["dx"] < (4e-3 if dt == "bf16" else 3e-7), errs
    for k in ("dgamma", "dbeta", "colsum"):
        assert errs[k] < 5e-7, (k, errs)


@pytest.mark.parametrize("dt", ["f32", "bf16"])
@pytest.mark.parametrize("shape", [pytest.param((3, 96, 5, 7), id="N3C96-5x7"), pytest.param((2, 1024, 8, 16), id="N2C1024-8x16")])
def test_gn_backward_vec_and_scalar_paths_agree(dt, shape):
    """Same data through both kernel pairs (Swish, dropout 0.2, overwrite): they differ only in summation order."""
    vec, _ = _gn_bwd_run(dt, "vec", shape, "swish", 0, 0.2, seed=9)
    sca, _ = _gn_bwd_run(dt, "scalar", shape, "swish", 0, 0.2, seed=9)
    errs = {k: rel_l2(vec[k], sca[k]) for k in ("dx", "dgamma", "dbeta", "colsum", "red")}
    _report("gn_bwd vec vs scalar %s %s" % (dt, shape), errs)
    for k in ("dgamma", "dbeta", "colsum", "red"):
        assert errs[k] < 4e-7, (k, errs)                                   # measured <= 1.4e-7
    assert errs["dx"] < (5e-6 if dt == "bf16" else 2e-7), errs             # measured 1.9e-6 (a few bf16 roundings flip) / 5.6e-8


# ----------------------------------------------------------------------------------------------------------------
# 5. SRDiff cond_proj = ConvTranspose2d(384 -> 64, k 8, s 4, p 2) (srdiff/unet.py:43-45) and its training-step gradients
# ----------------------------------------------------------------------------------------------------------------
CONVT_SHAPES = [pytest.param((2, 8, 16), id="N2-8x16"), pytest.param((1, 32, 64), id="N1-32x64")]
CIN_T, COUT_T = 384, 64


def _convt_inputs(shape, seed):
    N, h, w = shape
    g = _gen(seed)
    x = torch.randn(N, CIN_T, h, w, generator=g)
    wt = torch.randn(CIN_T, COUT_T, 8, 8, generator=g) / math.sqrt(CIN_T * 4)
    b = 0.1 * torch.randn(COUT_T, generator=g)
    gy = torch.randn(N, COUT_T, 4 * h, 4 * w, generator=g)
    return [t.to(_dev()) for t in (x, wt, b, gy)]


@pytest.mark.parametrize("xdt,ydt", [("f32", "f32"), ("f32", "bf16"), ("bf16", "f32"), ("bf16", "bf16")])
@pytest.mark.parametrize("shape", CONVT_SHAPES)
def test_conv_transpose_k8s4_vs_float64(shape, xdt, ydt):
    dev, st = _dev(), _st()
    eng = Engine(dev, "fp32")
    N, h, w = shape
    x, wt, b, _ = _convt_inputs(shape, 6000 + h)
    xd, yd = (nat.BF16 if xdt == "bf16" else nat.F32), (nat.BF16 if ydt == "bf16" else nat.F32)
    if xdt == "bf16":
        x, wt = _bf16(x), _bf16(wt)
    xa = _nhwc(x, eng, ld=CIN_T + 8, dt=xd)                                        # x_ld > Cin
    wp = torch.empty(64 * COUT_T * CIN_T, device=dev, dtype=torch.bfloat16 if xdt == "bf16" else torch.float32)
    nat.call("wsr_pack_convT_weight", wt.data_ptr(), CIN_T, COUT_T, 8, 8, wp.data_ptr(), xd, st)
    yf = eng.new_act(N, 4 * h, 4 * w, COUT_T + 8, dt=yd)
    yf.buf.fill_(SENT)
    ya = yf.slice(4, COUT_T)                                                       # y_ld > Cout, channel offset 4
    ya.buf[..., 4:4 + COUT_T] = NAN
    nat.call("wsr_conv_transpose_k8s4", xa.ptr, xd, N, h, w, CIN_T, xa.ld, wp.data_ptr(), b.data_ptr(), COUT_T, ya.ptr, yd, ya.ld, st)
    y = ya.to_nchw(eng)
    torch.cuda.synchronize()
    ref = F.conv_transpose2d(x.double(), wt.double(), b.double(), stride=4, padding=2)
    full = yf.buf.float()
    assert bool((full[..., :4] == SENT).all()) and bool((full[..., 4 + COUT_T:] == SENT).all())
    assert torch.isfinite(y).all()
    err = rel_l2(y, ref)
    _report("conv_transpose_k8s4 %s x %s y %s" % (shape, xdt, ydt), {"y": err})
    assert err < (3e-3 if ydt == "bf16" else 2e-6), err                   # measured 1.7e-3 (bf16 output rounding) / <= 7.0e-7


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("shape", CONVT_SHAPES)
def test_conv_transpose_k8s4_gradients_vs_float64_autograd(shape, precision):
    """dW: the four 16-tap weight-gradient tables with the operand roles swapped; dbias: column sums of dY; dcond: the four 16-tap
    stride-4 launches over dY on the (in, out, 8, 8) parameter packed as an OIHW convolution weight (unet_train.py backward tail)."""
    dev, st = _dev(), _st()
    eng = Engine(dev, precision)
    N, h, w = shape
    x, wt, b, gy = _convt_inputs(shape, 7000 + h)
    if precision == "bf16":
        x, wt, gy = _bf16(x), _bf16(wt), _bf16(gy)
    xa = _nhwc(x, eng)
    gya = _nhwc(gy, eng)
    x64, w64, b64 = (t.double().requires_grad_(True) for t in (x, wt, b))
    F.conv_transpose2d(x64, w64, b64, stride=4, padding=2).backward(gy.double())

    pre_w, pre_b = _prefill(w64.grad), _prefill(b64.grad)
    gw, gb = pre_w.clone(), pre_b.clone()
    for tp in T.conv_transpose_k8s4_wgrad_taps(h, w):
        eng.wgrad(gya, xa, tp, gw, (1, COUT_T * 64, 64), None, 1, force_simt=True)
    nat.call("wsr_col_sums", gya.ptr, gya.dt, N * 16 * h * w, COUT_T, gya.ld, gb.data_ptr(), st)
    pc = eng.pack_conv(wt, None)
    dcond = eng.new_act(N, h, w, CIN_T)
    dcond.buf.fill_(NAN)
    for q, tp in enumerate(T.conv_transpose_k8s4_wgrad_taps(h, w)):
        eng.conv(gya, pc, dcond, taps=tp, bias=False, res=dcond if q else None, force_simt=True)
    dc = dcond.to_nchw(eng)
    torch.cuda.synchronize()
    assert torch.isfinite(dc).all()
    errs = {"dW": rel_l2(gw - pre_w, w64.grad), "dbias": rel_l2(gb - pre_b, b64.grad), "dcond": rel_l2(dc, x64.grad)}
    _report("conv_transpose_k8s4 grads %s %s" % (shape, precision), errs)
    assert errs["dW"] < 1e-6 and errs["dbias"] < 5e-6, errs                # measured <= 3.7e-7 / 2.0e-6
    assert errs["dcond"] < (4e-3 if precision == "bf16" else 1.5e-6), errs  # measured 2.6e-3 (four bf16 partial sums) / 5.7e-7


# ----------------------------------------------------------------------------------------------------------------
# 6. wsr_stem_assemble: stem input = cat([x, cond, x * gate, lf, hf]) (fd_info_spliter.py:117) in a 64-channel NHWC buffer
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", ["f32", "bf16"])
@pytest.mark.parametrize("C", [pytest.param(1, id="C1"), pytest.param(3, id="C3")])
def test_stem_assemble_channels_padding_and_untouched_tail(C, dt):
    dev, st = _dev(), _st()
    B, H, W, Cpad = 2, 16, 40, 64
    g = _gen(8000 + C)
    x, cond, lf, hf = (torch.randn(B, C, H, W, generator=g).to(dev) for _ in range(4))
    gate = torch.randn(B, C, W, generator=g).to(dev)
    tdt = torch.bfloat16 if dt == "bf16" else torch.float32
    y = torch.full((B, H, W, Cpad), SENT, device=dev, dtype=tdt)
    nat.call("wsr_stem_assemble", x.data_ptr(), cond.data_ptr(), gate.data_ptr(), lf.data_ptr(), hf.data_ptr(), B, C, H, W,
             y.data_ptr(), nat.BF16 if dt == "bf16" else nat.F32, Cpad, st)
    torch.cuda.synchronize()
    ref = torch.cat([x, cond, x * gate[:, :, None, :], lf, hf], 1).permute(0, 2, 3, 1).to(tdt)
    assert torch.equal(y[..., :5 * C], ref)
    nwrite = (5 * C + 7) // 8 * 8 if dt == "bf16" else 5 * C
    assert bool((y[..., 5 * C:nwrite] == 0).all())             # bf16 writes whole 8-channel vectors: the pad up to nwrite is zero
    assert bool((y[..., nwrite:] == SENT).all())               # channels beyond are never touched
