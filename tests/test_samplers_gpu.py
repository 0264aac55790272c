"""Fewer-step samplers on the GPU: the multistep kernels (wsr_sampler_step_multistep, wsr_final_conv_sampler_step_multistep) against
float64 torch and against each other, the four architectures' DDIM / DPM-Solver++(2M) loops against the paper-form chains of
sampler_oracle.py, DDIM(eta = 1, S = T) against the DDPM loop, graph replay, repeatability, ensembles and ``sample.py --sampler``."""
import json
import os

import numpy as np
import pytest
import torch

import wsr
from conftest import ROOT, rel_l2
from oracle import nets
from oracle.cases import CASES, short_schedule
from oracle.weights import fill_module
from sampler_oracle import alphas_cumprod, ddim_chain, dpmpp2m_chain

pytestmark = pytest.mark.gpu

nat = wsr.pkg.native
dmod = wsr.sub("models.diffusion_models.diffusion")
member_key = dmod.member_key
DEV = "cuda:0"
TOL = {"fp32": 1e-5, "bf16": 2e-2}
SEED = 2026


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ms_tables(S, seed=5):
    """Random multistep tables [5][S]: c_prev = 0 on rows 0 and 1 (the final and a first-order step), non-zero on the others."""
    g = torch.Generator().manual_seed(seed)
    tab = torch.rand((5, S), generator=g) * 0.5 + 0.5
    tab[4] = torch.randn(S, generator=g) * 0.3
    tab[4, :2] = 0.0
    return tab.to(DEV).contiguous()


def _ms_ref(tab, t, x, eps, hist, clip):
    c = tab[:, t].double().cpu()
    x0 = c[0] * x.double() - c[1] * eps.double()
    if clip:
        x0 = x0.clamp(-1.0, 1.0)
    out = c[2] * x0 + c[3] * x.double()
    if c[4] != 0:
        out = out + c[4] * hist.double()
    return out, x0


# ---------------------------------------------------------------------------------------------------------------------
# 1.-2. wsr_sampler_step_multistep
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("edt", ["fp32", "bf16"])
@pytest.mark.parametrize("clip", [0, 1])
def test_sampler_step_multistep_vs_float64(clip, edt):
    S, n = 5, 4 * 1000 + 3                                       # n is not a multiple of 4
    g = torch.Generator().manual_seed(11)
    x = torch.randn(n, generator=g) * 2
    eps = torch.randn(n, generator=g)
    hist = torch.randn(n, generator=g)
    if edt == "bf16":
        eps = eps.to(torch.bfloat16)
    tab = _ms_tables(S)
    worst = 0.0
    for t in (3, 1, 0):                                          # c_prev != 0, c_prev = 0, final row
        t_dev = torch.tensor([t], dtype=torch.int32, device=DEV)
        xd, hd = x.to(DEV), hist.to(DEV)
        nat.call("wsr_sampler_step_multistep", xd.data_ptr(), eps.to(DEV).data_ptr(), nat.BF16 if edt == "bf16" else nat.F32, hd.data_ptr(),
                 tab.data_ptr(), S, t_dev.data_ptr(), clip, xd.data_ptr(), n, _stream())   # in place
        ref, ref_h = _ms_ref(tab, t, x, eps.float(), hist, clip)
        err = max(((xd.double().cpu() - ref).abs().max() / ref.abs().max()).item(),
                  ((hd.double().cpu() - ref_h).abs().max() / ref_h.abs().max()).item())
        worst = max(worst, err)
        assert int(t_dev.item()) == t
    print("\n[samplers] wsr_sampler_step_multistep clip=%d eps %s: max relative error %.2e" % (clip, edt, worst))
    assert worst < 1e-6, worst


def test_multistep_does_not_read_the_history_when_c_prev_is_zero():
    S, n = 5, 1023
    g = torch.Generator().manual_seed(12)
    x, eps = torch.randn(n, generator=g).to(DEV), torch.randn(n, generator=g).to(DEV)
    tab = _ms_tables(S)
    for t in (1, 0):                                             # c_prev = 0 on both rows
        hist = torch.full((n,), float("nan"), device=DEV)
        out = torch.empty_like(x)
        t_dev = torch.tensor([t], dtype=torch.int32, device=DEV)
        nat.call("wsr_sampler_step_multistep", x.data_ptr(), eps.data_ptr(), nat.F32, hist.data_ptr(), tab.data_ptr(), S, t_dev.data_ptr(),
                 1, out.data_ptr(), n, _stream())
        ref, ref_h = _ms_ref(tab, t, x.cpu(), eps.cpu(), torch.zeros(n), 1)
        assert torch.isfinite(out).all() and torch.isfinite(hist).all(), t
        assert (out.double().cpu() - ref).abs().max().item() < 1e-5
        assert (hist.double().cpu() - ref_h).abs().max().item() < 1e-6


# ---------------------------------------------------------------------------------------------------------------------
# 3.-4. wsr_final_conv_sampler_step_multistep
# ---------------------------------------------------------------------------------------------------------------------
def _head_inputs(B, H, W, Cin, Cout, groups=32, seed=17):
    g = torch.Generator(device=DEV).manual_seed(seed)
    feat = torch.randn((B, H, W, Cin), generator=g, device=DEV).to(torch.bfloat16).contiguous()
    stats = torch.zeros((B, 2 * Cin), dtype=torch.float64, device=DEV)
    nat.call("wsr_gn_stats", feat.data_ptr(), nat.BF16, B, H * W, Cin, Cin, stats.data_ptr(), 2 * Cin, _stream())
    gamma = 1 + 0.1 * torch.randn(Cin, generator=g, device=DEV)
    beta = 0.1 * torch.randn(Cin, generator=g, device=DEV)
    w32 = (0.05 * torch.randn((9, Cout, Cin), generator=g, device=DEV)).contiguous()
    wpk = torch.empty((Cin // 64) * 9 * 4 * 2 * 64, dtype=torch.bfloat16, device=DEV)
    nat.call("wsr_pack_head_weight", w32.data_ptr(), Cout, Cin, wpk.data_ptr(), _stream())
    bias = 0.1 * torch.randn(Cout, generator=g, device=DEV)
    x = torch.randn((B, Cout, H, W), generator=g, device=DEV)
    hist = torch.randn((B, Cout, H, W), generator=g, device=DEV)

    def head(eps_out, xs):
        return (feat.data_ptr(), Cin, B, H, W, Cin, stats.data_ptr(), 2 * Cin, gamma.data_ptr(), beta.data_ptr(), groups, 1e-5,
                wpk.data_ptr(), bias.data_ptr(), Cout, eps_out, xs)
    return head, x, hist


@pytest.mark.parametrize("shape", [(2, 8, 160, 64, 2), (3, 12, 128, 128, 4), (64, 128, 256, 64, 1)],
                         ids=["small", "cin128_cout4", "bench_b64"])
@pytest.mark.parametrize("clip", [0, 1])
def test_fused_multistep_head_matches_head_then_step(shape, clip):
    B, H, W, Cin, Cout = shape
    head, x, hist = _head_inputs(B, H, W, Cin, Cout)
    S = 5
    tab = _ms_tables(S)
    worst = 0.0
    for t in (3, 1, 0):
        t_dev = torch.tensor([t], dtype=torch.int32, device=DEV)
        # reference: the head with eps_out only, then the unfused multistep step
        eps = torch.empty_like(x)
        nat.call("wsr_final_conv_sampler_step", *head(eps.data_ptr(), 0), 0, 0, 0, tab.data_ptr(), S, t_dev.data_ptr(), clip, _stream())
        ref, ref_h = torch.empty_like(x), hist.clone()
        nat.call("wsr_sampler_step_multistep", x.data_ptr(), eps.data_ptr(), nat.F32, ref_h.data_ptr(), tab.data_ptr(), S, t_dev.data_ptr(),
                 clip, ref.data_ptr(), x.numel(), _stream())
        xs, hs, eps_f = x.clone(), hist.clone(), torch.empty_like(x)
        nat.call("wsr_final_conv_sampler_step_multistep", *head(eps_f.data_ptr(), xs.data_ptr()), hs.data_ptr(), tab.data_ptr(), S,
                 t_dev.data_ptr(), clip, _stream())
        assert torch.equal(eps_f, eps)
        err = max(((xs - ref).abs().max() / ref.abs().max()).item(), ((hs - ref_h).abs().max() / ref_h.abs().max()).item())
        worst = max(worst, err)
    del head
    print("\n[samplers] fused multistep head %s clip=%d vs head + step: max relative difference %.2e" % (shape, clip, worst))
    assert worst < 1e-6, worst                    # measured on B200: 0 (bit-identical) at all three shapes, clip 0 and 1


def test_fused_multistep_head_ignores_a_nan_history_when_c_prev_is_zero():
    head, x, _ = _head_inputs(2, 8, 160, 64, 2)
    tab = _ms_tables(5)
    for t in (1, 0):
        xs, hs = x.clone(), torch.full_like(x, float("nan"))
        t_dev = torch.tensor([t], dtype=torch.int32, device=DEV)
        nat.call("wsr_final_conv_sampler_step_multistep", *head(0, xs.data_ptr()), hs.data_ptr(), tab.data_ptr(), 5, t_dev.data_ptr(), 1,
                 _stream())
        assert torch.isfinite(xs).all() and torch.isfinite(hs).all(), t


def test_multistep_entries_reject_null_arguments():
    n = 64
    x, eps, hist = (torch.zeros(n, device=DEV) for _ in range(3))
    tab = _ms_tables(5)
    t_dev = torch.tensor([2], dtype=torch.int32, device=DEV)
    for hp, tp in ((0, tab.data_ptr()), (hist.data_ptr(), 0)):
        with pytest.raises(nat.WsrError):
            nat.call("wsr_sampler_step_multistep", x.data_ptr(), eps.data_ptr(), nat.F32, hp, tp, 5, t_dev.data_ptr(), 1, x.data_ptr(), n,
                     _stream())
    head, xs, hs = _head_inputs(2, 8, 160, 64, 2)
    for xp, hp, tp in ((xs.data_ptr(), 0, tab.data_ptr()), (xs.data_ptr(), hs.data_ptr(), 0), (0, hs.data_ptr(), tab.data_ptr())):
        with pytest.raises(nat.WsrError):
            nat.call("wsr_final_conv_sampler_step_multistep", *head(0, xp), hp, tp, 5, t_dev.data_ptr(), 1, _stream())


# ---------------------------------------------------------------------------------------------------------------------
# 5.-9. the reverse loops of the four architectures
# ---------------------------------------------------------------------------------------------------------------------
T_SHORT, S_SHORT = 8, 4


def _arch(arch, precision, T=T_SHORT):
    """(diffusion, x_in, oracle denoise(x, level), field added back or None) for the small CASES net of ``arch``."""
    spec = CASES["%s_chain_small" % arch]
    cfg = spec["cfg"]
    U = wsr.sub("models.diffusion_models.%s.unet" % arch).UNet

    def unet(prec):
        net = U(in_channel=cfg["in_channel"], out_channel=cfg["out_channel"], norm_groups=cfg["norm_groups"],
                inner_channel=cfg["inner_channel"], channel_mults=cfg["channel_mults"], attn_res=cfg["attn_res"],
                res_blocks=cfg["res_blocks"], dropout=cfg["dropout"], image_height=cfg["image_height"],
                image_width=cfg["image_width"], image_channels=cfg["image_channels"], precision=prec)
        return fill_module(net, spec["seed"]).to(DEV).eval()
    net = unet(precision)
    sd = {k: v.detach().cpu() for k, v in unet("fp32").state_dict().items()}
    mod = wsr.sub("models.diffusion_models.%s.%s_diffusion" % (arch, arch))
    D = {"resdiff": "ResDiffDiffusion", "sr3": "SR3Diffusion", "phydiff": "PhyDiffDiffusion", "srdiff": "SRDiffDiffusion"}[arch]
    diff = getattr(mod, D)(net, image_height=cfg["image_height"], image_width=cfg["image_width"], channels=cfg["image_channels"],
                           conditional=True).to(DEV)
    g = torch.Generator().manual_seed(7)
    B, C, H, W = 2, cfg["image_channels"], cfg["image_height"], cfg["image_width"]
    sr, lr = 0.5 * torch.randn((B, C, H, W), generator=g), 0.5 * torch.randn((B, C, H // 4, W // 4), generator=g)
    if arch == "srdiff":
        R = wsr.sub("models.rrdb_encoder.RRDBNet").RRDBNet
        diff.rrdb_encoder = fill_module(R(1, 1, 64, 17, 32, precision=precision), spec["seed"] + 1).to(DEV).eval()
        rsd = {k: v.detach().cpu() for k, v in fill_module(R(1, 1, 64, 17, 32), spec["seed"] + 1).state_dict().items()}
        with torch.no_grad():
            _, feas = nets.rrdb_net(rsd, lr)

        def denoise(x, level):
            return nets.srdiff_unet(sd, feas, x, level, cfg)
    else:
        fn = {"resdiff": nets.resdiff_unet, "sr3": nets.sr3_unet, "phydiff": nets.phydiff_unet}[arch]

        def denoise(x, level):
            return fn(sd, torch.cat([sr, x], dim=1), level, cfg)
    diff.set_new_noise_schedule(short_schedule(T), DEV)
    return diff, {"SR": sr.to(DEV), "LR": lr.to(DEV)}, denoise, (None if arch == "sr3" else sr.double())


def _loop_input(arch, x_in):
    return x_in if arch == "srdiff" else x_in["SR"]


ARCHS = ["resdiff", "srdiff", "sr3", "phydiff"]
SAMPLERS = {"ddim0": ("ddim", 0.0), "ddim05": ("ddim", 0.5), "dpmpp2m": ("dpmpp2m", None)}
_ORACLE = {}


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("sampler", list(SAMPLERS))
@pytest.mark.parametrize("arch", ARCHS)
def test_loop_vs_paper_form_chain(arch, sampler, precision):
    name, eta = SAMPLERS[sampler]
    diff, x_in, denoise, add = _arch(arch, precision)
    diff.set_sampler(name, S_SHORT, eta)
    shape = tuple(x_in["SR"].shape)
    noise = torch.randn((S_SHORT + 1,) + shape, generator=torch.Generator().manual_seed(31))
    if (arch, sampler) not in _ORACLE:                            # the float64 chain once per architecture and sampler
        abar = alphas_cumprod(short_schedule(T_SHORT))
        with torch.no_grad():
            ref = ddim_chain(denoise, abar, S_SHORT, noise, eta) if name == "ddim" else dpmpp2m_chain(denoise, abar, S_SHORT, noise)
        _ORACLE[arch, sampler] = ref if add is None else ref + add
    ref = _ORACLE[arch, sampler]
    errs = []
    for use_graph in (False, True):
        diff.use_cuda_graph = use_graph
        out = diff.p_sample_loop(_loop_input(arch, x_in), noise_chain=noise.to(DEV))
        errs.append(rel_l2(out.cpu(), ref))
    print("\n[samplers] %s %s-%d %s final-field rel-L2 vs float64 chain: eager %.3e graph %.3e" % (arch, sampler, S_SHORT, precision, *errs))
    assert max(errs) < TOL[precision], errs


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("arch", ARCHS)
def test_ddim_eta1_all_steps_matches_ddpm(arch, precision):
    """Same Philox noise (tag = counter = timestep); only the fp32 rounding of the folded tables differs."""
    diff, x_in, _, _ = _arch(arch, precision)
    ddpm = diff.p_sample_loop(_loop_input(arch, x_in), seed=SEED)
    diff.set_sampler("ddim", T_SHORT, 1.0)
    ddim = diff.p_sample_loop(_loop_input(arch, x_in), seed=SEED)
    err = rel_l2(ddim.cpu(), ddpm.cpu())
    print("\n[samplers] %s %s DDIM(eta=1, S=T) vs DDPM rel-L2 %.3e" % (arch, precision, err))
    assert err < TOL[precision], err


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_dpmpp2m_graph_replay_equals_eager_and_repeats(precision):
    diff, x_in, _, _ = _arch("resdiff", precision)
    diff.set_sampler("dpmpp2m", S_SHORT)
    diff.sample_seed = SEED
    outs = []
    for use_graph in (False, True, True):
        diff.use_cuda_graph = use_graph
        outs.append(diff.super_resolution(x_in).clone())
    assert torch.equal(outs[0], outs[1])                          # graph replay carries the history across steps
    assert torch.equal(outs[1], outs[2])                          # a second call starts from a fresh history
    diff.set_sampler("ddim", S_SHORT, 0.0)
    assert rel_l2(diff.super_resolution(x_in).cpu(), outs[0].cpu()) > 1e-4      # a different sampler


@pytest.mark.parametrize("sampler", ["ddim05", "dpmpp2m"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("arch", ["resdiff", "srdiff"])
def test_ensemble_members_match_independent_runs(arch, precision, sampler):
    name, eta = SAMPLERS[sampler]
    diff, x_in, _, _ = _arch(arch, precision)
    diff.set_sampler(name, S_SHORT, eta)
    ens = diff.super_resolution_ensemble(x_in, 3, seed=SEED)
    errs = [rel_l2(ens[m].cpu(), diff.p_sample_loop(_loop_input(arch, x_in), seed=member_key(SEED, m)).cpu()) for m in range(3)]
    print("\n[samplers] %s %s %s ensemble member rel-L2 vs independent runs: %s" % (arch, precision, sampler, " ".join("%.2e" % e for e in errs)))
    assert max(errs) < {"fp32": 1e-6, "bf16": 2e-2}[precision], errs
    assert rel_l2(ens[0].cpu(), ens[1].cpu()) > 1e-2


# ---------------------------------------------------------------------------------------------------------------------
# 10. sample.py --sampler
# ---------------------------------------------------------------------------------------------------------------------
def _config(tmp_path):
    cfgmod = wsr.sub("configs.config")
    opt = json.loads(cfgmod.strip_comments(open(os.path.join(ROOT, "configs_examples", "resdiff_eval_b200.json")).read()))
    opt["name"] = "t_samplers"
    opt["model"]["unet"].update(in_channel=5, attn_res=[4])
    opt["model"]["diffusion"].update(image_height=32, image_width=64)
    for ph in ("train", "val"):
        opt["model"]["beta_schedule"][ph]["n_timestep"] = T_SHORT
    opt["data"].update(batch_size=2, val_batch_size=2, height=32)
    for k in ("log", "tb_logger", "results", "checkpoint"):
        opt["path"][k] = str(tmp_path / k)
    p = tmp_path / "samplers.json"
    p.write_text(json.dumps(opt))
    return str(p)


def test_sample_py_sampler_flags(tmp_path):
    cfg = _config(tmp_path)
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        sample = wsr.sub("sample")
        torch.manual_seed(0)
        sample.main(["-c", cfg, "-o", str(tmp_path / "ddim"), "-gpu", "0", "--sampler", "ddim", "--steps", "4", "--seed", "77"])
        ddim = np.load(tmp_path / "ddim" / "sr.npy")
        assert ddim.shape == (2, 1, 32, 64) and np.isfinite(ddim).all()
        torch.manual_seed(0)
        sample.main(["-c", cfg, "-o", str(tmp_path / "plain"), "-gpu", "0", "--sampler", "dpmpp2m", "--steps", "4", "--seed", "77"])
        torch.manual_seed(0)
        sample.main(["-c", cfg, "-o", str(tmp_path / "ens"), "-gpu", "0", "--sampler", "dpmpp2m", "--steps", "4", "--ensemble", "3",
                     "--seed", "77"])
        ens = np.load(tmp_path / "ens" / "ensemble.npy")
        assert ens.shape == (3, 2, 1, 32, 64) and np.isfinite(ens).all()
        err = rel_l2(torch.from_numpy(ens[0]), torch.from_numpy(np.load(tmp_path / "plain" / "sr.npy")))
        print("\n[samplers] sample.py dpmpp2m ensemble member 0 vs the plain run rel-L2 %.2e" % err)
        assert err < 2e-2, err
        assert rel_l2(torch.from_numpy(ens[0]), torch.from_numpy(ens[1])) > 1e-2
        with pytest.raises(SystemExit):
            sample.main(["-c", cfg, "-o", str(tmp_path / "bad"), "-gpu", "0", "--sampler", "ddpm", "--steps", "4"])
    finally:
        os.chdir(cwd)
