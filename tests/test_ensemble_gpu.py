"""Ensemble sampling on the GPU: the member-keyed sampler kernels against the plain ones (bit-identical slices),
wsr_ensemble_stats against float64 torch, ``super_resolution_ensemble`` against independent ``p_sample_loop`` runs per
architecture, its invariances (one member, member_offset splits, plan reuse), ``EnsembleScores`` against numpy and
``sample.py --ensemble``."""
import json
import os

import numpy as np
import pytest
import torch

import wsr
from conftest import ROOT, rel_l2
from oracle.cases import CASES, short_schedule
from oracle.weights import fill_module

pytestmark = pytest.mark.gpu

nat = wsr.pkg.native
dmod = wsr.sub("models.diffusion_models.diffusion")
member_key = dmod.member_key
DEV = "cuda:0"


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _keys(seed, n):
    return torch.tensor([member_key(seed, m) for m in range(n)], dtype=torch.int64, device=DEV)


# ---------------------------------------------------------------------------------------------------------------------
# 1. member-keyed kernels
# ---------------------------------------------------------------------------------------------------------------------
def test_randn_members_slices_match_plain_stream():
    per, R, seed = 2 * 1 * 6 * 10, 4, 1234
    keys = _keys(seed, R)
    out = torch.empty(R * per, device=DEV)
    nat.call("wsr_randn_members", out.data_ptr(), out.numel(), keys.data_ptr(), per, 0xFFFFFFFF, _stream())
    for m in range(R):
        ref = torch.empty(per, device=DEV)
        nat.call("wsr_randn", ref.data_ptr(), per, member_key(seed, m), 0xFFFFFFFF, _stream())
        assert torch.equal(out[m * per:(m + 1) * per], ref), m
    one = torch.empty(per, device=DEV)
    nat.call("wsr_randn_members", one.data_ptr(), per, keys.data_ptr(), per, 7, _stream())
    ref = torch.empty(per, device=DEV)
    nat.call("wsr_randn", ref.data_ptr(), per, seed, 7, _stream())
    assert torch.equal(one, ref)          # member 0 keeps the seed
    with pytest.raises(nat.WsrError):
        nat.call("wsr_randn_members", out.data_ptr(), out.numel(), keys.data_ptr(), per + 2, 0, _stream())


def _tables(T):
    g = torch.Generator().manual_seed(5)
    tab = torch.rand((5, T), generator=g) * 0.5 + 0.5
    tab[4] = -torch.rand(T, generator=g) * 4          # log-variances
    return tab.to(DEV).contiguous()


@pytest.mark.parametrize("clip", [0, 1])
@pytest.mark.parametrize("injected", [False, True])
def test_sampler_step_members_matches_plain_step(clip, injected):
    T, R, per, seed = 6, 3, 2 * 1 * 8 * 12, 99
    g = torch.Generator().manual_seed(11)
    x = (torch.randn(R * per, generator=g) * 2).to(DEV)
    eps = torch.randn(R * per, generator=g).to(DEV)
    z = torch.randn(R * per, generator=g).to(DEV) if injected else None
    tab = _tables(T)
    t_dev = torch.tensor([3], dtype=torch.int32, device=DEV)
    keys = _keys(seed, R)

    def plain(xs, es, zs, s):
        o = torch.empty_like(xs)
        nat.call("wsr_sampler_step", xs.data_ptr(), es.data_ptr(), nat.F32, 0 if zs is None else zs.data_ptr(), 0, s, tab.data_ptr(), T,
                 t_dev.data_ptr(), clip, o.data_ptr(), xs.numel(), _stream())
        return o

    def keyed(xs, es, zs, k, pm):
        o = torch.empty_like(xs)
        nat.call("wsr_sampler_step_members", xs.data_ptr(), es.data_ptr(), nat.F32, 0 if zs is None else zs.data_ptr(), 0, k.data_ptr(),
                 pm, tab.data_ptr(), T, t_dev.data_ptr(), clip, o.data_ptr(), xs.numel(), _stream())
        return o

    out = keyed(x, eps, z, keys, per)
    for m in range(R):
        sl = slice(m * per, (m + 1) * per)
        ref = plain(x[sl], eps[sl], None if z is None else z[sl], member_key(seed, m))
        assert torch.equal(out[sl], ref), m
    one = keyed(x[:per], eps[:per], None if z is None else z[:per], keys, per)
    assert torch.equal(one, plain(x[:per], eps[:per], None if z is None else z[:per], seed))
    with pytest.raises(nat.WsrError):
        keyed(x, eps, z, keys, per - 1)


@pytest.mark.parametrize("clip", [0, 1])
@pytest.mark.parametrize("injected", [False, True])
def test_final_conv_sampler_step_members_matches_plain_head(clip, injected):
    Bc, R, H, W, Cin, Cout, groups, T, seed = 2, 3, 8, 160, 64, 2, 32, 6, 4242
    B = Bc * R
    g = torch.Generator().manual_seed(17)
    feat = torch.randn((B, H, W, Cin), generator=g).to(DEV, torch.bfloat16).contiguous()
    stats = torch.zeros((B, 2 * Cin), dtype=torch.float64, device=DEV)
    nat.call("wsr_gn_stats", feat.data_ptr(), nat.BF16, B, H * W, Cin, Cin, stats.data_ptr(), 2 * Cin, _stream())
    gamma = (1 + 0.1 * torch.randn(Cin, generator=g)).to(DEV)
    beta = (0.1 * torch.randn(Cin, generator=g)).to(DEV)
    w32 = (0.05 * torch.randn((9, Cout, Cin), generator=g)).to(DEV).contiguous()
    wpk = torch.empty((Cin // 64) * 9 * 4 * 2 * 64, dtype=torch.bfloat16, device=DEV)
    nat.call("wsr_pack_head_weight", w32.data_ptr(), Cout, Cin, wpk.data_ptr(), _stream())
    bias = (0.1 * torch.randn(Cout, generator=g)).to(DEV)
    x0 = torch.randn((B, Cout, H, W), generator=g).to(DEV)
    z = torch.randn((B, Cout, H, W), generator=g).to(DEV) if injected else None
    tab = _tables(T)
    t_dev = torch.tensor([4], dtype=torch.int32, device=DEV)
    keys = _keys(seed, R)
    per = Bc * Cout * H * W

    def common(n, f, st, xs, zs):
        return (f.data_ptr(), Cin, n, H, W, Cin, st.data_ptr(), 2 * Cin, gamma.data_ptr(), beta.data_ptr(), groups, 1e-5,
                wpk.data_ptr(), bias.data_ptr(), Cout, 0, xs.data_ptr(), 0 if zs is None else zs.data_ptr(), 0)

    xs = x0.clone()
    nat.call("wsr_final_conv_sampler_step_members", *common(B, feat, stats, xs, z), keys.data_ptr(), per, tab.data_ptr(), T,
             t_dev.data_ptr(), clip, _stream())
    for m in range(R):
        sl = slice(m * Bc, (m + 1) * Bc)
        ref = x0[sl].clone()
        zs = None if z is None else z[sl].contiguous()
        nat.call("wsr_final_conv_sampler_step", *common(Bc, feat[sl], stats[sl], ref, zs), member_key(seed, m), tab.data_ptr(), T,
                 t_dev.data_ptr(), clip, _stream())
        assert torch.equal(xs[sl], ref), m
    one = x0[:Bc].clone()
    nat.call("wsr_final_conv_sampler_step_members", *common(Bc, feat[:Bc], stats[:Bc], one, None if z is None else z[:Bc].contiguous()),
             keys.data_ptr(), per, tab.data_ptr(), T, t_dev.data_ptr(), clip, _stream())
    assert torch.equal(one, xs[:Bc])
    with pytest.raises(nat.WsrError):
        nat.call("wsr_final_conv_sampler_step_members", *common(B, feat, stats, x0.clone(), z), keys.data_ptr(), per + 6, tab.data_ptr(),
                 T, t_dev.data_ptr(), clip, _stream())


# ---------------------------------------------------------------------------------------------------------------------
# 2. wsr_ensemble_stats against float64
# ---------------------------------------------------------------------------------------------------------------------
def _stats_ref(ens, y, s):
    """ens (N, P, HW), y (P, HW) or None, s (P,) or None -> mean, spread, acc (P, 5), hist (P, N+1), all float64 / int64.
    acc: s * mean_i |x_i - y|, s * sum_ij |x_i - x_j| (from the sorted members), s^2 (mean - y)^2, s^2 var (unbiased), s (mean - y)."""
    e = ens.double()
    N, P, _ = e.shape
    sd = torch.ones(P, dtype=torch.float64, device=e.device) if s is None else s.double()
    mean, var = e.mean(0), e.var(0, unbiased=True)
    srt = e.sort(0).values
    k = torch.arange(N, dtype=torch.float64, device=e.device).view(N, 1, 1)
    pw = 2 * ((2 * k - N + 1) * srt).sum(0)
    acc = torch.zeros((P, 5), dtype=torch.float64, device=e.device)
    acc[:, 3] = sd ** 2 * var.sum(-1)
    hist = torch.zeros((P, N + 1), dtype=torch.int64, device=e.device)
    if y is not None:
        yd = y.double()
        acc[:, 0] = sd * (e - yd).abs().mean(0).sum(-1)
        acc[:, 1] = sd * pw.sum(-1)
        acc[:, 2] = sd ** 2 * ((mean - yd) ** 2).sum(-1)
        acc[:, 4] = sd * (mean - yd).sum(-1)
        rank = (e < yd).sum(0)
        for p in range(P):
            hist[p] = torch.bincount(rank[p], minlength=N + 1)
    return mean, var.sqrt(), acc, hist, pw


def _stats_dev(ens, y, s, twice=False):
    N, P, HW = ens.shape
    mean = torch.empty((P, HW), device=DEV)
    spread = torch.empty((P, HW), device=DEV)
    acc = torch.zeros((P, 5), dtype=torch.float64, device=DEV)
    hist = torch.zeros((P, N + 1), dtype=torch.int64, device=DEV)
    for _ in range(2 if twice else 1):
        nat.call("wsr_ensemble_stats", ens.data_ptr(), N, P * HW, 0 if y is None else y.data_ptr(), P, HW, 0 if s is None else s.data_ptr(),
                 mean.data_ptr(), spread.data_ptr(), acc.data_ptr(), 0 if y is None else hist.data_ptr(), _stream())
    return mean, spread, acc, hist


def _check_acc(acc, ref, e, y, s):
    # q4 = sum(mean - y) cancels: its tolerance is taken relative to sum |mean - y|
    mag = ref.abs().clone()
    if y is not None:
        sd = torch.ones(e.shape[1], dtype=torch.float64, device=DEV) if s is None else s.double()
        mag[:, 4] = sd * (e.double().mean(0) - y.double()).abs().sum(-1)
    err = ((acc - ref).abs() / mag.clamp_min(1e-30)).max().item()
    return err


@pytest.mark.parametrize("N", [2, 3, 8, 33, 64, 256])
def test_ensemble_stats_vs_float64(N):
    P, HW = 3, 1000 + 37                          # not a multiple of any block size
    g = torch.Generator().manual_seed(N)
    ens = torch.randn((N, P, HW), generator=g).to(DEV)
    y = (torch.randn((P, HW), generator=g) * 1.3).to(DEV)
    s = torch.tensor([1.0, 21.26, 0.5], device=DEV)
    worst = 0.0
    for yy in (y, None):
        for ss in (None, s):
            mean, spread, acc, hist = _stats_dev(ens, yy, ss)
            rm, rs, racc, rh, _ = _stats_ref(ens, yy, ss)
            assert (mean.double() - rm).abs().max().item() < 1e-6
            assert ((spread.double() - rs).abs() / rs).max().item() < 1e-6
            if yy is None:
                assert torch.all(acc[:, [0, 1, 2, 4]] == 0)
                err = ((acc[:, 3] - racc[:, 3]).abs() / racc[:, 3]).max().item()
            else:
                err = _check_acc(acc, racc, ens, yy, ss)
                assert torch.equal(hist, rh)
            worst = max(worst, err)
    # accumulation: a second call adds the same sums
    _, _, acc2, hist2 = _stats_dev(ens, y, s, twice=True)
    _, _, racc, rh, _ = _stats_ref(ens, y, s)
    assert torch.equal(hist2, 2 * rh)
    worst = max(worst, _check_acc(acc2 / 2, racc, ens, y, s))
    print("\n[ensemble_stats] N=%d worst relative sum error %.2e" % (N, worst))
    assert worst < 1e-6, worst                    # measured 2.2e-16 .. 4.4e-16 on B200 (fp32 inputs, double sums)


@pytest.mark.parametrize("N", [3, 8, 33])
def test_ensemble_stats_ties_and_rank_convention(N):
    """Quantised members (many ties) and targets equal to a member: the rank counts members STRICTLY below the target, and the
    sorted-order pairwise term equals the O(N^2) sum of |x_i - x_j|."""
    P, HW = 2, 777
    g = torch.Generator().manual_seed(100 + N)
    ens = (torch.randint(-3, 4, (N, P, HW), generator=g).float() * 0.5).to(DEV)
    y = ens[1].clone()
    y[:, ::3] = 0.25                               # between levels on every third pixel
    mean, spread, acc, hist = _stats_dev(ens, y, None)
    rm, rs, racc, rh, pw = _stats_ref(ens, y, None)
    pair = (ens.double()[:, None] - ens.double()[None]).abs().sum((0, 1))
    assert torch.allclose(pw, pair, rtol=0, atol=1e-9)
    assert torch.equal(hist, rh)
    assert _check_acc(acc, racc, ens, y, None) < 1e-6
    assert (mean.double() - rm).abs().max().item() < 1e-6


def test_ensemble_stats_rejects_unsupported_member_counts():
    ens = torch.zeros((1, 1, 64), device=DEV)
    acc = torch.zeros(5, dtype=torch.float64, device=DEV)
    with pytest.raises(nat.WsrError):
        nat.call("wsr_ensemble_stats", ens.data_ptr(), 1, 64, 0, 1, 64, 0, 0, 0, acc.data_ptr(), 0, _stream())


# ---------------------------------------------------------------------------------------------------------------------
# 3.-4. super_resolution_ensemble
# ---------------------------------------------------------------------------------------------------------------------
TOL = {"fp32": 1e-6, "bf16": 2e-2}
SEED = 2026


def _arch_diffusion(arch, precision, T=4):
    name = {"resdiff": "resdiff_chain_small", "sr3": "sr3_chain_small", "phydiff": "phydiff_chain_small",
            "srdiff": "srdiff_chain_small"}[arch]
    spec = CASES[name]
    cfg = spec["cfg"]
    U = wsr.sub("models.diffusion_models.%s.unet" % arch).UNet
    net = U(in_channel=cfg["in_channel"], out_channel=cfg["out_channel"], norm_groups=cfg["norm_groups"],
            inner_channel=cfg["inner_channel"], channel_mults=cfg["channel_mults"], attn_res=cfg["attn_res"],
            res_blocks=cfg["res_blocks"], dropout=cfg["dropout"], image_height=cfg["image_height"],
            image_width=cfg["image_width"], image_channels=cfg["image_channels"], precision=precision)
    net = fill_module(net, spec["seed"]).to(DEV).eval()
    mod = wsr.sub("models.diffusion_models.%s.%s_diffusion" % (arch, arch))
    D = {"resdiff": "ResDiffDiffusion", "sr3": "SR3Diffusion", "phydiff": "PhyDiffDiffusion", "srdiff": "SRDiffDiffusion"}[arch]
    kw = dict(image_height=cfg["image_height"], image_width=cfg["image_width"], channels=cfg["image_channels"], conditional=True)
    diff = getattr(mod, D)(net, **kw).to(DEV)
    if arch == "srdiff":
        R = wsr.sub("models.rrdb_encoder.RRDBNet").RRDBNet
        diff.rrdb_encoder = fill_module(R(1, 1, 64, 17, 32, precision=precision), spec["seed"] + 1).to(DEV).eval()
    diff.set_new_noise_schedule(short_schedule(T), DEV)
    g = torch.Generator().manual_seed(7)
    B, C, H, W = 2, cfg["image_channels"], cfg["image_height"], cfg["image_width"]
    x_in = {"SR": (0.5 * torch.randn((B, C, H, W), generator=g)).to(DEV),
            "LR": (0.5 * torch.randn((B, C, H // 4, W // 4), generator=g)).to(DEV)}
    return diff, x_in


def _independent(diff, arch, x_in, seed):
    return diff.p_sample_loop(x_in if arch == "srdiff" else x_in["SR"], seed=seed)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("arch", ["resdiff", "srdiff", "sr3", "phydiff"])
def test_ensemble_members_match_independent_runs(arch, precision):
    diff, x_in = _arch_diffusion(arch, precision)
    ens = diff.super_resolution_ensemble(x_in, 3, seed=SEED)
    assert tuple(ens.shape) == (3,) + tuple(x_in["SR"].shape)
    errs = []
    for m in range(3):
        ref = _independent(diff, arch, x_in, member_key(SEED, m))
        errs.append(rel_l2(ens[m].cpu(), ref.cpu()))
    print("\n[ensemble] %s %s member rel-L2 vs independent runs: %s" % (arch, precision, " ".join("%.2e" % e for e in errs)))
    assert max(errs) < TOL[precision], errs        # measured on B200: 0 (bit-identical) for all four, fp32 and bf16
    assert rel_l2(ens[0].cpu(), ens[1].cpu()) > 1e-2           # members differ


def test_resdiff_members_see_their_own_fd_group():
    """The FD splitter's 4-D FFT couples the batch: with repeats, lf / hf of every member slice equal those of the B conditions alone,
    and the ensemble is NOT what a plan conditioned on the FFT of the stacked 3 x B batch samples."""
    diff, x_in = _arch_diffusion("resdiff", "fp32")
    sr = x_in["SR"]
    B = sr.shape[0]
    single = diff._plan(B, DEV)
    single.set_condition(sr)
    lf1, hf1 = single.lf.clone(), single.hf.clone()
    plan = diff._plan(3 * B, DEV)
    plan.set_condition(sr, repeats=3)
    for m in range(3):
        assert torch.equal(plan.lf[m * B:(m + 1) * B], lf1) and torch.equal(plan.hf[m * B:(m + 1) * B], hf1)
    ens = diff.super_resolution_ensemble(x_in, 3, seed=SEED)
    plan.set_condition(sr.repeat(3, 1, 1, 1))             # the stacked FFT
    stacked_hf = rel_l2(plan.hf[:B].cpu(), hf1.cpu())
    img = diff._reverse_loop(plan, (3 * B,) + tuple(sr.shape[1:]), member_keys=_keys(SEED, 3))
    stacked = (img.view((3,) + tuple(sr.shape)) + sr.unsqueeze(0)).clone()
    d = rel_l2(stacked.cpu(), ens.cpu())
    print("\n[ensemble] resdiff stacked-FFT hf rel diff %.3e, stacked vs grouped ensemble rel-L2 %.3e" % (stacked_hf, d))
    assert d > 1e-4, d                             # measured on B200: 1.2e-1 (hf of the stacked FFT: 7.0e-2 off)


def test_ensemble_invariances_bf16():
    diff, x_in = _arch_diffusion("resdiff", "bf16")
    # one member is the plain super_resolution with the same seed, bit for bit
    diff.sample_seed = SEED
    sr = diff.super_resolution(x_in)
    one = diff.super_resolution_ensemble(x_in, 1, seed=SEED)
    assert torch.equal(one[0], sr)
    # chunks of 2 members (max_images = 2 * B): one call == two member_offset calls, and plan reuse == fresh plans
    whole = diff.super_resolution_ensemble(x_in, 4, seed=SEED, max_images=4)
    parts = torch.cat([diff.super_resolution_ensemble(x_in, 2, seed=SEED, member_offset=o, max_images=4) for o in (0, 2)], 0)
    assert torch.equal(whole, parts)
    fresh = []
    for o in (0, 2):
        diff.denoise_fn._plans.clear()
        fresh.append(diff.super_resolution_ensemble(x_in, 2, seed=SEED, member_offset=o, max_images=4))
    assert torch.equal(whole, torch.cat(fresh, 0))


# ---------------------------------------------------------------------------------------------------------------------
# 5. EnsembleScores
# ---------------------------------------------------------------------------------------------------------------------
def _scores_np(ens, y, std):
    e = ens.astype(np.float64) * std[None, None, :, None, None]
    t = y.astype(np.float64) * std[None, :, None, None]
    N = e.shape[0]
    out = {}
    for c in list(range(e.shape[2])) + ["all"]:
        ec = e[:, :, c] if c != "all" else np.moveaxis(e, 2, 1).reshape(N, -1)
        tc = t[:, c] if c != "all" else np.moveaxis(t, 1, 0).reshape(-1)
        ec = ec.reshape(N, -1)
        tc = tc.reshape(-1)
        n = tc.size
        ae = np.abs(ec - tc[None]).mean(0).sum()
        pair = np.abs(ec[:, None] - ec[None]).sum((0, 1)).sum()
        mean = ec.mean(0)
        rmse = np.sqrt(((mean - tc) ** 2).sum() / n)
        spread = np.sqrt(ec.var(0, ddof=1).sum() / n)
        hist = np.bincount((ec < tc[None]).sum(0), minlength=N + 1)
        out[c] = dict(crps=ae / n - pair / (2 * N * N * n), crps_fair=ae / n - pair / (2 * N * (N - 1) * n), rmse=rmse, spread=spread,
                      spread_skill=np.sqrt((N + 1) / N) * spread / rmse, rank_hist=hist / hist.sum())
    return out


def test_ensemble_scores_vs_numpy():
    Sc = wsr.sub("training.metrics").EnsembleScores
    g = np.random.default_rng(3)
    N, B, C, H, W = 6, 2, 3, 16, 24
    ens = g.standard_normal((N, B, C, H, W)).astype(np.float32)
    y = (g.standard_normal((B, C, H, W)) * 1.2).astype(np.float32)
    std = np.array([21.26, 3.5, 0.8])
    sc = Sc(DEV)
    # two updates over halves of the batch = one update over all of it
    for b in range(B):
        sc.update(torch.from_numpy(ens[:, b:b + 1]).to(DEV), torch.from_numpy(y[b:b + 1]).to(DEV), torch.tensor(std, device=DEV))
    got = sc.compute()
    ref = _scores_np(ens, y, std)
    for k in ("crps", "crps_fair", "rmse", "spread", "spread_skill"):
        np.testing.assert_allclose(got[k], [ref[c][k] for c in range(C)], rtol=1e-6)
        np.testing.assert_allclose(got["overall"][k], ref["all"][k], rtol=1e-6)
    for c in range(C):
        np.testing.assert_allclose(got["rank_hist"][c], ref[c]["rank_hist"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(got["overall"]["rank_hist"], ref["all"]["rank_hist"], rtol=0, atol=1e-12)


# ---------------------------------------------------------------------------------------------------------------------
# 6. sample.py --ensemble
# ---------------------------------------------------------------------------------------------------------------------
def _config(tmp_path, arch="resdiff", in_channel=5, data=None):
    cfgmod = wsr.sub("configs.config")
    opt = json.loads(cfgmod.strip_comments(open(os.path.join(ROOT, "configs_examples", "resdiff_eval_b200.json")).read()))
    opt["name"] = "t_ens"
    opt["model"]["architecture"] = arch
    opt["model"]["unet"].update(in_channel=in_channel, attn_res=[4])
    opt["model"]["diffusion"].update(image_height=32, image_width=64)
    for ph in ("train", "val"):
        opt["model"]["beta_schedule"][ph]["n_timestep"] = 4
    opt["data"].update(batch_size=2, val_batch_size=2, height=32)
    if data:
        opt["data"].update(data)
    for k in ("log", "tb_logger", "results", "checkpoint"):
        opt["path"][k] = str(tmp_path / k)
    p = tmp_path / "ens.json"
    p.write_text(json.dumps(opt))
    return str(p)


def test_sample_ensemble_entry_point(tmp_path):
    cfg = _config(tmp_path)
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        sample = wsr.sub("sample")
        # the two runs build their random-init weights from torch's global generator: same state, same model
        torch.manual_seed(0)
        sample.main(["-c", cfg, "-o", str(tmp_path / "plain"), "-gpu", "0", "--seed", "77"])
        torch.manual_seed(0)
        sample.main(["-c", cfg, "-o", str(tmp_path / "ens"), "-gpu", "0", "--ensemble", "3", "--seed", "77"])
        ens = np.load(tmp_path / "ens" / "ensemble.npy")
        sr = np.load(tmp_path / "plain" / "sr.npy")
        assert ens.shape == (3, 2, 1, 32, 64) and np.isfinite(ens).all()
        assert np.load(tmp_path / "ens" / "ensemble_mean.npy").shape == (2, 1, 32, 64)
        assert np.load(tmp_path / "ens" / "ensemble_spread.npy").shape == (2, 1, 32, 64)
        # member 0 is the plain run with the same seed (batch 6 vs batch 2 on the bf16 path: measured rel-L2 0, bit-identical, on B200)
        err = rel_l2(torch.from_numpy(ens[0]), torch.from_numpy(sr))
        print("\n[ensemble] sample.py member 0 vs sr.npy rel-L2 %.2e" % err)
        assert err < 2e-2, err
        scores = json.load(open(tmp_path / "ens" / "ensemble_scores.json"))
        assert scores["members"] == 3 and len(scores["overall"]["rank_hist"]) == 4
    finally:
        os.chdir(cwd)


def test_sample_ensemble_on_the_store(tmp_path):
    from oracle import store
    root = store.write_store(str(tmp_path / "store"), variables=("t2m",), hours=24 * 40)
    cfg = _config(tmp_path, "sr3", 2, dict(dataroot=root, batch_size=4, val_batch_size=4, variables=["t2m"], months_subset=[1, 2],
                                           transform_groups={"winter": [1, 2]}, transformation="GlobalStandardScaling", num_workers=2,
                                           train_min_date="2000-01-01-00", train_max_date="2000-02-05-00",
                                           val_min_date="2000-02-05-00", val_max_date="2000-02-06-00"))
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        wsr.sub("sample").main(["-c", cfg, "-o", str(tmp_path / "out"), "-gpu", "0", "--ensemble", "3", "--seed", "5"])
        out = tmp_path / "out"
        ens, phys = np.load(out / "ensemble.npy"), np.load(out / "ensemble_physical.npy")
        assert ens.shape == phys.shape and ens.shape[0] == 3 and np.isfinite(phys).all()
        assert 150.0 < phys.mean() < 400.0
        scores = json.load(open(out / "ensemble_scores.json"))
        assert scores["overall"]["rmse"] > 0 and abs(sum(scores["overall"]["rank_hist"]) - 1) < 1e-9
    finally:
        os.chdir(cwd)
