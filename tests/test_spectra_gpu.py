"""Spectral and latitude-weighted scores on the GPU: wsr_zonal_spectra against float64 numpy (np.fft.rfft on the same fp32 inputs),
known answers, accumulation semantics and rejections; training.metrics.FieldScores against a numpy restatement, against
ValidationMetrics and on a bicubic baseline; ``train.py -p val --scores`` and ``sample.py --scores`` end to end."""
import json
import logging
import math
import os

import numpy as np
import pytest
import torch

import wsr
from conftest import ROOT

pytestmark = pytest.mark.gpu

nat = wsr.pkg.native
metrics = wsr.sub("training.metrics")
DEV = "cuda:0"


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _slots(W):
    return 3 * (W // 2 + 1) + 3


def _run(pred, target=None, scale=None, shift=None, acc=None):
    P, H, W = pred.shape
    if acc is None:
        acc = torch.zeros((P, H, _slots(W)), dtype=torch.float64, device=DEV)
    ptr = lambda t: 0 if t is None else t.data_ptr()          # noqa: E731
    nat.call("wsr_zonal_spectra", pred.data_ptr(), ptr(target), P, H, W, ptr(scale), ptr(shift), acc.data_ptr(), _stream())
    torch.cuda.synchronize()
    return acc


def _ref(pred, target=None, scale=None, shift=None):
    """float64 numpy restatement of the slots: rfft of the physical fields and of the error, row sums of the error."""
    p = pred.cpu().numpy().astype(np.float64)
    P, H, W = p.shape
    nb = W // 2 + 1
    sc = np.ones(P) if scale is None else scale.cpu().numpy().astype(np.float64)
    sh = np.zeros(P) if shift is None else shift.cpu().numpy().astype(np.float64)
    c = np.full(nb, 2.0)
    c[0] = c[-1] = 1.0

    def power(x):
        return c * np.abs(np.fft.rfft(x, axis=-1)) ** 2 / W ** 2

    out = np.zeros((P, H, _slots(W)))
    out[..., :nb] = power(sc[:, None, None] * p + sh[:, None, None])
    if target is not None:
        t = target.cpu().numpy().astype(np.float64)
        d = sc[:, None, None] * (p - t)
        out[..., nb:2 * nb] = power(sc[:, None, None] * t + sh[:, None, None])
        out[..., 2 * nb:3 * nb] = power(d)
        out[..., 3 * nb] = np.abs(d).sum(-1)
        out[..., 3 * nb + 1] = (d * d).sum(-1)
        out[..., 3 * nb + 2] = d.sum(-1)
    return out


def _check(got, ref, W, with_target):
    nb = W // 2 + 1
    for j in range(3 if with_target else 1):
        g, r = got[..., j * nb:(j + 1) * nb], ref[..., j * nb:(j + 1) * nb]
        total = r.sum(-1, keepdims=True)
        assert (np.abs(g - r) <= 1e-10 * total + 1e-300).all(), np.abs(g - r).max()
    if with_target:
        g, r = got[..., 3 * nb:], ref[..., 3 * nb:]
        scale = np.maximum(np.abs(r), r[..., :1])                  # sum d is measured against sum |d|
        assert (np.abs(g - r) <= 1e-12 * scale).all(), (np.abs(g - r) / scale).max()


def _fields(P, H, W, seed, offset=0.0):
    g = torch.Generator().manual_seed(seed)
    lon = torch.arange(W, dtype=torch.float64) * 2 * math.pi / W
    smooth = torch.cos(3 * lon)[None, None, :] + 0.5 * torch.sin(lon + 0.3)[None, None, :]
    x = smooth * torch.randn(P, H, 1, generator=g, dtype=torch.float64) + 0.2 * torch.randn(P, H, W, generator=g, dtype=torch.float64)
    return (x + offset).float().to(DEV)


# ---------------------------------------------------------------------------------------------------------------------
# 1. wsr_zonal_spectra against float64 numpy
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("H,W,P", [(128, 256, 3), (64, 128, 5), (32, 64, 8), (7, 6, 4)])
@pytest.mark.parametrize("with_target,with_scale,with_shift", [(True, True, True), (True, False, False), (False, True, True),
                                                               (False, False, False), (True, True, False)])
def test_zonal_spectra_vs_numpy(H, W, P, with_target, with_scale, with_shift):
    pred = _fields(P, H, W, 1)
    target = (pred + 0.3 * _fields(P, H, W, 2)).contiguous() if with_target else None
    scale = (torch.rand(P, generator=torch.Generator().manual_seed(3)) * 20 + 1).to(DEV) if with_scale else None
    shift = (torch.rand(P, generator=torch.Generator().manual_seed(4)) * 300 - 50).to(DEV) if with_shift else None
    got = _run(pred, target, scale, shift).cpu().numpy()
    ref = _ref(pred, target, scale, shift)
    _check(got, ref, W, with_target)
    if not with_target:
        assert (got[..., W // 2 + 1:] == 0).all()


# ---------------------------------------------------------------------------------------------------------------------
# 2. known answers
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("W,k0", [(256, 1), (256, 37), (256, 127), (64, 5)])
def test_pure_zonal_cosine(W, k0):
    H, a = 4, 2.5
    n = np.arange(W)
    rows = np.stack([a * np.cos(2 * np.pi * k0 * n / W + ph) for ph in (0.0, 0.7, 1.9, -2.4)])
    pred = torch.from_numpy(rows[None]).float().to(DEV)
    got = _run(pred).cpu().numpy()[0, :, :W // 2 + 1]
    assert np.allclose(got[:, k0], a * a / 2, rtol=1e-6, atol=0)
    other = np.delete(got, k0, axis=1)
    assert (other < 1e-12 * a * a).all(), other.max()


@pytest.mark.parametrize("W", [256, 6, 2048])
def test_parseval_per_row(W):
    pred, target = _fields(2, 3, W, 5, offset=1.5), _fields(2, 3, W, 6)
    got = _run(pred, target).cpu().numpy()
    nb = W // 2 + 1
    p, t = pred.cpu().numpy().astype(np.float64), target.cpu().numpy().astype(np.float64)
    for j, x in enumerate((p, t, p - t)):
        np.testing.assert_allclose(got[..., j * nb:(j + 1) * nb].sum(-1), (x * x).mean(-1), rtol=1e-12, atol=0)


# ---------------------------------------------------------------------------------------------------------------------
# 3. accumulation semantics
# ---------------------------------------------------------------------------------------------------------------------
def test_second_call_doubles_and_runs_are_bit_identical():
    pred, target = _fields(6, 32, 64, 7), _fields(6, 32, 64, 8)
    scale = torch.full((6,), 3.0, device=DEV)
    once = _run(pred, target, scale).clone()
    again = _run(pred, target, scale)
    assert torch.equal(once, again)
    _run(pred, target, scale, acc=again)
    assert torch.equal(again, 2 * once)


def test_null_target_leaves_the_other_slots_untouched():
    P, H, W = 3, 16, 64
    nb = W // 2 + 1
    pred = _fields(P, H, W, 9)
    acc = torch.full((P, H, _slots(W)), -7.25, dtype=torch.float64, device=DEV)
    _run(pred, None, acc=acc)
    got = acc.cpu().numpy()
    assert (got[..., nb:] == -7.25).all()
    ref = _ref(pred)[..., :nb] - 7.25
    assert np.abs(got[..., :nb] - ref).max() < 1e-10 * np.abs(ref).max()


@pytest.mark.parametrize("case", ["odd_W", "W_below_4", "W_above_2048", "planes_0", "H_0", "null_pred", "null_acc"])
def test_rejections_write_nothing(case):
    P, H, W = 2, 4, 8
    args = dict(P=P, H=H, W=W)
    if case == "odd_W":
        args["W"] = 7
    elif case == "W_below_4":
        args["W"] = 2
    elif case == "W_above_2048":
        args["W"] = 2050
    elif case == "planes_0":
        args["P"] = 0
    elif case == "H_0":
        args["H"] = 0
    pred = torch.ones(P * H * 2050, device=DEV)
    acc = torch.full((P * H * _slots(2050),), 3.5, dtype=torch.float64, device=DEV)
    before = acc.clone()
    with pytest.raises(nat.WsrError):
        nat.call("wsr_zonal_spectra", 0 if case == "null_pred" else pred.data_ptr(), pred.data_ptr(), args["P"], args["H"], args["W"], 0, 0,
                 0 if case == "null_acc" else acc.data_ptr(), _stream())
    torch.cuda.synchronize()
    assert torch.equal(acc, before)


# ---------------------------------------------------------------------------------------------------------------------
# 4. FieldScores
# ---------------------------------------------------------------------------------------------------------------------
def test_field_scores_vs_numpy_and_validation_metrics():
    B, C, H, W = 4, 3, 128, 256
    pred = _fields(B * C, H, W, 11).view(B, C, H, W)
    target = (pred + 0.4 * _fields(B * C, H, W, 12).view(B, C, H, W) + 0.05).contiguous()
    g = torch.Generator().manual_seed(13)
    std = (torch.rand(B, C, generator=g) * 10 + 1).to(DEV)
    mean = (torch.rand(B, C, generator=g) * 300).to(DEV)
    lat = metrics.equal_angle_latitudes(H)
    fs = metrics.FieldScores(DEV, lat)
    fs.update(pred[:2], target[:2], std[:2].reshape(-1), mean[:2].reshape(-1))
    fs.update(pred[2:], target[2:], std[2:], mean[2:])             # (B, C) statistics, as batch_statistics returns them
    out = fs.compute()
    assert out["fields"] == B and out["lr_width"] == W // 4

    p, t = pred.double().cpu().numpy(), target.double().cpu().numpy()
    s, m = std.double().cpu().numpy()[..., None, None], mean.double().cpu().numpy()[..., None, None]
    d = s * (p - t)
    w = np.cos(np.deg2rad(lat))
    w = w / w.mean()
    nb = W // 2 + 1
    c = np.full(nb, 2.0)
    c[0] = c[-1] = 1.0
    spec = lambda x: c * np.abs(np.fft.rfft(x, axis=-1)) ** 2 / W ** 2          # noqa: E731
    for ci, v in enumerate(out["variables"] + [out["overall"]]):
        sl = slice(None) if ci == C else slice(ci, ci + 1)
        dv = d[:, sl]
        assert v["rmse"] == pytest.approx(math.sqrt((dv ** 2).mean()), rel=1e-12)
        assert v["mae"] == pytest.approx(np.abs(dv).mean(), rel=1e-12)
        assert v["bias"] == pytest.approx(dv.mean(), rel=1e-10)
        assert v["rmse_w"] == pytest.approx(math.sqrt((w[:, None] * dv ** 2).mean()), rel=1e-12)
        assert v["mae_w"] == pytest.approx((w[:, None] * np.abs(dv)).mean(), rel=1e-12)
        assert v["bias_w"] == pytest.approx((w[:, None] * dv).mean(), rel=1e-10)
        for name, lo, hi in metrics.LAT_BANDS:
            rows = (np.abs(lat) >= lo) & (np.abs(lat) < hi)
            wr = np.cos(np.deg2rad(lat[rows]))[:, None]
            ps = (wr * spec(s[:, sl] * p[:, sl] + m[:, sl])[:, :, rows]).sum((0, 1, 2)) / (wr.sum() * dv.shape[0] * dv.shape[1])
            ts = (wr * spec(s[:, sl] * t[:, sl] + m[:, sl])[:, :, rows]).sum((0, 1, 2)) / (wr.sum() * dv.shape[0] * dv.shape[1])
            es = (wr * spec(dv)[:, :, rows]).sum((0, 1, 2)) / (wr.sum() * dv.shape[0] * dv.shape[1])
            b = v["bands"][name]
            assert b["rows"] == rows.sum()
            for key, ref in (("spectrum", ps), ("target_spectrum", ts), ("error_spectrum", es)):
                np.testing.assert_allclose(b[key], ref, rtol=0, atol=1e-10 * ref.sum())
            hi_k = np.arange(nb) > W // 8
            assert b["unresolved_power_ratio"] == pytest.approx(ps[hi_k].sum() / ts[hi_k].sum(), rel=1e-9)
            lsd = math.sqrt(np.mean((10 * np.log10(ps[1:] / ts[1:])) ** 2))
            assert b["lsd_db"] == pytest.approx(lsd, rel=1e-6)

    # the unweighted errors are those of ValidationMetrics on the same batch (fp32 partial sums there)
    vm = metrics.ValidationMetrics(metrics.create_metric_dict(DEV))
    vm.update(pred, target, scale=std.reshape(-1))
    vals = {k: float(x) for k, x in vm.compute_metrics().items()}
    o = out["overall"]
    assert o["rmse"] == pytest.approx(vals["RMSE"], rel=1e-5)
    assert o["mae"] == pytest.approx(vals["MAE"], rel=1e-5)
    assert o["bias"] == pytest.approx(vals["MR"], rel=1e-4, abs=1e-6 * o["mae"])


def test_bicubic_baseline_lacks_the_unresolved_scales():
    B, C, H, W = 4, 2, 128, 256
    g = torch.Generator().manual_seed(21)
    lon = torch.arange(W, dtype=torch.float64) * 2 * math.pi / W
    hr = (torch.cos(2 * lon)[None, None, None, :] * torch.randn(B, C, H, 1, generator=g, dtype=torch.float64)
          + 0.5 * torch.randn(B, C, H, W, generator=g, dtype=torch.float64)).float().to(DEV)
    lr = hr.view(B, C, H // 4, 4, W // 4, 4).mean((3, 5)).contiguous()
    up = torch.empty_like(hr)
    nat.call("wsr_bicubic_upsample", lr.data_ptr(), B * C, H // 4, W // 4, 4, up.data_ptr(), _stream())
    lat = metrics.equal_angle_latitudes(H)
    bic, same = metrics.FieldScores(DEV, lat, lr_width=W // 4), metrics.FieldScores(DEV, lat, lr_width=W // 4)
    bic.update(up, hr)
    same.update(hr, hr)
    rb = bic.compute()["overall"]["bands"]["global"]
    rs = same.compute()["overall"]["bands"]["global"]
    print("\n[spectra] bicubic unresolved_power_ratio %.4f lsd_db %.2f" % (rb["unresolved_power_ratio"], rb["lsd_db"]))
    assert rb["unresolved_power_ratio"] < 0.3
    assert rs["unresolved_power_ratio"] == 1.0 and rs["lsd_db"] == 0.0
    assert all(e == 0.0 for e in rs["error_spectrum"]) and same.compute()["overall"]["rmse_w"] == 0.0


# ---------------------------------------------------------------------------------------------------------------------
# 5. entry points
# ---------------------------------------------------------------------------------------------------------------------
def _config(tmp_path, arch="resdiff", in_channel=5, data=None):
    cfgmod = wsr.sub("configs.config")
    opt = json.loads(cfgmod.strip_comments(open(os.path.join(ROOT, "configs_examples", "resdiff_eval_b200.json")).read()))
    opt["name"] = "t_scores"
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
    p = tmp_path / "cfg.json"
    p.write_text(json.dumps(opt))
    return str(p)


def _check_section(sec, W=64):
    nb = W // 2 + 1
    for v in sec["variables"] + [sec["overall"]]:
        for k in ("rmse_w", "mae_w", "bias_w", "rmse", "mae", "bias"):
            assert math.isfinite(v[k]), k
        g = v["bands"]["global"]
        for k in ("spectrum", "target_spectrum", "error_spectrum", "ratio", "wavelength_km"):
            assert len(g[k]) == nb, k
        assert all(math.isfinite(x) for x in g["spectrum"] + g["target_spectrum"] + g["error_spectrum"])
        assert math.isfinite(g["lsd_db"]) and math.isfinite(g["unresolved_power_ratio"])
        assert set(v["bands"]) == {"global", "tropics", "midlatitudes"}


def test_train_val_scores(tmp_path, caplog):
    cfg = _config(tmp_path)
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        train = wsr.sub("train")
        with caplog.at_level(logging.INFO, logger="base"):
            plain = train.main(["-c", cfg, "-p", "val", "-gpu", "0"])
            lines_plain = [r.getMessage() for r in caplog.records if r.name == "base"]
            caplog.clear()
            scored = train.main(["-c", cfg, "-p", "val", "-gpu", "0", "--scores", str(tmp_path / "val_scores.json")])
            lines_scored = [r.getMessage() for r in caplog.records if r.name == "base" and "scores written" not in r.getMessage()]
        assert lines_plain == lines_scored
        for a, b in zip(plain, scored):
            assert {k: float(v) for k, v in a.items()} == {k: float(v) for k, v in b.items()}
        rep = json.load(open(tmp_path / "val_scores.json"))
        assert rep["units"] == "standardised" and rep["lat_source"] == "equal_angle"
        _check_section(rep["model"])
        _check_section(rep["bicubic"])
        assert rep["model"]["overall"]["rmse"] == pytest.approx(float(plain[0]["RMSE"]), rel=1e-5)
    finally:
        os.chdir(cwd)


def test_sample_scores_plain_and_ensemble(tmp_path):
    cfg = _config(tmp_path)
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        sample = wsr.sub("sample")
        sample.main(["-c", cfg, "-o", str(tmp_path / "plain"), "-gpu", "0", "--scores", "--sampler", "ddim", "--steps", "3"])
        rep = json.load(open(tmp_path / "plain" / "scores.json"))
        assert set(rep) >= {"units", "lat_source", "model", "bicubic"}
        _check_section(rep["model"])
        _check_section(rep["bicubic"])
        # synthetic HR = bicubic + 0.3 white noise: the bicubic field lacks the power above the input's wavenumbers
        assert rep["bicubic"]["overall"]["bands"]["global"]["unresolved_power_ratio"] < 1.0
        assert rep["model"]["fields"] == 2
        sample.main(["-c", cfg, "-o", str(tmp_path / "ens"), "-gpu", "0", "--scores", "--ensemble", "4", "--seed", "3"])
        rep = json.load(open(tmp_path / "ens" / "scores.json"))
        assert set(rep) >= {"members", "ensemble_mean", "bicubic"}
        assert rep["members"]["fields"] == 8 and rep["ensemble_mean"]["fields"] == 2
        for k in ("members", "ensemble_mean", "bicubic"):
            _check_section(rep[k])
        assert os.path.exists(tmp_path / "ens" / "ensemble_scores.json")
    finally:
        os.chdir(cwd)


def test_scores_on_the_store(tmp_path):
    from oracle import store
    root = store.write_store(str(tmp_path / "store"), variables=("t2m",), hours=24 * 40)
    cfg = _config(tmp_path, "sr3", 2, dict(dataroot=root, batch_size=4, val_batch_size=4, variables=["t2m"], months_subset=[1, 2],
                                           transform_groups={"winter": [1, 2]}, transformation="GlobalStandardScaling", num_workers=2,
                                           train_min_date="2000-01-01-00", train_max_date="2000-02-05-00",
                                           val_min_date="2000-02-05-00", val_max_date="2000-02-06-00"))
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        wsr.sub("train").main(["-c", cfg, "-p", "val", "-gpu", "0", "--scores", str(tmp_path / "val_scores.json")])
        wsr.sub("sample").main(["-c", cfg, "-o", str(tmp_path / "out"), "-gpu", "0", "--scores"])
        for path in (tmp_path / "val_scores.json", tmp_path / "out" / "scores.json"):
            rep = json.load(open(path))
            assert rep["units"] == "physical" and rep["lat_source"] == "store" and rep["variable_names"] == ["t2m"]
            _check_section(rep["bicubic"])
            # physical units: the target's mean power (k = 0) is that of a ~270 K field
            t0 = rep["bicubic"]["overall"]["bands"]["global"]["target_spectrum"][0]
            assert 150.0 ** 2 < t0 < 400.0 ** 2
    finally:
        os.chdir(cwd)
