"""Host side of the spectral and latitude-weighted scores (training.metrics.FieldScores): the reduction of the accumulators to the
scores dict, the row latitudes (equal-angle grid and store metadata) and the ``--scores`` flags of train.py and sample.py."""
import json
import math
import os

import numpy as np
import pytest

import wsr

metrics = wsr.sub("training.metrics")


def _acc(C, H, W, pred, target, err, sums):
    """(C, H, S) accumulators from per-(variable, row) spectra (broadcast to (C, H, W/2+1)) and row sums (C, H, 3)."""
    nb = W // 2 + 1
    a = np.zeros((C, H, 3 * nb + 3))
    a[:, :, :nb] = pred
    a[:, :, nb:2 * nb] = target
    a[:, :, 2 * nb:3 * nb] = err
    a[:, :, 3 * nb:] = sums
    return a


def test_equal_angle_latitudes_are_the_weatherbench_grid():
    lat = metrics.equal_angle_latitudes(128)
    assert lat[0] == -89.296875 and lat[-1] == 89.296875
    np.testing.assert_array_equal(np.diff(lat), np.full(127, 1.40625))
    np.testing.assert_array_equal(metrics.equal_angle_latitudes(32), -87.1875 + 5.625 * np.arange(32))
    np.testing.assert_array_equal(metrics.equal_angle_latitudes(2), [-45.0, 45.0])


def test_weighted_and_unweighted_errors():
    H, W, n = 4, 8, 3
    lat = np.array([-50.0, -20.0, 20.0, 70.0])
    sums = np.zeros((1, H, 3))
    sums[0, :, 0] = [1.0, 2.0, 3.0, 4.0]          # sum |d| per row
    sums[0, :, 1] = [4.0, 8.0, 12.0, 16.0]        # sum d^2
    sums[0, :, 2] = [-1.0, 0.5, 1.0, 2.0]         # sum d
    out = metrics.field_summary(_acc(1, H, W, 1.0, 1.0, 0.0, sums), lat, W, n)
    v = out["variables"][0]
    npix = n * H * W
    assert v["mae"] == pytest.approx(10.0 / npix, rel=1e-15)
    assert v["rmse"] == pytest.approx(math.sqrt(40.0 / npix), rel=1e-15)
    assert v["bias"] == pytest.approx(2.5 / npix, rel=1e-15)
    w = np.cos(np.deg2rad(lat))
    w = w / w.mean()
    assert v["mae_w"] == pytest.approx((w * sums[0, :, 0]).sum() / npix, rel=1e-14)
    assert v["rmse_w"] == pytest.approx(math.sqrt((w * sums[0, :, 1]).sum() / npix), rel=1e-14)
    assert v["bias_w"] == pytest.approx((w * sums[0, :, 2]).sum() / npix, rel=1e-14)
    g = v["bands"]["global"]
    assert g["rows"] == H and g["rmse_w"] == pytest.approx(v["rmse_w"], rel=1e-14)
    # tropics: rows 1 and 2 (equal weights); midlatitudes: row 0 only; row 3 (|lat| = 70) is in no band but global
    t = v["bands"]["tropics"]
    assert t["rows"] == 2 and t["mae_w"] == pytest.approx(5.0 / (2 * n * W), rel=1e-14)
    m = v["bands"]["midlatitudes"]
    assert m["rows"] == 1 and m["rmse_w"] == pytest.approx(math.sqrt(4.0 / (n * W)), rel=1e-14)
    assert m["mean_abs_lat"] == 50.0
    # overall = the variables pooled
    out2 = metrics.field_summary(np.concatenate([_acc(1, H, W, 1.0, 1.0, 0.0, sums)] * 2), lat, W, n)
    assert out2["overall"]["rmse"] == pytest.approx(v["rmse"], rel=1e-15)
    assert out2["overall"]["bias_w"] == pytest.approx(v["bias_w"], rel=1e-14)


def test_band_spectra_are_cos_weighted_means_and_empty_bands_are_none():
    H, W, n = 3, 16, 2
    lat = np.array([0.0, 10.0, 80.0])
    nb = W // 2 + 1
    pred = np.zeros((1, H, nb))
    pred[0, 0], pred[0, 1], pred[0, 2] = 1.0, 3.0, 100.0
    out = metrics.field_summary(_acc(1, H, W, pred, 2.0 * n, 0.5, 1.0), lat, W, n)
    b = out["variables"][0]["bands"]
    w0, w1 = 1.0, math.cos(math.radians(10.0))
    np.testing.assert_allclose(b["tropics"]["spectrum"], (w0 * 1.0 + w1 * 3.0) / ((w0 + w1) * n), rtol=1e-15)
    np.testing.assert_allclose(b["tropics"]["target_spectrum"], 2.0, rtol=1e-15)
    np.testing.assert_allclose(b["tropics"]["error_spectrum"], 0.5 / n, rtol=1e-15)
    assert b["midlatitudes"] is None
    assert len(b["global"]["spectrum"]) == nb and out["wavenumbers"] == list(range(nb))


def test_lsd_unresolved_ratio_and_wavelengths():
    H, W = 2, 64
    nb = W // 2 + 1
    lat = np.array([-20.0, 20.0])
    k = np.arange(nb)
    target = np.where(k == 0, 0.0, 1.0 / np.maximum(k, 1) ** 2)[None, None, :].repeat(H, 1)
    pred = target.copy()
    pred[..., k > 8] *= 0.25                          # -6.02 dB above the input's resolved range (lr_width 16 -> k > 8)
    out = metrics.field_summary(_acc(1, H, W, pred, target, 0.0, 0.0), lat, W, 1)
    assert out["lr_width"] == 16
    g = out["variables"][0]["bands"]["global"]
    assert g["unresolved_power_ratio"] == pytest.approx(0.25, rel=1e-14)
    n_low, n_high = 8, nb - 9                         # k = 1..8 exact, k = 9..32 at 10 log10(0.25)
    assert g["lsd_db"] == pytest.approx(math.sqrt(n_high * (10 * math.log10(0.25)) ** 2 / (n_low + n_high)), rel=1e-12)
    assert g["ratio"][0] is None and g["ratio"][1] == 1.0 and g["ratio"][20] == pytest.approx(0.25, rel=1e-15)
    assert g["wavelength_km"][0] is None
    assert g["mean_abs_lat"] == pytest.approx(20.0, rel=1e-15)
    circ = 2 * math.pi * 6371.0 * math.cos(math.radians(20.0))
    assert g["wavelength_km"][1] == pytest.approx(circ, rel=1e-14) and g["wavelength_km"][32] == pytest.approx(circ / 32, rel=1e-14)
    # an explicit lr_width moves the cut: k > 16 keeps only damped bins
    out = metrics.field_summary(_acc(1, H, W, pred, target, 0.0, 0.0), lat, W, 1, lr_width=32)
    assert out["variables"][0]["bands"]["global"]["unresolved_power_ratio"] == pytest.approx(0.25, rel=1e-14)
    # identical spectra: ratio exactly 1, lsd 0; a JSON round trip keeps every value
    same = metrics.field_summary(_acc(1, H, W, target, target, 0.0, 0.0), lat, W, 1)
    g = same["overall"]["bands"]["global"]
    assert g["unresolved_power_ratio"] == 1.0 and g["lsd_db"] == 0.0
    assert json.loads(json.dumps(same)) == same


def _meta_store(root, var, lat_values, H):
    base = os.path.join(root, "hr", var)
    os.makedirs(os.path.join(base, "meta"))
    os.makedirs(os.path.join(base, "samples"))
    coords = [{"name": "lon", "values": list(np.linspace(0, 360, 8, endpoint=False))}]
    if lat_values is not None:
        coords.insert(0, {"name": "lat", "values": list(lat_values)})
    meta = {"name": var, "time_variate": True, "dims": ["lat", "lon"], "shape": [H, 8], "coords": coords, "attrs": {}}
    with open(os.path.join(base, "meta", "metadata.json"), "w") as fh:
        json.dump(meta, fh)
    return root


def test_latitudes_from_the_store_metadata(tmp_path):
    lat = np.linspace(-80.0, 80.0, 5)
    root = _meta_store(str(tmp_path / "a"), "t2m", lat, 5)
    got, src = metrics.field_latitudes(root, "t2m", 5)
    assert src == "store"
    np.testing.assert_array_equal(got, lat)


@pytest.mark.parametrize("case", ["no_lat", "wrong_length", "other_variable", "not_a_store"])
def test_latitudes_fall_back_to_the_equal_angle_grid(tmp_path, case):
    root = str(tmp_path / "a")
    if case == "no_lat":
        _meta_store(root, "t2m", None, 5)
    elif case == "wrong_length":
        _meta_store(root, "t2m", np.linspace(-80.0, 80.0, 4), 5)
    elif case == "other_variable":
        _meta_store(root, "z500", np.linspace(-80.0, 80.0, 5), 5)
    else:
        root = "synthetic"
    got, src = metrics.field_latitudes(root, "t2m", 5)
    assert src == "equal_angle"
    np.testing.assert_array_equal(got, metrics.equal_angle_latitudes(5))


def test_field_scores_run_on_cuda_only():
    with pytest.raises(wsr.pkg.native.WsrError):
        metrics.FieldScores("cpu", metrics.equal_angle_latitudes(4))


def test_scores_flags(tmp_path):
    sample = wsr.sub("sample")
    assert sample.parse_args(["-c", "x.json", "-o", str(tmp_path)]).scores is False
    args = sample.parse_args(["-c", "x.json", "-o", str(tmp_path), "--scores", "--ensemble", "4", "--sampler", "ddim", "--steps", "5"])
    assert args.scores and args.ensemble == 4
    train = wsr.sub("train")
    assert train.parse_args(["-c", "x.json", "-p", "val"]).scores is None
    assert train.parse_args(["-c", "x.json", "-p", "val", "--scores", "s.json", "--ema"]).scores == "s.json"
    with pytest.raises(SystemExit):
        train.parse_args(["-c", "x.json", "-p", "train", "--scores", "s.json"])
