"""Validation metric accumulators of the reference (training/metrics.py:30-201: MAE, MSE, RMSE, MR; containers :300-365) on
the device.  ``update`` is one ``wsr_error_sums`` launch per metric object -- or ONE launch for all four through
``ErrorSums`` / ``ValidationMetrics`` -- with double accumulators on the device and no host synchronisation until ``compute``.
``update(predicted, target, scale=std)`` folds the inverse StandardScaling into the same pass (the means cancel in the
difference), so RMSE in Kelvin never needs the de-normalised tensors.  PSNR / SSIM (torcheval / skimage wrappers in the
reference) are outside the accelerated path.

``FieldScores`` adds what a weather user asks of a downscaler beyond those four numbers: zonal power spectra of the output, the target
and the error per latitude band (does the model synthesise the scales the low-resolution input lacks?) and errors weighted by
cos(latitude) (error per unit area on the equal-angle grid)."""
import math
import os
from abc import ABC, abstractmethod

import numpy as np
import torch

from .. import _native as nat


class ErrorSums:
    """Device accumulators (sum |d|, sum d^2, sum d) and the element count."""

    def __init__(self, device=None):
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.type != "cuda":
            raise nat.WsrError("metric accumulators run on the CUDA path only (got device %s)" % self.device)
        self.reset()

    def reset(self):
        self.acc = torch.zeros(3, dtype=torch.float64, device=self.device)
        self.count = 0

    def update(self, predicted, target, scale=None):
        p = predicted.to(device=self.device, dtype=torch.float32).contiguous()
        t = target.to(device=self.device, dtype=torch.float32).contiguous()
        assert p.shape == t.shape
        if scale is not None:
            sc = scale.to(device=self.device, dtype=torch.float32).contiguous()
            planes = sc.numel()
            assert p.numel() % planes == 0
            hw = p.numel() // planes
            sp = sc.data_ptr()
            self._keep = sc
        else:
            planes, hw, sp = 1, p.numel(), 0
        nat.call("wsr_error_sums", p.data_ptr(), t.data_ptr(), planes, hw, sp, self.acc.data_ptr(),
                 torch.cuda.current_stream(self.device).cuda_stream)
        self.count += p.numel()


class Metric(ABC):
    """Same interface as the reference's Metric (:30-72): reset / update(predicted, target) / compute."""
    _shared = None

    def __init__(self, device=None, sums=None):
        self.device = device
        self._sums = sums if sums is not None else ErrorSums(device)
        self._own = sums is None

    def reset(self):
        self._sums.reset()

    def update(self, predicted, target, scale=None):
        if self._own:
            self._sums.update(predicted, target, scale)

    @property
    def count(self):
        return self._sums.count

    @abstractmethod
    def compute(self):
        pass


class MAE(Metric):
    def compute(self):
        return 0.0 if self.count == 0 else (self._sums.acc[0] / self.count).to(torch.float32)


class MSE(Metric):
    def compute(self):
        return 0.0 if self.count == 0 else (self._sums.acc[1] / self.count).to(torch.float32)


class RMSE(Metric):
    def compute(self):
        return 0.0 if self.count == 0 else torch.sqrt(self._sums.acc[1] / self.count).to(torch.float32)


class MR(Metric):
    def compute(self):
        return 0.0 if self.count == 0 else (self._sums.acc[2] / self.count).to(torch.float32)


def create_metric_dict(torch_device=None):
    """The reference's dictionary (:478-492) restricted to the four error metrics; they share ONE accumulator set."""
    sums = ErrorSums(torch_device)
    return {"MSE": MSE(torch_device, sums), "RMSE": RMSE(torch_device, sums), "MAE": MAE(torch_device, sums), "MR": MR(torch_device, sums),
            "_sums": sums}


class ValidationMetrics:
    """Container with the reference's interface (:300-365): reset / update / compute_metrics / metrics2dict / metrics2str."""

    def __init__(self, metrics_dict):
        self._sums = metrics_dict.get("_sums")
        self.metrics_objects = {k: v for k, v in metrics_dict.items() if k != "_sums"}
        self.metrics = {}
        self.reset()

    def reset(self):
        if self._sums is not None:
            self._sums.reset()
        for m in self.metrics_objects.values():
            if m._own:
                m.reset()

    def update(self, predicted, target, scale=None):
        if self._sums is not None:
            self._sums.update(predicted, target, scale)
        for m in self.metrics_objects.values():
            m.update(predicted, target, scale)

    def compute_metrics(self):
        self.metrics = {name: m.compute() for name, m in self.metrics_objects.items()}
        return self.metrics

    def metrics2dict(self):
        return self.metrics

    def metrics2str(self):
        message = ""
        for metric, value in self.metrics.items():
            message = f"{message}  |  {metric:s}: {float(value):.5f}"
        return message


class EnsembleScores:
    """Probabilistic scores of ensembles against their targets: per-plane double accumulators and rank histograms on the device,
    filled by one ``wsr_ensemble_stats`` launch per ``update``; the host synchronises only in ``compute``.

    ``update(ensemble, target, scale=None)``: ensemble (N, B, C, H, W), target (B, C, H, W); ``scale`` = std per variable (C values) or
    per plane (B * C values) puts every score in physical units (the inverse StandardScaling; the means cancel in differences).
    ``compute()`` returns, per variable (lists of C values) and over all variables ("overall"): CRPS (standard, 1/(2N^2) pairwise
    term) and fair CRPS (1/(2N(N-1))), the RMSE of the ensemble mean, the mean spread sqrt(mean unbiased variance), the spread-skill
    ratio sqrt((N+1)/N) * spread / RMSE and the rank histogram normalised to sum 1 (rank = members strictly below the target)."""

    def __init__(self, device=None):
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.type != "cuda":
            raise nat.WsrError("metric accumulators run on the CUDA path only (got device %s)" % self.device)
        self.reset()

    def reset(self):
        self.N = self.C = None
        self.acc = self.hist = None
        self.pixels = 0              # pixels per variable seen so far

    def update(self, ensemble, target, scale=None):
        ens = ensemble.to(device=self.device, dtype=torch.float32).contiguous()
        tgt = target.to(device=self.device, dtype=torch.float32).contiguous()
        N, B, C, H, W = ens.shape
        assert tuple(tgt.shape) == (B, C, H, W), (tuple(ens.shape), tuple(tgt.shape))
        if self.N is None:
            self.N, self.C = N, C
            self.acc = torch.zeros((C, 5), dtype=torch.float64, device=self.device)
            self.hist = torch.zeros((C, N + 1), dtype=torch.int64, device=self.device)
        assert (N, C) == (self.N, self.C), "every update of one EnsembleScores needs the same member and variable count"
        planes = B * C
        sp = 0
        if scale is not None:
            sc = scale.to(device=self.device, dtype=torch.float32).reshape(-1)
            if sc.numel() == C:
                sc = sc.repeat(B)
            assert sc.numel() == planes
            sc = sc.contiguous()
            sp = sc.data_ptr()
        acc = torch.zeros((planes, 5), dtype=torch.float64, device=self.device)
        hist = torch.zeros((planes, N + 1), dtype=torch.int64, device=self.device)
        nat.call("wsr_ensemble_stats", ens.data_ptr(), N, planes * H * W, tgt.data_ptr(), planes, H * W, sp, 0, 0, acc.data_ptr(),
                 hist.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream)
        self.acc += acc.view(B, C, 5).sum(0)
        self.hist += hist.view(B, C, N + 1).sum(0)
        self.pixels += B * H * W
        self._keep = (ens, tgt, sc if scale is not None else None, acc, hist)

    def compute(self):
        if self.N is None or self.pixels == 0:
            return {}
        N = self.N
        acc = self.acc.cpu().double()
        hist = self.hist.cpu().double()

        def scores(a, h, n):
            crps = a[0] / n - a[1] / (2.0 * N * N * n)
            fair = a[0] / n - a[1] / (2.0 * N * (N - 1) * n)
            rmse = float(torch.sqrt(a[2] / n))
            spread = float(torch.sqrt(a[3] / n))
            return {"crps": float(crps), "crps_fair": float(fair), "rmse": rmse, "spread": spread,
                    "spread_skill": (((N + 1) / N) ** 0.5) * spread / rmse if rmse > 0 else float("inf"),
                    "rank_hist": (h / h.sum()).tolist()}

        per = [scores(acc[c], hist[c], self.pixels) for c in range(self.C)]
        out = {k: [p[k] for p in per] for k in per[0]}
        out["overall"] = scores(acc.sum(0), hist.sum(0), self.pixels * self.C)
        out["members"] = N
        return out


EARTH_RADIUS_KM = 6371.0
# latitude bands of FieldScores: name -> |lat| range [lo, hi) in degrees
LAT_BANDS = (("global", 0.0, math.inf), ("tropics", 0.0, 30.0), ("midlatitudes", 30.0, 60.0))


def equal_angle_latitudes(H):
    """Cell-centre latitudes (degrees, south to north) of an equal-angle grid with H rows: -90 + (i + 0.5) * 180 / H.  For H = 128 this
    is the WeatherBench 1.40625 degree grid, -89.296875 .. 89.296875."""
    return -90.0 + (np.arange(H, dtype=np.float64) + 0.5) * 180.0 / H


def field_latitudes(dataroot, variable, H):
    """(latitudes in degrees, source) of the H rows of ``variable``'s high-resolution fields: the ``lat`` coordinate of the store's
    ``hr/<variable>/meta/metadata.json`` when it exists and has H values (source "store"), else the equal-angle cell centres
    (source "equal_angle")."""
    path = os.path.join(str(dataroot or ""), "hr", str(variable or ""))
    if dataroot and variable and os.path.isdir(path):
        from ..data.npy_reader import WNPYReader
        meta = WNPYReader(path, sample_index=[]).meta_data          # metadata only: no scan of the sample files
        for c in meta.get("coords", []):
            values = np.asarray(c.get("values", []), dtype=np.float64).reshape(-1)
            if c.get("name") == "lat" and values.size == H:
                return values, "store"
    return equal_angle_latitudes(H), "equal_angle"


def field_summary(acc, lat_deg, W, fields, lr_width=None):
    """The JSON-ready scores of ``FieldScores`` from its accumulators (a pure function of its arguments).

    acc: (C, H, S) float64, S = 3 (W/2 + 1) + 3, the wsr_zonal_spectra slots of each (variable, row) summed over ``fields`` fields:
    spectra of the prediction, the target and the error, then sum |d|, sum d^2, sum d over the row.  lat_deg: the H row latitudes.
    Rows are weighted by w_r = cos(lat_r) normalised to mean 1 over the rows.  Per variable (list ``variables``) and over all variables
    (``overall``): rmse_w / mae_w / bias_w (cos-weighted), rmse / mae / bias (unweighted, as ValidationMetrics), and per latitude band
    (``bands``: global, tropics |lat| < 30, midlatitudes 30 <= |lat| < 60; None for a band without rows):
      spectrum, target_spectrum, error_spectrum  cos-weighted mean one-sided power per wavenumber k = 0 .. W/2 (sum over k = mean square)
      ratio                                      spectrum / target_spectrum (None where the target has no power)
      lsd_db                                     log-spectral distance sqrt(mean_k (10 log10(P_k / T_k))^2) over k >= 1 with P_k, T_k > 0
      unresolved_power_ratio                     sum P_k / sum T_k over k > lr_width / 2 (the scales the low-resolution input lacks)
      wavelength_km                              2 pi R cos(phi) / k, R = 6371 km, phi the band's weighted mean |lat| (None at k = 0)
    lr_width: width of the low-resolution input (default W / 4)."""
    acc = np.asarray(acc, dtype=np.float64)
    C, H, S = acc.shape
    nb = W // 2 + 1
    assert S == 3 * nb + 3, (S, W)
    lat = np.asarray(lat_deg, dtype=np.float64).reshape(-1)
    assert lat.size == H, (lat.size, H)
    lr_width = W // 4 if lr_width is None else int(lr_width)
    w = np.cos(np.deg2rad(lat))
    w = w / w.mean()
    k = np.arange(nb)
    unresolved = k > lr_width / 2.0

    def errors(a, wr, n, suffix):
        den = wr.sum() * n * W
        return {"rmse" + suffix: math.sqrt(float((wr * a[:, 3 * nb + 1]).sum() / den)),
                "mae" + suffix: float((wr * a[:, 3 * nb]).sum() / den), "bias" + suffix: float((wr * a[:, 3 * nb + 2]).sum() / den)}

    def band(a, n, lo, hi):
        m = (np.abs(lat) >= lo) & (np.abs(lat) < hi)
        if not m.any():
            return None
        wm = w[m]
        p, t, e = ((wm[:, None] * a[m][:, j * nb:(j + 1) * nb]).sum(0) / (wm.sum() * n) for j in range(3))
        pos = (k >= 1) & (p > 0) & (t > 0)
        t_hi = t[unresolved].sum()
        phi = float((wm * np.abs(lat[m])).sum() / wm.sum())
        out = {"rows": int(m.sum()), "mean_abs_lat": phi}
        out.update(errors(a[m], wm, n, "_w"))
        out.update(spectrum=p.tolist(), target_spectrum=t.tolist(), error_spectrum=e.tolist(),
                   ratio=[float(pk / tk) if tk > 0 else None for pk, tk in zip(p, t)],
                   lsd_db=math.sqrt(float(np.mean((10.0 * np.log10(p[pos] / t[pos])) ** 2))) if pos.any() else None,
                   unresolved_power_ratio=float(p[unresolved].sum() / t_hi) if t_hi > 0 else None,
                   wavelength_km=[None] + [2.0 * math.pi * EARTH_RADIUS_KM * math.cos(math.radians(phi)) / kk for kk in range(1, nb)])
        return out

    def section(a, n):
        out = errors(a, w, n, "_w")
        out.update(errors(a, np.ones(H), n, ""))
        out["bands"] = {name: band(a, n, lo, hi) for name, lo, hi in LAT_BANDS}
        return out

    return {"fields": int(fields), "W": int(W), "lr_width": lr_width, "wavenumbers": k.tolist(),
            "variables": [section(acc[c], fields) for c in range(C)], "overall": section(acc.sum(0), fields * C)}


class FieldScores:
    """Zonal power spectra and latitude-weighted errors of output fields against their targets: one ``wsr_zonal_spectra`` launch per
    ``update`` into per-(variable, row) double accumulators on the device; the host synchronises only in ``compute``.

    ``FieldScores(device, lat_deg, lr_width=None)``: lat_deg = the H row latitudes in degrees (``field_latitudes``), lr_width = width
    of the low-resolution input (default W / 4).  ``update(pred, target, scale=None, shift=None)``: pred, target (B, C, H, W) with W
    along longitude; scale / shift per variable (C values) or per plane (B * C values) map to physical units x = scale * in + shift
    (the inverse StandardScaling: std and mean).  ``compute()`` returns ``field_summary`` of the accumulated sums."""

    def __init__(self, device, lat_deg, lr_width=None):
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.type != "cuda":
            raise nat.WsrError("metric accumulators run on the CUDA path only (got device %s)" % self.device)
        self.lat = np.asarray(lat_deg, dtype=np.float64).reshape(-1)
        self.lr_width = lr_width
        self.reset()

    def reset(self):
        self.C = self.W = None
        self.acc = None
        self.fields = 0              # fields per variable seen so far

    def _per_plane(self, v, B, C):
        if v is None:
            return None
        v = v.to(device=self.device, dtype=torch.float32).reshape(-1)
        if v.numel() == C:
            v = v.repeat(B)
        assert v.numel() == B * C, (v.numel(), B, C)
        return v.contiguous()

    def update(self, pred, target, scale=None, shift=None):
        p = pred.to(device=self.device, dtype=torch.float32).contiguous()
        t = target.to(device=self.device, dtype=torch.float32).contiguous()
        B, C, H, W = p.shape
        assert tuple(t.shape) == (B, C, H, W), (tuple(p.shape), tuple(t.shape))
        assert H == self.lat.size, "FieldScores was given %d latitudes for fields of %d rows" % (self.lat.size, H)
        S = 3 * (W // 2 + 1) + 3
        if self.acc is None:
            self.C, self.W = C, W
            self.acc = torch.zeros((C, H, S), dtype=torch.float64, device=self.device)
        assert (C, W) == (self.C, self.W), "every update of one FieldScores needs the same variable count and width"
        sc, sh = self._per_plane(scale, B, C), self._per_plane(shift, B, C)
        part = torch.zeros((B, C, H, S), dtype=torch.float64, device=self.device)
        nat.call("wsr_zonal_spectra", p.data_ptr(), t.data_ptr(), B * C, H, W, 0 if sc is None else sc.data_ptr(),
                 0 if sh is None else sh.data_ptr(), part.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream)
        self.acc += part.sum(0)
        self.fields += B

    def compute(self):
        if self.acc is None:
            return {}
        return field_summary(self.acc.cpu().numpy(), self.lat, self.W, self.fields, self.lr_width)


def write_field_scores(path, sections, units, lat_source, variable_names):
    """Write {name: FieldScores.compute()} for every FieldScores in ``sections`` to ``path`` (JSON), with the units the scores are in
    ("physical" or "standardised"), where the row latitudes came from and the variable names."""
    import json
    report = {"units": units, "lat_source": lat_source, "variable_names": list(variable_names or [])}
    report.update({name: f.compute() for name, f in sections.items()})
    with open(path, "w") as fh:
        json.dump(report, fh, indent=1)
