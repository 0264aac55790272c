"""Validation metric accumulators of the reference (training/metrics.py:30-201: MAE, MSE, RMSE, MR; containers :300-365) on
the device.  ``update`` is one ``wsr_error_sums`` launch per metric object -- or ONE launch for all four through
``ErrorSums`` / ``ValidationMetrics`` -- with double accumulators on the device and no host synchronisation until ``compute``.
``update(predicted, target, scale=std)`` folds the inverse StandardScaling into the same pass (the means cancel in the
difference), so RMSE in Kelvin never needs the de-normalised tensors.  PSNR / SSIM (torcheval / skimage wrappers in the
reference) are outside the accelerated path."""
from abc import ABC, abstractmethod

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
