"""Ensemble sampling on one GPU, three measurements (JSON lines on stdout):

  1. per-step time of a graph-replayed ensemble loop (ResDiff Cfg-A, 128x256) at N x B = 8 x 8 and 16 x 4 members x conditions,
     against the plain batch-64 loop, alternated in the same process (member-keyed noise is the only per-step difference);
  2. the time one SRDiff ensemble chunk saves by running the RRDB-17 encoder on its B conditions once instead of on R x B;
  3. the bandwidth of wsr_ensemble_stats at N = 8, 32, 256 on 64 planes of 128x256 (device-bound: >= 0.3 GB per call), against the
     measured HBM peak of 6512 GB/s.  Bytes = (N + 1) * 4 read + 8 written (mean, spread) per pixel.

    python tools/prof_ensemble.py [--steps 30] [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import wsr  # noqa: E402
from bench import CFG_A, LINEAR_1000  # noqa: E402

HBM_PEAK_GBS = 6512.0
DEV = "cuda:0"


def _gpu():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
        return q.stdout.strip().splitlines()[0]
    except Exception:
        return torch.cuda.get_device_name(0)


def _events():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def _resdiff():
    U = wsr.sub("models.diffusion_models.resdiff.unet").UNet
    D = wsr.sub("models.diffusion_models.resdiff.resdiff_diffusion").ResDiffDiffusion
    networks = wsr.sub("models.diffusion_models.networks")
    torch.manual_seed(0)
    net = U(precision="bf16", **CFG_A)
    networks.init_weights(net, "orthogonal")
    net = net.to(DEV).eval()
    diff = D(net, image_height=CFG_A["image_height"], image_width=CFG_A["image_width"], channels=1, conditional=True).to(DEV)
    diff.set_new_noise_schedule(LINEAR_1000, DEV)
    return diff


def _loop(diff, n_members, B, steps):
    """ms per graph-replayed step of a loop over n_members x B images (n_members = 0: the plain loop of B images)."""
    dmod = wsr.sub("models.diffusion_models.diffusion")
    H, W = CFG_A["image_height"], CFG_A["image_width"]
    cond = torch.randn((B, 1, H, W), device=DEV)
    R = max(n_members, 1)
    plan = diff._plan(R * B, DEV)
    keys = None
    if n_members:
        plan.set_condition(cond, repeats=R)
        keys = torch.tensor([dmod.member_key(1, m) for m in range(R)], dtype=torch.int64, device=DEV)
    else:
        plan.set_condition(cond)
    loop = diff.begin_loop(plan, (R * B, 1, H, W), seed=1, member_keys=keys)
    loop.step()
    loop.capture()
    for _ in range(3):
        loop.replay()
    s, e = _events()
    s.record()
    for _ in range(steps):
        loop.replay()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / steps


def loop_times(steps, reps):
    diff = _resdiff()
    rows = {"plain_b64": [], "ens_8x8": [], "ens_16x4": []}
    for _ in range(reps):                                       # alternated: the three loops see the same box state
        rows["plain_b64"].append(_loop(diff, 0, 64, steps))
        rows["ens_8x8"].append(_loop(diff, 8, 8, steps))
        rows["ens_16x4"].append(_loop(diff, 16, 4, steps))
    out = {k: {"ms_per_step": v, "median": sorted(v)[len(v) // 2]} for k, v in rows.items()}
    base = out["plain_b64"]["median"]
    for k in ("ens_8x8", "ens_16x4"):
        out[k]["vs_plain_b64"] = out[k]["median"] / base
    return out


def srdiff_encoder(reps=10):
    """Encoder time of one chunk of R members x B conditions: once on B (ensemble) vs on R x B stacked copies."""
    Rn = wsr.sub("models.rrdb_encoder.RRDBNet").RRDBNet
    S = wsr.sub("models.diffusion_models.srdiff.srdiff_diffusion").SRDiffDiffusion
    torch.manual_seed(0)
    d = S.__new__(S)
    torch.nn.Module.__init__(d)
    d.rrdb_encoder = Rn(1, 1, 64, 17, 32, precision="bf16").to(DEV).eval()
    out = {}
    for R, B in ((8, 8), (16, 4)):
        lr = torch.randn((B, 1, 32, 64), device=DEV)
        t = {}
        for name, x in (("once", lr), ("stacked", lr.repeat(R, 1, 1, 1))):
            d._condition(x)
            s, e = _events()
            s.record()
            for _ in range(reps):
                d._condition(x)
            e.record()
            torch.cuda.synchronize()
            t[name] = s.elapsed_time(e) / reps
        out["%dx%d" % (R, B)] = {"encoder_once_ms": t["once"], "encoder_stacked_ms": t["stacked"], "saved_ms_per_chunk": t["stacked"] - t["once"]}
    return out


def stats_bandwidth(reps=20):
    nat = wsr.pkg.native
    P, HW = 64, 128 * 256
    st = torch.cuda.current_stream().cuda_stream
    y = torch.randn((P, HW), device=DEV)
    mean = torch.empty((P, HW), device=DEV)
    spread = torch.empty((P, HW), device=DEV)
    out = {}
    for N in (8, 32, 256):
        ens = torch.randn((N, P, HW), device=DEV)
        acc = torch.zeros((P, 5), dtype=torch.float64, device=DEV)
        hist = torch.zeros((P, N + 1), dtype=torch.int64, device=DEV)
        args = (ens.data_ptr(), N, P * HW, y.data_ptr(), P, HW, 0, mean.data_ptr(), spread.data_ptr(), acc.data_ptr(), hist.data_ptr(), st)
        for _ in range(3):
            nat.call("wsr_ensemble_stats", *args)
        s, e = _events()
        s.record()
        for _ in range(reps):
            nat.call("wsr_ensemble_stats", *args)
        e.record()
        torch.cuda.synchronize()
        ms = s.elapsed_time(e) / reps
        nbytes = P * HW * ((N + 1) * 4 + 8)
        out["N%d" % N] = {"ms": ms, "GB": nbytes / 1e9, "GBps": nbytes / ms / 1e6, "share_of_hbm_peak": nbytes / ms / 1e6 / HBM_PEAK_GBS}
        del ens
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    gpu = _gpu()
    for name, fn in (("ensemble_stats", stats_bandwidth), ("srdiff_encoder", srdiff_encoder),
                     ("loop_step", lambda: loop_times(a.steps, a.reps))):
        print(json.dumps({"measure": name, "gpu": gpu, "result": fn()}), flush=True)


if __name__ == "__main__":
    main()
