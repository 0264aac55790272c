"""Kernel time of ``wsr_zonal_spectra`` (JSON lines, appended to --out and printed): CUDA events over --launches launches of one
(pred, target, scale, shift) call, after a warm-up, for

  1. a validation batch: B = 64 fields, C = 1, 128x256 (8192 rows);
  2. an ensemble: 16 members x 64 conditions = 1024 fields of 128x256 (131,072 rows).

The fp64 work is counted as three DFTs (pred, target, error) of W/2 + 1 bins over W longitudes per row, at two FMAs (4 flops) per
real-by-complex multiply-add.  The inputs (8.4 MB and 134 MB for each of pred and target) are re-read every launch; the first fits
the 126 MB L2, the second does not.  The card name and power limit are read in the same run.

    python tools/prof_spectra.py [--launches 50] [--out profiles/spectra_prof_b200.jsonl]
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

DEV = "cuda:0"


def _gpu():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def kernel_time(fields, H, W, launches):
    nat = wsr.pkg.native
    g = torch.Generator(device=DEV).manual_seed(0)
    pred = torch.randn(fields, H, W, device=DEV, generator=g)
    target = torch.randn(fields, H, W, device=DEV, generator=g)
    scale = torch.full((fields,), 5.0, device=DEV)
    shift = torch.full((fields,), 280.0, device=DEV)
    acc = torch.zeros(fields * H * (3 * (W // 2 + 1) + 3), dtype=torch.float64, device=DEV)
    stream = torch.cuda.current_stream().cuda_stream

    def launch():
        nat.call("wsr_zonal_spectra", pred.data_ptr(), target.data_ptr(), fields, H, W, scale.data_ptr(), shift.data_ptr(), acc.data_ptr(),
                 stream)

    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(launches):
        launch()
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / launches
    gflop = 4.0 * 3 * fields * H * (W // 2 + 1) * W / 1e9
    return {"fields": fields, "H": H, "W": W, "launches": launches, "ms": ms, "fp64_gflop": gflop, "fp64_tflops": gflop / ms}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "spectra_prof_b200.jsonl"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_spectra: no CUDA device")
    gpu = _gpu()
    rows = [{"measure": "zonal_spectra_validation_batch", "gpu": gpu, "result": kernel_time(64, 128, 256, a.launches)},
            {"measure": "zonal_spectra_ensemble_16x64", "gpu": gpu, "result": kernel_time(16 * 64, 128, 256, max(1, a.launches // 5))}]
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as fh:
        for r in rows:
            line = json.dumps(r)
            print(line)
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
