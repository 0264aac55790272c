"""Cost of the EMA weights on one GPU, two measurements (JSON lines, appended to --out and printed):

  1. ``wsr_adam_step`` against ``wsr_adam_step_ema`` (blend branch) over the 98,870,734 parameters of ResDiff Cfg-A: CUDA events
     over --launches launches of each, alternated in blocks of 10.  Bytes per parameter: Adam reads p, g, m, v and writes p, m, v
     (28 B); the fused EMA adds one read and one write of the EMA (36 B).  The 2.8-3.6 GB working set is far above the 126 MB L2.
     Rates are given against the measured HBM peak of 6512 GB/s.
  2. the training step at the bench shape (ResDiff Cfg-A, 128x256, B = 4, bf16, dropout 0.2, one-launch Adam) with EMA off and on
     (schedule 0 / 1 / 0.9999: every step blends), alternated, --reps repetitions of --steps steps each.

    python tools/prof_ema.py [--launches 60] [--steps 20] [--reps 2] [--out profiles/ema_prof_b200.jsonl]
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
N_PARAMS = 98_870_734
DEV = "cuda:0"


def _gpu():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def adam_kernels(launches):
    nat = wsr.pkg.native
    n = N_PARAMS
    g = torch.Generator(device=DEV).manual_seed(0)
    p, grad, m, ema = (0.05 * torch.randn(n, device=DEV, generator=g) for _ in range(4))
    v = torch.rand(n, device=DEV, generator=g) * 1e-4
    stream = torch.cuda.current_stream().cuda_stream
    hyper = (1e-4, 0.9, 0.999, 1e-8, 0.0)

    def adam(step):
        nat.call("wsr_adam_step", p.data_ptr(), grad.data_ptr(), m.data_ptr(), v.data_ptr(), n, *hyper, step, stream)

    def adam_ema(step):
        nat.call("wsr_adam_step_ema", p.data_ptr(), grad.data_ptr(), m.data_ptr(), v.data_ptr(), ema.data_ptr(), n, *hyper, step, 0.9999,
                 stream)

    arms = {"wsr_adam_step": (adam, 28), "wsr_adam_step_ema": (adam_ema, 36)}
    ms = {k: 0.0 for k in arms}
    count = {k: 0 for k in arms}
    step = 1
    for fn, _ in arms.values():                              # warm-up
        for _ in range(5):
            fn(step); step += 1
    torch.cuda.synchronize()
    block = 10
    while min(count.values()) < launches:
        for k, (fn, _) in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(block):
                fn(step); step += 1
            e1.record()
            e1.synchronize()
            ms[k] += e0.elapsed_time(e1)
            count[k] += block
    out = {}
    for k, (_, bpp) in arms.items():
        t = ms[k] / count[k]
        gb = bpp * n / 1e9
        out[k] = {"launches": count[k], "ms": t, "GB": gb, "GBps": gb / t * 1e3, "share_of_hbm_peak": gb / t * 1e3 / HBM_PEAK_GBS}
    out["ema_over_adam"] = out["wsr_adam_step_ema"]["ms"] / out["wsr_adam_step"]["ms"]
    return out


def train_steps(steps, reps):
    glue = wsr.sub("autograd_glue")
    U = wsr.sub("models.diffusion_models.resdiff.unet").UNet
    D = wsr.sub("models.diffusion_models.resdiff.resdiff_diffusion").ResDiffDiffusion
    networks = wsr.sub("models.diffusion_models.networks")
    torch.manual_seed(0)
    net = U(precision="bf16", **CFG_A)
    networks.init_weights(net, "orthogonal")
    net = net.to(DEV).train()
    diff = D(net, image_height=CFG_A["image_height"], image_width=CFG_A["image_width"], channels=1, conditional=True).to(DEV)
    diff.set_new_noise_schedule(LINEAR_1000, DEV)
    diff.set_loss(DEV)
    B = 4
    plan = net.train_plan(B, DEV)
    params = list(diff.parameters())
    # two optimizers over the same flat parameter buffer, each with its own moments: only the EMA differs between the arms
    opts = {"ema_off": glue.FusedAdam(params, lr=1e-4), "ema_on": glue.FusedAdam(params, lr=1e-4, ema=(0, 1, 0.9999))}
    for o in opts.values():
        o.attach_flat(plan)
    g = torch.Generator().manual_seed(1234)
    lr = torch.randn(B, 1, 32, 64, generator=g)
    sr = torch.nn.functional.interpolate(lr, scale_factor=4, mode="bicubic").to(DEV)
    hr = sr + 0.3 * torch.randn(sr.shape, generator=g).to(DEV)

    def step(opt):
        opt.zero_grad()
        loss = diff.p_losses({"HR": hr, "SR": sr})
        (loss.sum() / hr.numel()).backward()
        opt.step()

    for o in opts.values():
        for _ in range(3):
            step(o)
    torch.cuda.synchronize()
    runs = {k: [] for k in opts}
    for _ in range(reps):
        for k, o in opts.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step(o)
            e1.record()
            e1.synchronize()
            runs[k].append(e0.elapsed_time(e1) / steps)
    return {"shape": "ResDiff Cfg-A 128x256, B=4, bf16", "steps_per_run": steps, "ms_per_step": runs,
            "ema_on_minus_off_ms": [a - b for a, b in zip(runs["ema_on"], runs["ema_off"])],
            "run_to_run_spread_ms": {k: max(v) - min(v) for k, v in runs.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=60)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ema_prof_b200.jsonl"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_ema.py needs a CUDA device")
    gpu = _gpu()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as fh:
        for name, fn in (("adam_kernels", lambda: adam_kernels(a.launches)), ("train_step", lambda: train_steps(a.steps, a.reps))):
            line = json.dumps({"measure": name, "gpu": gpu, "result": fn()})
            print(line, flush=True)
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
