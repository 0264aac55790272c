#!/usr/bin/env python
"""bench.py -- headline benchmark of the diffusion super-resolution hot path (BASELINE.json).

Metric: 128x256 t2m super-resolution samples/s for the full 1000-step DDPM reverse loop (ResDiff Cfg-A UNet, bf16,
batch 64 IN TOTAL sharded over the N GPUs = BASELINE.json configs[1] / SURVEY 8(d) C2, i.e. strong scaling; synthetic
WeatherBench-shaped fields, random-init weights).  The same JSON line carries, as sub-records: ``weak`` (64 samples PER GPU),
``train`` (configs[2]: the training step, NCCL all-reduce at N > 1), ``configs`` (configs[3] SRDiff + RRDB-17 at B = 32 and
configs[4] the 3-variable stress model, N = 1), ``eager_gpu_baseline`` (the reference's algorithm in eager PyTorch on the same GPU).

    python bench.py --gpus N --steps K --warmup W            # our CUDA path (one rank per GPU under torchrun for N>1)
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host CPU cores
    python bench.py --impl reference --ref-device cuda [--ref-batch 16] [--ref-autocast]     # optional extra: the same algorithm run
                                                             # op by op by eager PyTorch on cuda:0 (never the default arm)
    python bench.py --workload train [--profile-ops]         # configs[2]: the training step
    python bench.py --gpus N --steps K --warmup W --dump-outputs DIR   # also writes DIR/x.npy, the image after the last timed step

A "step" is ONE reverse (p_sample) step of the loop over the whole local batch: level-projection select, FD gate,
stem assembly, the UNet (~270 kernel launches, replayed as one CUDA graph), the fused sampler update.  Every one of the
1000 steps of a chain is the same work, so
    value = samples/s = global_batch / (T * seconds_per_step + once-per-batch precompute seconds),  T = 1000,
with K timed steps (K = 1000 times the whole chain; past the end of the chain its step counter restarts).  The activations
of one step (GBs at batch 64) far exceed the 126 MB L2, so no L2 flush is needed between timed steps.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

T_FULL = 1000
FLOPS_PER_SAMPLE_STEP = 206.39e9        # SURVEY.md 8(d): algorithmic FLOPs of one ResDiff Cfg-A UNet call per sample
LINEAR_1000 = {"schedule": "linear", "n_timestep": T_FULL, "linear_start": 1e-6, "linear_end": 1e-2}
CFG_A = dict(in_channel=5, out_channel=1, norm_groups=32, inner_channel=64, channel_mults=[1, 2, 4, 8, 8], attn_res=[16],
             res_blocks=2, dropout=0.2, image_height=128, image_width=256, image_channels=1)


_REAL_STDOUT = None


def _claim_stdout():
    """stdout must carry exactly ONE JSON line.  Libraries write there too (NCCL prints its version banner on stdout when NCCL_DEBUG
    is set, as it is on the GPU boxes): file descriptor 1 is pointed at stderr for the rest of the run and the JSON line goes to the
    saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def _emit(text):
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        print(text, flush=True)
    else:
        os.write(_REAL_STDOUT, (text + "\n").encode())


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return p, "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region: NVML polled every 5 ms from a thread (a timed region can be as short
    as 60 ms at 8 images per GPU, where ``nvidia-smi -lms`` delivers nothing); falls back to an ``nvidia-smi -lms 100`` child process."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.nvml, self.samples, self._stop = None, [], threading.Event()

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.handle = None
            try:      # the CUDA ordinal need not be the NVML index (CUDA_VISIBLE_DEVICES): go through the UUID when torch exposes it
                import torch
                uuid = str(torch.cuda.get_device_properties(int(self.index)).uuid)
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid if uuid.startswith("GPU-") else "GPU-" + uuid)
            except Exception:
                self.handle = None
            if self.handle is None:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(int(self.index))
            self.nvml = pynvml
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv = self.nvml
        while not self._stop.is_set():
            try:
                self.samples.append((float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)),
                                     int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))))
            except Exception:
                pass
            time.sleep(0.005)

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.nvml is not None:
            self._stop.set()
            self.th.join(timeout=2)
            nv = self.nvml
            bits = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                    "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                    "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                    "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            sm = [c for c, _ in self.samples]
            reasons = sorted(n for n, b in bits.items() if any(r & b for _, r in self.samples))
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.sm_max if sm else None, "reasons": reasons,
                    "samples": len(sm), "source": "nvml, 5 ms poll"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 100"}


# ----------------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference algorithm on the host cores
# ----------------------------------------------------------------------------------------------------------------------
def workload_text(global_batch):
    return ("configs[1]: ResDiff Cfg-A UNet (inner 64, mults 1-2-4-8-8, attn@16) + bicubic prior, t2m 32x64->128x256, "
            "1000-step DDPM reverse loop, bf16, batch %d in total sharded over the GPUs" % global_batch)


def cpu_reference_steps(n_steps, warmup, seed=0):
    """Times reverse steps of the reference algorithm (oracle/ port, fp32 torch-CPU, all host threads) at B=1, 128x256.
    Returns (seconds per step list, cores)."""
    import torch
    from oracle import nets, process
    from oracle.schedule import ddpm_tables
    from oracle.weights import seeded_randn, seeded_state_dict
    import numpy as np
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    man = np.load(os.path.join(ROOT, "tests", "golden", "manifest.npz"))
    keys = [str(k) for k in man["resdiff.keys"]]
    shapes = [tuple(int(x) for x in str(s).split(",")) if str(s) else () for s in man["resdiff.shapes"]]
    sd = seeded_state_dict(zip(keys, shapes), seed)
    cfg = dict(CFG_A)
    cfg["dropout"] = 0.0
    tab32, sap = ddpm_tables(LINEAR_1000)
    tab = {k: torch.from_numpy(v) for k, v in tab32.items()}
    cond = torch.nn.functional.interpolate(seeded_randn("bench.lr", (1, 1, 32, 64), 1234), scale_factor=4, mode="bicubic")
    x = seeded_randn("bench.x", (1, 1, 128, 256), 4321)

    def denoise(xx, level):
        return nets.resdiff_unet(sd, torch.cat([cond, xx], 1), level, cfg)

    times = []
    t = T_FULL - 1
    with torch.no_grad():
        for i in range(warmup + n_steps):
            z = seeded_randn("bench.z%d" % i, (1, 1, 128, 256), 99)
            t0 = time.perf_counter()
            x, _ = process.p_sample_step(denoise, tab, sap, x, t, z)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
            t = (t - 1) % T_FULL                      # past the end of the chain, restart it
    return times, cores


def gpu_eager_reference_steps(n_steps, warmup, batch, autocast, seed=0):
    """OPTIONAL extra arm (``--impl reference --ref-device cuda``, never the default): the same oracle port of the reference's
    algorithm, but executed by eager PyTorch (cuDNN / cuBLAS, one launch per op, fp32 or bf16 autocast) on cuda:0 at ``batch``
    samples -- what running the reference's own modules on a B200 amounts to.  Returns seconds per step (CUDA events)."""
    import torch
    from oracle import nets, process
    from oracle.schedule import ddpm_tables
    from oracle.weights import seeded_randn, seeded_state_dict
    import numpy as np
    dev = torch.device("cuda:0")
    torch.backends.cudnn.benchmark = True                    # the reference sets it (train.py:24-25)
    man = np.load(os.path.join(ROOT, "tests", "golden", "manifest.npz"))
    keys = [str(k) for k in man["resdiff.keys"]]
    shapes = [tuple(int(x) for x in str(s).split(",")) if str(s) else () for s in man["resdiff.shapes"]]
    sd = {k: v.to(dev) for k, v in seeded_state_dict(zip(keys, shapes), seed).items()}
    cfg = dict(CFG_A)
    cfg["dropout"] = 0.0
    tab32, sap = ddpm_tables(LINEAR_1000)
    tab = {k: torch.from_numpy(v).to(dev) for k, v in tab32.items()}
    cond = torch.nn.functional.interpolate(seeded_randn("bench.lr", (batch, 1, 32, 64), 1234), scale_factor=4, mode="bicubic").to(dev)
    x = seeded_randn("bench.x", (batch, 1, 128, 256), 4321).to(dev)
    z = seeded_randn("bench.z", (batch, 1, 128, 256), 99).to(dev)

    def denoise(xx, level):
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
            return nets.resdiff_unet(sd, torch.cat([cond, xx], 1), level.to(dev), cfg).float()

    times = []
    t = T_FULL - 1
    with torch.no_grad():
        for i in range(warmup + n_steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            x, _ = process.p_sample_step(denoise, tab, sap, x, t, z)
            e1.record()
            torch.cuda.synchronize()
            if i >= warmup:
                times.append(e0.elapsed_time(e1) * 1e-3)
            t = (t - 1) % T_FULL                      # past the end of the chain, restart it
    return times


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.ref_device == "cuda":
        times = gpu_eager_reference_steps(args.steps, max(args.warmup, 2), args.ref_batch, args.ref_autocast)
        ms = 1e3 * sum(times) / len(times)
        val = args.ref_batch / (T_FULL * ms * 1e-3)
        _emit(json.dumps({
            "impl": "reference", "device": "cuda:0 eager PyTorch (%s)" % ("bf16 autocast" if args.ref_autocast else "fp32"),
            "metric": "128x256 t2m SR samples/sec (1000-step loop)", "value": val, "unit": "samples/s", "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.ref_autocast else "f32", "data": "synthetic",
            "config": {"workload": "ResDiff Cfg-A UNet, 128x256, 1000-step DDPM reverse loop; oracle port of the reference run by eager PyTorch",
                       "batch_per_gpu": args.ref_batch, "T": T_FULL},
            "note": "extra arm, not the CPU baseline: same algorithm, library kernels (cuDNN / cuBLAS) launched op by op", "gpu_launches": 0}))
        return
    times, cores = cpu_reference_steps(args.steps, args.warmup)
    ms = 1e3 * sum(times) / len(times)
    val = 1.0 / (T_FULL * ms * 1e-3)
    sample = ("B=1 of the batch of 64, %d reverse steps of the 1000-step chain at 128x256 (oracle port of the reference, fp32 torch-CPU, all "
              "host threads); samples/s = 1 / (1000 x s per step): the CPU runs the samples of a batch one after the other.  The port computes "
              "attention without the reference's .contiguous() copies of the (B,N,N) matrices (39%% of the reference's CPU step in the survey), "
              "so it is FASTER than the reference's own modules would be" % len(times))
    line = {
        "impl": "reference", "metric": "128x256 t2m SR samples/sec (1000-step loop)", "value": val, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text(64), "global_batch": 64, "T": T_FULL, "cpu_arm": "bounded sample: batch 1 of the 64, fp32"},
        "cpu_baseline": {"value": val, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------------
def _conv_traffic():
    """DRAM bytes per gemm_tc_kernel launch (read + write, averaged over the launches of a B=64 sampler step) from the
    committed ncu pass (profiles/*conv_traffic.json, newest round first); None if no file is there."""
    pdir = os.path.join(ROOT, "profiles")
    for name in ("r02_conv_traffic.json", "r01c_conv_traffic.json"):
        try:
            with open(os.path.join(pdir, name)) as f:
                return json.load(f)["dram_bytes_per_launch"], name
        except Exception:
            continue
    return None, None


class _Ctx:
    """Process-wide state of one bench run (rank, device, barrier helpers)."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, *vals):
        t = self.torch.tensor([float(v) for v in vals], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def close(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def _resdiff(ctx, precision="bf16", **over):
    import wsr
    torch = ctx.torch
    U = wsr.sub("models.diffusion_models.resdiff.unet").UNet
    D = wsr.sub("models.diffusion_models.resdiff.resdiff_diffusion").ResDiffDiffusion
    networks = wsr.sub("models.diffusion_models.networks")
    cfg = dict(CFG_A)
    cfg.update(over)
    torch.manual_seed(0)
    net = U(precision=precision, **cfg)
    networks.init_weights(net, "orthogonal")          # the reference's "random-init weights" (networks.py:164-165)
    net = net.to(ctx.dev).eval()
    diff = D(net, image_height=cfg["image_height"], image_width=cfg["image_width"], channels=cfg["image_channels"], conditional=True).to(ctx.dev)
    diff.set_new_noise_schedule(LINEAR_1000, ctx.dev)
    return net, diff


def _time_loop(ctx, diff, plan, set_condition, shape, K, warmup, sample_clocks=False):
    """Precompute (timed separately), W eager warm-up steps, graph capture, K timed graph replays bracketed by barrier + synchronize.
    Returns dict(ms_per_step, pre_ms, launches_per_step, clocks, loop) -- times are the MAX over ranks."""
    torch = ctx.torch
    import wsr
    nat = wsr.pkg.native
    ev = lambda: torch.cuda.Event(enable_timing=True)
    set_condition()                                   # untimed first call (lazy init)
    loop = diff.begin_loop(plan, shape, seed=7)
    torch.cuda.synchronize(ctx.dev)
    e0, e1 = ev(), ev()
    e0.record()
    set_condition()
    loop = diff.begin_loop(plan, shape, seed=7)
    e1.record()
    torch.cuda.synchronize(ctx.dev)
    pre_ms = e0.elapsed_time(e1)
    l0 = nat.launches
    loop.step()
    launches_per_step = nat.launches - l0
    for _ in range(max(0, warmup - 1)):
        loop.step()
    loop.capture()
    loop.replay()                                   # one graph warm-up replay
    left = T_FULL - 2 - max(0, warmup - 1)          # steps left in the chain after the warm-up steps and replay
    sampler = ClockSampler(ctx.local) if sample_clocks else None
    ctx.barrier()
    if sampler:
        sampler.start()
    e0, e1 = ev(), ev()
    e0.record()
    for _ in range(K):
        if left == 0:                               # chain finished: restart its step counter on the current x, same work per step
            loop.reset_counter()
            left = T_FULL
        loop.replay()
        left -= 1
    e1.record()
    ctx.barrier()
    if left < 2:                                    # the roofline pass and --profile-ops step the loop twice more: keep t >= 0
        loop.reset_counter()
    clocks = sampler.stop() if sampler else None
    ms_total, pre = ctx.max_over_ranks(e0.elapsed_time(e1), pre_ms)
    return dict(ms_per_step=ms_total / K, pre_ms=pre, launches_per_step=launches_per_step, clocks=clocks, loop=loop, K=K)


DUMP_LIMIT_BYTES = 64 << 20


def _dump_outputs(ctx, out_dir, arrays):
    """--dump-outputs: each (B, ...) array, the shards of all ranks concatenated in rank order, is written by rank 0 as
    <out_dir>/<name>.npy in float32.  Above DUMP_LIMIT_BYTES in all, a fixed seeded subset of the batch rows is kept (sorted)."""
    import numpy as np
    torch = ctx.torch
    full = {}
    for name, t in arrays.items():
        t = t.detach().float().contiguous()
        if ctx.world > 1:
            parts = [torch.empty_like(t) for _ in range(ctx.world)]
            ctx.dist.all_gather(parts, t)
            t = torch.cat(parts)
        full[name] = t.cpu().numpy()
    if ctx.rank != 0:
        return
    total = sum(a.nbytes for a in full.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, a in full.items():
        if total > DUMP_LIMIT_BYTES:
            keep = max(1, int(a.shape[0] * DUMP_LIMIT_BYTES // total))
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _synthetic_sr(ctx, B, c=1, lr_hw=(32, 64), scale=4, pinned=True):
    """Synthetic WeatherBench-shaped standardised fields (SURVEY 8d): LR randn, SR = bicubic upsample, in PINNED host memory."""
    torch = ctx.torch
    g = torch.Generator().manual_seed(1234 + ctx.rank)
    lr = torch.randn(B, c, lr_hw[0], lr_hw[1], generator=g)
    sr = torch.nn.functional.interpolate(lr, scale_factor=scale, mode="bicubic").contiguous()
    return lr, (sr.pin_memory() if pinned else sr)


def _roofline(ctx, plan, loop, B, ms_per_step, profile_ops):
    """One eager step with per-launch CUDA events on the launching stream -> the conv_tc (gemm_tc_kernel) roofline record."""
    plan.eng.prof = []
    loop.step()
    summ = plan.eng.prof_summary()
    plan.eng.prof = None
    peaks, peak_src = _peaks()
    conv = summ.get("conv_tc", [0, 1e-9, 0, 0, 0])
    conv_tflops = conv[2] / (conv[1] * 1e-3) / 1e12 if conv[1] > 0 else 0.0
    conv_xtflops = conv[4] / (conv[1] * 1e-3) / 1e12 if conv[1] > 0 else 0.0
    step_ms_prof = sum(v[1] for v in summ.values())
    traffic, traffic_src = _conv_traffic()
    whole = B * FLOPS_PER_SAMPLE_STEP / (ms_per_step * 1e-3) / 1e12
    roofline = {
        "bound": "tensor", "kernel": "gemm_tc_kernel (conv_tc launches)", "achieved": conv_tflops, "peak": peaks["bf16_tflops"],
        "unit": "TFLOP/s", "frac": conv_tflops / peaks["bf16_tflops"],
        "executed_flops_per_step": conv[4], "algorithmic_flops_per_step": conv[2],
        "achieved_executed": conv_xtflops, "frac_executed": conv_xtflops / peaks["bf16_tflops"],
        "executed_note": "the four nearest-x2 + 3x3 convolutions run 4 phase-merged taps instead of the reference's 9: 'achieved' counts the "
                         "reference's FLOPs (SURVEY 8d), 'achieved_executed' what the tensor pipe really did (compare with ncu)",
        "traffic": traffic, "traffic_note": "ncu dram__bytes_read+write per gemm_tc_kernel launch, averaged over one B=64 step (profiles/%s)" % traffic_src,
        "peak_source": peak_src + " burst",
        "launches_per_step": conv[0], "kernel_ms_per_step": conv[1], "kernel_share_of_step": conv[1] / step_ms_prof if step_ms_prof else None,
        "whole_step_tflops": whole,
        "whole_step_frac_of_burst": whole / peaks["bf16_tflops"],
        "whole_step_frac_of_sustained": whole / peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]),
        "per_op_ms": {k: round(v[1], 4) for k, v in sorted(summ.items(), key=lambda kv: -kv[1][1])[:8]},
    }
    if profile_ops and ctx.rank == 0:
        plan.eng.prof, plan.eng.prof_detail = [], True
        loop.step()
        detail = plan.eng.prof_summary()
        plan.eng.prof, plan.eng.prof_detail = None, False
        print("# per-shape breakdown of the tensor-core launches (B=%d): name launches ms TFLOP/s(algorithmic) TFLOP/s(executed)" % B, file=sys.stderr)
        for name, (n, ms, fl, nb, xf) in sorted(detail.items(), key=lambda kv: -kv[1][1]):
            if name.startswith(("conv_tc", "gemm_tc", "attn_tc")):
                print("#   %-40s %3d %8.3f %8.1f %8.1f" % (name, n, ms, fl / (ms * 1e-3) / 1e12 if ms > 0 else 0, xf / (ms * 1e-3) / 1e12 if ms > 0 else 0), file=sys.stderr)
        rows = sorted(summ.items(), key=lambda kv: -kv[1][1])
        print("# per-op breakdown of one eager step (B=%d): name launches ms TFLOP/s GB/s" % B, file=sys.stderr)
        for name, (n, ms, fl, nb, xf) in rows:
            print("#   %-22s %4d %9.3f %9.1f %9.1f" % (name, n, ms, fl / (ms * 1e-3) / 1e12 if ms > 0 else 0, nb / (ms * 1e-3) / 1e9 if ms > 0 else 0), file=sys.stderr)
        print("#   total %.3f ms (graph: %.3f ms/step)" % (step_ms_prof, ms_per_step), file=sys.stderr)
    return roofline


def _e2e(ctx, diff, sr_host, B, ms_per_step, budget_s):
    """The same metric through the public API with HOST buffers: H2D of the condition, the whole reverse loop and D2H of the result
    inside the timed region (a shorter schedule, scaled to 1000 steps, when the full loop does not fit the budget)."""
    torch = ctx.torch
    out_host = torch.empty_like(sr_host).pin_memory()
    t_e2e = T_FULL
    est = T_FULL * ms_per_step * 1e-3
    if est > budget_s:
        t_e2e = max(10, int(T_FULL * budget_s / est))
    sched = dict(LINEAR_1000)
    sched["n_timestep"] = t_e2e
    diff.set_new_noise_schedule(sched, ctx.dev)
    diff.sample_seed = 11
    ctx.barrier()
    t0 = time.perf_counter()
    x_in = {"SR": sr_host.to(ctx.dev, non_blocking=True)}
    res = diff.super_resolution(x_in)
    out_host.copy_(res, non_blocking=True)
    torch.cuda.synchronize(ctx.dev)
    el = time.perf_counter() - t0
    (el,) = ctx.max_over_ranks(el)
    diff.set_new_noise_schedule(LINEAR_1000, ctx.dev)
    return {"value": B * ctx.world / (el * T_FULL / t_e2e), "unit": "samples/s", "h2d_bytes_per_step": sr_host.numel() * 4,
            "d2h_bytes_per_step": out_host.numel() * 4, "api": "ResDiffDiffusion.super_resolution({'SR': host tensor}) + .cpu()",
            "loop_steps_run": t_e2e, "seconds": el,
            "note": "one public-API call = one whole reverse loop; H2D of the condition and D2H of the result inside the timed region"
                    + ("" if t_e2e == T_FULL else "; run with a %d-step schedule and scaled to 1000 steps" % t_e2e)}


def measure_sampling(ctx, net, diff, B, args, full):
    """configs[1] at B samples on this GPU.  full: also roofline pass, e2e and clocks (the headline record)."""
    torch = ctx.torch
    _, sr_host = _synthetic_sr(ctx, B)
    plan = net.plan(B, ctx.dev, strict_tc=False)
    cond = sr_host.to(ctx.dev, non_blocking=True)
    torch.cuda.synchronize(ctx.dev)
    r = _time_loop(ctx, diff, plan, lambda: plan.set_condition(cond), tuple(cond.shape), args.steps, args.warmup, sample_clocks=full)
    if full and args.dump_outputs:
        # the image of the reverse loop after the last timed step, before the roofline pass steps it again
        _dump_outputs(ctx, args.dump_outputs, {"x": r["loop"].x})
    ms, pre = r["ms_per_step"], r["pre_ms"]
    rec = {"batch_per_gpu": B, "global_batch": B * ctx.world, "ms_per_step": ms, "precompute_ms_per_batch": pre,
           "value": B * ctx.world / (T_FULL * ms * 1e-3 + pre * 1e-3), "unit": "samples/s", "steps": r["K"],
           "launches_per_step": r["launches_per_step"], "clocks": r["clocks"]}
    if full:
        rec["roofline"] = _roofline(ctx, plan, r["loop"], B, ms, args.profile_ops)
        rec["e2e"] = None if args.no_e2e else _e2e(ctx, diff, sr_host, B, ms, args.e2e_budget)
        rec["tc_launches_per_step"], rec["simt_launches_total"] = plan.eng.n_tc, plan.eng.n_simt
    del r["loop"]
    return rec


def measure_train(ctx, args, steps, warmup, profile=False):
    """configs[2]: one training step = q_sample + UNet forward (dropout 0.2) + loss + hand-written backward + bucketed gradient
    all-reduce + one-launch Adam over the flat parameter buffer, batch 4 per GPU at 128x256.  Returns the record (ms per step is the
    max over ranks); for N > 1 also the step time WITHOUT the all-reduce, so its exposed (non-overlapped) part is visible."""
    import numpy as np
    import wsr
    torch, dist = ctx.torch, ctx.dist
    nat = wsr.pkg.native
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    B = args.train_batch
    glue = wsr.sub("autograd_glue")
    par = wsr.sub("parallel")
    np.random.seed(rank)
    net, diff = _resdiff(ctx, args.train_precision)
    net.train()
    diff.set_loss(dev)
    plan = net.train_plan(B, dev)
    opt = glue.FusedAdam(list(diff.parameters()), lr=1e-4)
    opt.attach_flat(plan)
    reducer = par.FlatGradReducer(plan) if world > 1 else None
    g = torch.Generator().manual_seed(1234 + rank)
    lr = torch.randn(B, 1, 32, 64, generator=g)
    sr = torch.nn.functional.interpolate(lr, scale_factor=4, mode="bicubic").to(dev)
    hr = sr + 0.3 * torch.randn(sr.shape, generator=g).to(dev)
    numel = hr.numel() * world

    def step(reduce=True):
        opt.zero_grad()
        loss = diff.p_losses({"HR": hr, "SR": sr})
        (loss.sum() / numel).backward()
        if reducer is not None:
            if reduce:
                reducer.finish()
        opt.step()
        return loss

    def timed(n, reduce=True):
        if reducer is not None:
            plan.on_ready = reducer._on_ready if reduce else None
        for _ in range(warmup):
            step(reduce)
        ctx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = nat.launches
        e0.record()
        for _ in range(n):
            loss = step(reduce)
        e1.record()
        ctx.barrier()
        (ms,) = ctx.max_over_ranks(e0.elapsed_time(e1) / n)
        return ms, nat.launches - l0, loss

    sampler = ClockSampler(ctx.local)
    sampler.start()
    ms, launches, loss = timed(steps)
    clocks = sampler.stop()
    ms_noar = None
    if world > 1:
        ms_noar, _, _ = timed(steps, reduce=False)
        plan.on_ready = reducer._on_ready
    if profile and rank == 0:
        # issued call by call (no launch-list replay): with the per-launch events on, the weight-gradient launches stay on the main
        # stream (unet_train._on_side), so every kernel is timed alone
        plan.replay_enabled = False
        plan.eng.prof = []
        step()
        summ = plan.eng.prof_summary()
        plan.eng.prof = None
        plan.replay_enabled = True
        tot = sum(v[1] for v in summ.values())
        print("# per-op breakdown of one training step (B=%d, %s): name launches ms TFLOP/s" % (B, args.train_precision), file=sys.stderr)
        for name, (n, t, fl, nb, xf) in sorted(summ.items(), key=lambda kv: -kv[1][1]):
            print("#   %-22s %4d %9.3f %9.1f" % (name, n, t, fl / (t * 1e-3) / 1e12 if t > 0 else 0), file=sys.stderr)
        print("#   total of timed kernels %.3f ms (wall per step %.3f ms)" % (tot, ms), file=sys.stderr)
        # per-shape detail: the recorded launch lists carry no shape tags, so this one step is issued call by call
        plan.replay_enabled = False
        plan.eng.prof, plan.eng.prof_detail = [], True
        step()
        detail = plan.eng.prof_summary()
        plan.eng.prof, plan.eng.prof_detail = None, False
        plan.replay_enabled = True
        print("# per-shape breakdown of the tensor-core launches of one training step: name launches ms TFLOP/s", file=sys.stderr)
        for name, (n, t, fl, nb, xf) in sorted(detail.items(), key=lambda kv: -kv[1][1])[:90]:
            if name.startswith(("wgrad_tc", "conv_tc", "gemm_tc", "conv_taps", "attn")):
                print("#   %-42s %3d %8.3f %8.1f" % (name, n, t, fl / (t * 1e-3) / 1e12 if t > 0 else 0), file=sys.stderr)
            elif name.startswith("gn_bwd"):
                print("#   %-42s %3d %8.3f %8.1f GB/s" % (name, n, t, nb / (t * 1e-3) / 1e9 if t > 0 else 0), file=sys.stderr)
    peaks, peak_src = _peaks()
    tfl = 3 * FLOPS_PER_SAMPLE_STEP * B / (ms * 1e-3) / 1e12
    return {"workload": "configs[2]: ResDiff Cfg-A training step (q_sample + fwd + bwd + bucketed all-reduce + Adam), 128x256, dropout 0.2",
            "batch_per_gpu": B, "global_batch": B * world, "ms_per_step": ms, "value": B * world / (ms * 1e-3), "unit": "samples/s",
            "steps": steps, "dtype": args.train_precision, "gpu_launches": launches, "loss": float(loss), "clocks": clocks,
            "ms_per_step_without_allreduce": ms_noar, "allreduce_exposed_ms": None if ms_noar is None else max(0.0, ms - ms_noar),
            "allreduce_bytes": plan.gflat.numel() * 4 if world > 1 else 0,
            "parallelism": "data-parallel x%d, bucketed NCCL gradient all-reduce overlapped with backward" % world,
            "tflops": tfl, "frac_of_burst": tfl / peaks["bf16_tflops"],
            "note": "3 x forward algorithmic FLOPs (SURVEY 8d) / step time, per GPU; peak " + peak_src}


def measure_c4(ctx, args):
    """configs[3]: SRDiff UNet + RRDB-17 encoder (random init), B = 32: encoder once per batch + the reverse loop (graph replays)."""
    import wsr
    torch, dev = ctx.torch, ctx.dev
    U = wsr.sub("models.diffusion_models.srdiff.unet").UNet
    D = wsr.sub("models.diffusion_models.srdiff.srdiff_diffusion").SRDiffDiffusion
    networks = wsr.sub("models.diffusion_models.networks")
    torch.manual_seed(0)
    cfg = dict(CFG_A)
    cfg["in_channel"] = 1
    net = U(precision="bf16", **cfg)
    networks.init_weights(net, "orthogonal")
    diff = D(net.to(dev).eval(), image_height=128, image_width=256, channels=1, conditional=True).to(dev)
    diff.init_rrdb_encoder(None, lock_weights=True)
    diff.rrdb_encoder.to(dev)
    diff.set_new_noise_schedule(LINEAR_1000, dev)
    B = 32
    lr, sr = _synthetic_sr(ctx, B, pinned=False)
    lr, sr = lr.to(dev), sr.to(dev)
    plan = net.plan(B, dev)

    def set_condition():
        plan.set_condition(diff._condition(lr))          # RRDB-17 encoder forward + cond_proj: once per batch

    r = _time_loop(ctx, diff, plan, set_condition, tuple(sr.shape), args.steps, args.warmup)
    ms, pre = r["ms_per_step"], r["pre_ms"]
    fl = B * 192.24e9 / (ms * 1e-3) / 1e12
    return {"workload": "configs[3]: SRDiff UNet + RRDB-17 encoder (once per batch), 128x256, 1000-step loop, bf16", "batch_per_gpu": B,
            "ms_per_step": ms, "encoder_and_precompute_ms_per_batch": pre, "value": B / (T_FULL * ms * 1e-3 + pre * 1e-3), "unit": "samples/s",
            "tflops": fl, "flops_note": "192.24 GF per sample-step as the reference executes it (SURVEY 8d)", "steps": r["K"]}


def measure_c5(ctx, args):
    """configs[4]: 3 variables, inner 128, 16x32 -> 128x256 (8x), B = 8."""
    torch, dev = ctx.torch, ctx.dev
    net, diff = _resdiff(ctx, "bf16", image_channels=3, in_channel=15, out_channel=3, inner_channel=128)
    B = 8
    _, sr = _synthetic_sr(ctx, B, c=3, lr_hw=(16, 32), scale=8, pinned=False)
    sr = sr.to(dev)
    plan = net.plan(B, dev)
    r = _time_loop(ctx, diff, plan, lambda: plan.set_condition(sr), tuple(sr.shape), args.steps, args.warmup)
    ms, pre = r["ms_per_step"], r["pre_ms"]
    fl = B * 781.32e9 / (ms * 1e-3) / 1e12
    peaks, _ = _peaks()
    return {"workload": "configs[4]: ResDiff, 3 variables (t2m, z500, t850), inner 128, 16x32 -> 128x256, 1000-step loop, bf16", "batch_per_gpu": B,
            "ms_per_step": ms, "precompute_ms_per_batch": pre, "value": B / (T_FULL * ms * 1e-3 + pre * 1e-3), "unit": "samples/s",
            "tflops": fl, "frac_of_burst": fl / peaks["bf16_tflops"], "flops_note": "781.32 GF per sample-step (SURVEY 8d)", "steps": r["K"]}


def _free(ctx):
    import gc
    gc.collect()
    ctx.torch.cuda.empty_cache()


def run_ours(args):
    ctx = _Ctx()
    torch = ctx.torch
    world, rank = ctx.world, ctx.rank
    # ---- headline: configs[1] = batch 64 IN TOTAL, sharded over the N GPUs (SURVEY 8d C2: 64 / 32 / 16 / 8 per GPU) -> strong scaling
    total = args.batch
    B_strong = max(1, total // world)
    net, diff = _resdiff(ctx)
    main = measure_sampling(ctx, net, diff, B_strong if args.scaling == "strong" else total, args, full=True)
    # ---- the weak-scaling companion (64 samples PER GPU): identical to the headline at N = 1
    weak = None
    if world > 1 and args.scaling == "strong" and not args.no_extras:
        net._plans.clear(); _free(ctx)
        w = measure_sampling(ctx, net, diff, total, args, full=False)
        weak = {k: w[k] for k in ("batch_per_gpu", "global_batch", "ms_per_step", "value", "unit", "steps")}
        weak["scaling"] = "weak"
    elif args.scaling == "strong":
        weak = {k: main[k] for k in ("batch_per_gpu", "global_batch", "ms_per_step", "value", "unit", "steps")}
        weak["scaling"] = "weak"
        weak["note"] = "N = 1: the weak and the strong configuration coincide"
    net._plans.clear()
    del net, diff
    _free(ctx)

    extras = {}
    if not args.no_extras:
        # ---- configs[2]: the training step (NCCL all-reduce path at N > 1); every rank takes part
        try:
            # 6 warm-up steps: the first creates the gradient buffers, the second records the launch lists, the third is the first replay,
            # and at N > 1 NCCL builds its channels during the first collectives (3 warm-up steps measured 21.7 ms on 8 GPUs where the
            # standalone --workload train run of the same tree measures 19.9)
            extras["train"] = measure_train(ctx, args, steps=max(10, args.steps // 2), warmup=6)
        except Exception as e:                               # a secondary record must never take the headline down
            extras["train"] = {"error": "%s: %s" % (type(e).__name__, e)}
        _free(ctx)
        if world == 1:
            for key, fn in (("c4_srdiff_rrdb17_b32", measure_c4), ("c5_3var_inner128_b8", measure_c5)):
                try:
                    extras[key] = fn(ctx, args)
                except Exception as e:
                    extras[key] = {"error": "%s: %s" % (type(e).__name__, e)}
                _free(ctx)

    # ---- CPU baseline + the eager-PyTorch-on-this-GPU baseline (rank 0, N=1 only; after every timed region of ours) -----------
    cpu = eager = None
    if rank == 0 and world == 1 and not args.no_cpu:
        times, cores = cpu_reference_steps(args.cpu_steps, 1)
        mean = sum(times) / len(times)
        cpu = {"value": 1.0 / (T_FULL * mean), "unit": "samples/s", "cores": cores, "kind": "port",
               "sample": "B=1, %d reverse steps at 128x256 of the oracle port (fp32 torch-CPU), %.2f s/step; the port computes attention "
                         "without the reference's .contiguous() copies of the (B,N,N) matrices (39%% of the reference's CPU step in the survey), "
                         "so this baseline is FASTER than the reference's own modules would be" % (len(times), mean)}
        if not args.no_extras:
            try:
                rb = 16
                tms = gpu_eager_reference_steps(3, 2, rb, True)
                em = sum(tms) / len(tms)
                eager = {"value": rb / (T_FULL * em), "unit": "samples/s", "ms_per_step": em * 1e3, "batch": rb, "dtype": "bf16 autocast",
                         "what": "BASELINE.md section 4: the reference's algorithm (oracle port, op by op) run by eager PyTorch (cuDNN / cuBLAS) on "
                                 "this same B200 -- the 'existing implementation' on this hardware; 3 timed reverse steps",
                         "speedup_of_ours": main["value"] / (rb / (T_FULL * em))}
            except Exception as e:
                eager = {"error": "%s: %s" % (type(e).__name__, e)}

    if rank == 0:
        B = main["batch_per_gpu"]
        line = {
            "metric": "128x256 t2m SR samples/sec (1000-step loop)", "value": main["value"], "unit": "samples/s", "n_gpus": world,
            "steps": main["steps"], "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload_text(B * world), "global_batch": B * world, "batch_per_gpu": B, "T": T_FULL,
                       "step": "one reverse step over the local batch (CUDA-graph replay)", "precompute_ms_per_batch": main["precompute_ms_per_batch"],
                       "l2": "per-step activations (%.1f GB at this batch) >> 126 MB L2, no flush needed" % (0.47 * B),
                       "parallelism": "batch-sharded x%d, no collective in the loop" % world},
            "clocks": main["clocks"], "e2e": main.get("e2e"), "gpu_launches": main["launches_per_step"] * main["steps"],
            "launches_per_step": main["launches_per_step"], "roofline": main["roofline"], "cpu_baseline": cpu,
            "tc_launches_per_step": main.get("tc_launches_per_step"), "simt_launches_total": main.get("simt_launches_total"),
            "weak": weak, "train": extras.get("train"),
            "configs": {k: v for k, v in extras.items() if k != "train"} or None,
            "eager_gpu_baseline": eager,
        }
        _emit(json.dumps(line))
    ctx.close()


# ----------------------------------------------------------------------------------------------------------------------
# secondary workload: configs[2], the training step (not the headline metric; `--workload train`)
# ----------------------------------------------------------------------------------------------------------------------
def run_train(args):
    ctx = _Ctx()
    rec = measure_train(ctx, args, steps=args.steps, warmup=args.warmup, profile=args.profile_ops)
    if ctx.rank == 0:
        peaks, peak_src = _peaks()
        _emit(json.dumps({
            "metric": "ResDiff training step samples/sec (fwd+bwd+allreduce+Adam)", "value": rec["value"], "unit": "samples/s",
            "n_gpus": ctx.world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": rec["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": args.train_precision, "data": "synthetic",
            "config": {"workload": rec["workload"], "global_batch": rec["global_batch"], "parallelism": rec["parallelism"]},
            "clocks": rec["clocks"], "gpu_launches": rec["gpu_launches"], "loss": rec["loss"],
            "allreduce_exposed_ms": rec["allreduce_exposed_ms"], "ms_per_step_without_allreduce": rec["ms_per_step_without_allreduce"],
            "roofline": {"bound": "tensor", "achieved": rec["tflops"], "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": rec["frac_of_burst"],
                         "note": rec["note"], "peak_source": peak_src}}))
    ctx.close()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ref-device", default="cpu", choices=["cpu", "cuda"], help="reference arm: cpu (the contract) or the optional eager-PyTorch-on-GPU arm")
    ap.add_argument("--ref-batch", type=int, default=8)
    ap.add_argument("--ref-autocast", action="store_true")
    ap.add_argument("--batch", type=int, default=64, help="TOTAL batch sharded over the GPUs (strong, the default = configs[1]) or batch per GPU (weak)")
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"])
    ap.add_argument("--no-extras", action="store_true", help="headline record only: skip the weak / train / configs[3,4] / eager-GPU sub-records")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--e2e-budget", type=float, default=60.0, help="seconds allowed for the end-to-end public-API call")
    ap.add_argument("--cpu-steps", type=int, default=8)
    ap.add_argument("--profile-ops", action="store_true")
    ap.add_argument("--workload", default="sample", choices=["sample", "train"], help="sample = headline metric; train = configs[2]")
    ap.add_argument("--train-batch", type=int, default=4)
    ap.add_argument("--train-precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="sampling workload of --impl ours only: after the timed steps of the headline record, write the reverse loop's "
                         "image after its last timed step (all ranks' shards, float32) as DIR/x.npy; the inputs depend only on the "
                         "arguments, so two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "ours" and args.workload == "sample" and args.warmup > T_FULL - 1:
        ap.error("--warmup must leave the warm-up steps inside the %d-step chain" % T_FULL)
    if args.dump_outputs and (args.impl != "ours" or args.workload != "sample"):
        ap.error("--dump-outputs applies to the sampling workload of --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "train":
        run_train(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
