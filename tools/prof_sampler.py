"""Fewer-step samplers on one GPU, two measurements (JSON lines on stdout), ResDiff Cfg-A, 128x256, B = 64, bf16, graph replay:

  1. ms per graph-replayed step of the ddpm, ddim and dpmpp2m loops, alternated in the same process, ``--reps`` repetitions.  The ddim
     and dpmpp2m loops run on all T timesteps here so that a window of steps never reaches the end of the chain; a step's cost does not
     depend on S.  DPM-Solver++(2M) adds the x0 history: 8 bytes per pixel and step.
  2. whole ``super_resolution`` calls (condition precompute, level table, initial noise, graph capture, every step; host clock around a
     device synchronise), after one warm-up call per sampler: samples/s of DDPM-1000, DDIM-50 and DPM-Solver++(2M)-20, alternated,
     ``--reps`` repetitions; ``vs_ddpm`` compares the fastest repetitions.

    python tools/prof_sampler.py [--steps 30] [--reps 2]
"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench import CFG_A, LINEAR_1000  # noqa: E402
from prof_ensemble import DEV, _events, _gpu, _resdiff  # noqa: E402

B = 64
CALLS = (("ddpm", None), ("ddim", 50), ("dpmpp2m", 20))


def _step_ms(diff, name, cond, steps):
    diff.set_sampler(name, None)
    plan = diff._plan(B, DEV)
    plan.set_condition(cond)
    loop = diff.begin_loop(plan, tuple(cond.shape), seed=1)
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


def step_times(diff, cond, steps, reps):
    rows = {name: [] for name, _ in CALLS}
    for _ in range(reps):                                       # alternated: the three loops see the same box state
        for name in rows:
            rows[name].append(_step_ms(diff, name, cond, steps))
    return {k: {"ms_per_step": v, "median": sorted(v)[len(v) // 2]} for k, v in rows.items()}


def whole_calls(diff, cond, reps):
    x_in = {"SR": cond}
    for name, S in CALLS[1:]:                                   # warm-up: plan, level tables, first launches (ddim's kernels are ddpm's)
        diff.set_sampler(name, S)
        diff.super_resolution(x_in)
    torch.cuda.synchronize()
    out = {}
    for _ in range(reps):                                       # alternated
        for name, S in CALLS:
            diff.set_sampler(name, S)
            t0 = time.perf_counter()
            diff.super_resolution(x_in)
            torch.cuda.synchronize()
            out.setdefault("%s-%d" % (name, S or diff.num_timesteps), []).append(time.perf_counter() - t0)
    base = min(out["ddpm-%d" % diff.num_timesteps])
    return {k: {"seconds": v, "samples_per_s": [B / x for x in v], "vs_ddpm": base / min(v)} for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--reps", type=int, default=2)
    a = ap.parse_args()
    gpu = _gpu()
    diff = _resdiff()
    diff.sample_seed = 1
    cond = torch.randn((B, 1, CFG_A["image_height"], CFG_A["image_width"]), device=DEV)
    print(json.dumps({"measure": "step", "gpu": gpu, "batch": B, "schedule": LINEAR_1000, "result": step_times(diff, cond, a.steps, a.reps)}),
          flush=True)
    print(json.dumps({"measure": "whole_call", "gpu": gpu, "batch": B, "result": whole_calls(diff, cond, a.reps)}), flush=True)


if __name__ == "__main__":
    main()
