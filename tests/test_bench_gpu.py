"""bench.py on the GPU: --steps sets the number of timed steps, also at and past the end of the 1000-step chain, and --dump-outputs
writes the image the timed graph replays computed, checked against the same chain run eagerly step by step."""
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu

BATCH, WARMUP = 2, 3


def _bench(out_dir, steps, *extra):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(WARMUP),
                        "--batch", str(BATCH), "--no-extras", "--no-e2e", "--no-cpu", "--dump-outputs", str(out_dir), *extra],
                       capture_output=True, text=True, cwd=str(out_dir.parent), timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    assert sorted(os.listdir(out_dir)) == ["x.npy"]
    return json.loads(lines[0]), np.load(os.path.join(out_dir, "x.npy"))


def _eager_chain(n_steps):
    """The headline chain of bench.py (same weights, condition and Philox seed) run by n_steps eager steps; like the timed loop,
    the step counter restarts after every 1000 steps."""
    import bench
    ctx = types.SimpleNamespace(torch=torch, dev=torch.device("cuda:0"), rank=0)
    net, diff = bench._resdiff(ctx)
    _, sr = bench._synthetic_sr(ctx, BATCH, pinned=False)
    cond = sr.to(ctx.dev)
    plan = net.plan(BATCH, ctx.dev, strict_tc=False)
    plan.set_condition(cond)
    loop = diff.begin_loop(plan, tuple(cond.shape), seed=7)
    x0 = loop.x.clone()
    for i in range(n_steps):
        if i and i % bench.T_FULL == 0:
            loop.reset_counter()
        loop.step()
    torch.cuda.synchronize()
    return x0.cpu().numpy(), loop.x.cpu().numpy()


# 995 timed steps end the chain at t = 0 (then the roofline pass and --profile-ops step the loop twice more), 996 end it exactly,
# 1500 run past its end
@pytest.mark.parametrize("steps,extra", [(995, ("--profile-ops",)), (996, ()), (1500, ())])
def test_dumped_outputs_match_the_chain_run_eagerly(tmp_path, steps, extra):
    d, x = _bench(tmp_path / "out", steps, *extra)
    assert d["steps"] == steps
    assert x.shape == (BATCH, 1, 128, 256) and x.dtype == np.float32 and np.isfinite(x).all()
    # warm-up: WARMUP eager steps and one graph replay, then the timed replays
    x0, ref = _eager_chain(WARMUP + 1 + steps)
    err = float(np.linalg.norm((x - ref).astype(np.float64)) / np.linalg.norm(ref.astype(np.float64)))
    moved = float(np.linalg.norm((x - x0).astype(np.float64)) / np.linalg.norm(x0.astype(np.float64)))
    print("\n[bench] %d timed steps: dumped x vs eager chain rel-L2 %.3e, distance from the initial noise %.3e" % (steps, err, moved))
    assert err < 1e-3
    assert moved > 0.1
