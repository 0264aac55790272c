"""Profiling helper: one 3x3 conv with and without the fused GroupNorm input.
usage: python tools/prof_fuse.py N Cin Cout H W [reps]"""
import math
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import wsr

nat = wsr.pkg.native
em = wsr.sub("engine")


def main():
    N, Cin, Cout, H, W = [int(v) for v in sys.argv[1:6]]
    reps = int(sys.argv[6]) if len(sys.argv) > 6 else 5
    dev = torch.device("cuda:0")
    eng = em.Engine(dev, "bf16")
    torch.manual_seed(0)
    arena = em.StatsArena()
    x = eng.new_act(N, H, W, Cin, stats=arena)
    arena2 = em.StatsArena()
    y = eng.new_act(N, H, W, Cout, stats=arena2)
    arena.finalize(dev); arena2.finalize(dev)
    x.buf.copy_(torch.randn_like(x.buf, dtype=torch.float32))
    eng.gn_stats(x)
    w = torch.randn(Cout, Cin, 3, 3, device=dev) / math.sqrt(Cin * 9)
    pc = eng.pack_conv(w, torch.randn(Cout, device=dev))
    gamma, beta = torch.ones(Cin, device=dev), torch.zeros(Cin, device=dev)
    tab = eng.empty((N, Cin, 2), torch.float32)
    eng.gn_finalize(x, gamma, beta, 32, tab)
    a = eng.new_act(N, H, W, Cin)

    def timed(fn):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(reps):
            fn()
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) / reps

    t_plain = timed(lambda: eng.conv(a, pc, y))
    t_gn = timed(lambda: eng.gn_apply(x, gamma, beta, 32, nat.ACT_SWISH, a))
    t_fused = timed(lambda: eng.conv(x, pc, y, gn=(tab, nat.ACT_SWISH)))
    fl = 2.0 * N * H * W * Cout * Cin * 9
    print("conv %d->%d %dx%d N=%d: plain %.3f ms (%.0f TF/s), gn_apply %.3f ms, fused %.3f ms (%.0f TF/s)" % (
        Cin, Cout, H, W, N, t_plain, fl / t_plain / 1e9, t_gn, t_fused, fl / t_fused / 1e9))


if __name__ == "__main__":
    main()
