"""Times single tcgen05 convolution shapes as CUDA-graph replays (no host overhead in the timed region), for calibrating the
column-tile / split-K cost model of csrc/gemm_tc.cu.
usage: python tools/prof_conv.py [B]"""
import math
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import wsr

nat = wsr.pkg.native
eng_mod = wsr.sub("engine")
dev = torch.device("cuda:0")
B = int(sys.argv[1]) if len(sys.argv) > 1 else 8
SHAPES = [  # Cin, Cout, H, W, k, stride, up, Cin2
    (512, 512, 8, 16, 3, 1, False, 0), (1024, 512, 8, 16, 3, 1, False, 0), (512, 512, 8, 16, 3, 1, False, 1024), (512, 512, 8, 16, 1, 1, False, 0),
    (512, 512, 16, 32, 3, 1, False, 0), (1024, 512, 16, 32, 3, 1, False, 0), (512, 512, 16, 32, 1, 1, False, 0), (512, 1024, 16, 32, 1, 1, False, 0),
    (256, 256, 32, 64, 3, 1, False, 0), (768, 256, 32, 64, 3, 1, False, 0),
]
if os.environ.get("WSR_PROF_SHAPES"):      # comma-separated indices into SHAPES (ncu captures of one shape)
    SHAPES = [SHAPES[int(i)] for i in os.environ["WSR_PROF_SHAPES"].split(",")]
eng = eng_mod.Engine(dev, "bf16")
R = int(os.environ.get("WSR_PROF_REPS", "20"))
for (Cin, Cout, H, W, k, stride, up, Cin2) in SHAPES:
    torch.manual_seed(0)
    x = eng.new_act(B, H, W, Cin); x.buf.normal_()
    w = torch.randn(Cout, Cin, k, k, device=dev) / math.sqrt(Cin * k * k)
    pc = eng.pack_conv(w, torch.zeros(Cout, device=dev))
    arena = eng_mod.StatsArena()
    OH, OW = H // stride, W // stride
    # rotate over several output / input buffers so that consecutive replays do not find everything in L2
    ys = [eng.new_act(B, OH, OW, Cout, stats=arena) for _ in range(4)]
    arena.finalize(dev)
    kw = {}
    if Cin2:
        x2 = eng.new_act(B, H, W, Cin2); x2.buf.normal_()
        w2 = torch.randn(Cout, Cin2, 1, 1, device=dev) / math.sqrt(Cin2)
        kw = dict(x2=x2, w2=eng.pack_conv(w2, None))
    rv = torch.randn(B, Cout, device=dev)
    def run():
        for i in range(R):
            eng.conv(x, pc, ys[i % 4], stride=stride, rowvec=rv.data_ptr(), rowvec_ld=Cout, **kw)
    run()
    cfg = nat.call("wsr_debug_last_tc_config")
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        run()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / (5 * R)
    fl = 2 * B * OH * OW * Cout * (k * k * Cin + Cin2)
    print("B=%d %4d->%4d k%d s%d %3dx%-3d +%4d : bn=%3d S=%d  %7.2f us  %7.1f TFLOP/s" % (B, Cin, Cout, k, stride, H, W, Cin2, (cfg >> 8) & 0xfff, (cfg & 0xff) + 100 * (cfg >> 20), us, fl / us / 1e6), flush=True)
