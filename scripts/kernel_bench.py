"""Stand-alone launches of the hot kernels at config-2 shapes (for ncu captures and CUDA-event timing).
Usage: python scripts/kernel_bench.py {corr|corr2|ransac|conv|c64} [reps]"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ransac_flow_b200 as rf  # noqa: E402
import synthdata as synth  # noqa: E402

which = sys.argv[1] if len(sys.argv) > 1 else "corr"
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
dev = "cuda"
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def timed(fn):
    for _ in range(2):
        fn()
    ts = []
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.mean(ts)), float(np.min(ts))


if which == "corr":
    g = torch.Generator(device="cpu").manual_seed(0)
    A = torch.nn.functional.normalize(torch.rand(13065, 1024, generator=g), dim=1).to(dev)
    B = torch.nn.functional.normalize(torch.rand(1200, 1024, generator=g), dim=1).to(dev)
    for prec in (2, 1, 0):
        m, mn = timed(lambda: rf.ops.corr_mutual_nn(A, B, prec))
        print("corr_mutual_nn precision=%d: mean %.1f us, min %.1f us -> %.1f TFLOP/s algorithmic" % (prec, m * 1e3, mn * 1e3, 32.108544 / m))
elif which == "corr2":                  # precision 2 only
    g = torch.Generator(device="cpu").manual_seed(0)
    A = torch.nn.functional.normalize(torch.rand(13065, 1024, generator=g), dim=1).to(dev)
    B = torch.nn.functional.normalize(torch.rand(1200, 1024, generator=g), dim=1).to(dev)
    m, mn = timed(lambda: rf.ops.corr_mutual_nn(A, B, 2))
    i1, i2, n = rf.ops.corr_mutual_nn(A, B, 2)
    print("corr_mutual_nn precision=2 (%d launches): mean %.1f us, min %.1f us -> %.1f TFLOP/s algorithmic, %d pairs"
          % (rf._lib.lib.rf_corr_mutual_nn_launches(2), m * 1e3, mn * 1e3, 32.108544 / m, int(n)))
elif which == "ransac":
    m1, m2, _ = synth.make_matches(1, 636, 0.6)
    t1, t2 = torch.from_numpy(m1).to(dev), torch.from_numpy(m2).to(dev)
    for nb in (1000, 50000):
        s = torch.from_numpy(synth.draw_samples(1, 636, nb)).to(dev)
        m, mn = timed(lambda: rf.ops.ransac_homography(t1, t2, s, 0.05))
        print("ransac nbIter=%d M=636: mean %.1f us, min %.1f us" % (nb, m * 1e3, mn * 1e3))
elif which == "c64":
    sizes = [(240, 320), (200, 264), (160, 212), (120, 160), (100, 132), (80, 104), (60, 80), (120, 160)]   # layer1 grids of config 2
    P = sum(h * w for h, w in sizes)
    x = rf.ops.Ragged(torch.randn(P, 64, device=dev), sizes)
    w = torch.randn(64, 64, 3, 3, device=dev) / 24
    fc = rf.model.FoldedConv(w, None, 1)
    m, mn = timed(lambda: fc(x, relu=True, engine=1))
    fl = 2.0 * P * 64 * 64 * 9 / 1e9
    print("conv3x3 64->64 on %d px: mean %.1f us -> %.1f TFLOP/s" % (P, m * 1e3, fl / m))
else:
    sizes = [(60, 80), (50, 66), (40, 53), (30, 40), (25, 33), (20, 26), (15, 20), (30, 40)]      # layer3 grids of config 2
    P = sum(h * w for h, w in sizes)
    x = rf.ops.Ragged(torch.randn(P, 256, device=dev), sizes)
    w = torch.randn(256, 256, 3, 3, device=dev) / 48
    fc = rf.model.FoldedConv(w, None, 1)
    for eng in (1, 0):
        m, mn = timed(lambda: fc(x, relu=True, engine=eng))
        fl = 2.0 * P * 256 * 256 * 9 / 1e9
        print("conv3x3 256->256 on %d px, engine %d: mean %.1f us -> %.1f TFLOP/s" % (P, eng, m * 1e3, fl / m))
torch.cuda.synchronize()
