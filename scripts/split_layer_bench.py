"""CUDA-event timing of the ResNet-50 trunk's layer shapes on the split engine (rf_conv2d_nhwc engine 4) at config-2 sizes:
the 8 images of one pair (7 source scales + target).  One line per distinct layer shape, L2 flushed between launches, and the
trunk total weighted by how often each shape occurs.
Usage: python scripts/split_layer_bench.py [reps]"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ransac_flow_b200 as rf  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 7
dev = "cuda"
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
L1 = [(240, 320), (200, 264), (160, 212), (120, 160), (100, 132), (80, 104), (60, 80), (120, 160)]
L2 = [((h + 1) // 2, (w + 1) // 2) for h, w in L1]
L3 = [((h + 1) // 2, (w + 1) // 2) for h, w in L2]

# name, input grid, cin, cout, k, stride, residual, occurrences in the trunk
LAYERS = [
    ("l1 c1 first 1x1 64->64", L1, 64, 64, 1, 1, False, 1),
    ("l1 c2 3x3 64->64", L1, 64, 64, 3, 1, False, 3),
    ("l1 ds 1x1 64->256", L1, 64, 256, 1, 1, False, 1),
    ("l1 c3+res 1x1 64->256", L1, 64, 256, 1, 1, True, 3),
    ("l1 c1 1x1 256->64", L1, 256, 64, 1, 1, False, 2),
    ("l2 c1 first 1x1 256->128", L1, 256, 128, 1, 1, False, 1),
    ("l2 c2 3x3/2 128->128", L1, 128, 128, 3, 2, False, 1),
    ("l2 ds 1x1/2 256->512", L1, 256, 512, 1, 2, False, 1),
    ("l2 c3+res 1x1 128->512", L2, 128, 512, 1, 1, True, 4),
    ("l2 c1 1x1 512->128", L2, 512, 128, 1, 1, False, 3),
    ("l2 c2 3x3 128->128", L2, 128, 128, 3, 1, False, 3),
    ("l3 c1 first 1x1 512->256", L2, 512, 256, 1, 1, False, 1),
    ("l3 c2 3x3/2 256->256", L2, 256, 256, 3, 2, False, 1),
    ("l3 ds 1x1/2 512->1024", L2, 512, 1024, 1, 2, False, 1),
    ("l3 c3+res 1x1 256->1024", L3, 256, 1024, 1, 1, True, 6),
    ("l3 c1 1x1 1024->256", L3, 1024, 256, 1, 1, False, 5),
    ("l3 c2 3x3 256->256", L3, 256, 256, 3, 1, False, 5),
]


def split_ragged(sizes, c, g):
    P = sum(h * w for h, w in sizes)
    return rf.ops.Ragged(rf.ops.to_split(torch.randn(P, c, generator=g, device=dev)), sizes)


def main():
    g = torch.Generator(device=dev).manual_seed(0)
    total = 0.0
    for name, sizes, cin, cout, k, stride, res, count in LAYERS:
        x = split_ragged(sizes, cin, g)
        ws = rf.ops.to_split(torch.randn(cout, k * k * cin, generator=g, device=dev) / np.sqrt(k * k * cin))
        bias = torch.randn(cout, generator=g, device=dev)
        osz = [((h - 1) // stride + 1, (w - 1) // stride + 1) for h, w in sizes]
        r = split_ragged(osz, cout, g) if res else None

        def run():
            return rf.ops.conv2d(x, None, bias, cout, k, stride, k // 2, True, r, rf.ops.ENGINE_SPLIT, ws)

        for _ in range(2):
            run()
        ts = []
        for _ in range(reps):
            flush.zero_()
            torch.cuda._sleep(1000000)          # ~0.5 ms: the host queues the launch behind it, so the events bracket the kernel alone
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            run()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) * 1e3)
        med = float(np.median(ts))
        total += med * count
        print("%-28s x%d  median %7.1f us  min %7.1f us" % (name, count, med, min(ts)))
    print("trunk convolutions (weighted): %.1f us" % total)
    # conv3 + down-sampling branch as one dual-input GEMM (replaces "ds" + "c3+res" of a stage's first block)
    for name, s1, s2, c1, c2, cout, stride2 in [("l1.0 c3 + ds fused 64|64->256", L1, L1, 64, 64, 256, 1),
                                                ("l2.0 c3 + ds/2 fused 128|256->512", L2, L1, 128, 256, 512, 2),
                                                ("l3.0 c3 + ds/2 fused 256|512->1024", L3, L2, 256, 512, 1024, 2)]:
        x1, x2 = split_ragged(s1, c1, g), split_ragged(s2, c2, g)
        ws = rf.ops.to_split(torch.randn(cout, c1 + c2, generator=g, device=dev) / np.sqrt(c1 + c2))
        bias = torch.randn(cout, generator=g, device=dev)
        for _ in range(2):
            rf.ops.conv1x1_dual_split(x1, x2, stride2, ws, bias, True)
        ts = []
        for _ in range(reps):
            flush.zero_()
            torch.cuda._sleep(1000000)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            rf.ops.conv1x1_dual_split(x1, x2, stride2, ws, bias, True)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) * 1e3)
        print("%-36s median %7.1f us  min %7.1f us" % (name, float(np.median(ts)), min(ts)))


if __name__ == "__main__":
    main()
