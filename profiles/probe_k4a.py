"""Tuning aid (not a test): K4a (offset2joint_weight, bf16 fast path) alone, graph-timed over rotating input sets, at batch 64 and 512.
The launcher picks 3 or 7 joints per CTA by grid size (geometry.cu): batch 64 runs the 3-joint kernel, batch 512 the 7-joint one."""
import os, sys, torch
sys.path.insert(0, os.getcwd())
from keypointfusion_b200 import ops
dev = "cuda"
J, H = 21, 32
def t(B, nsets):
    maps = [torch.randn(B, 5 * J, H, H, device=dev).bfloat16() for _ in range(nsets)]
    imgs = [torch.rand(B, 1, 128, 128, device=dev) for _ in range(nsets)]
    for m, im in zip(maps, imgs): ops.offset2joint_weight(m, im, 0.8)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(4):
            for m, im in zip(maps, imgs): ops.offset2joint_weight(m, im, 0.8)
    g.replay(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5): g.replay()
    e1.record(); torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / (5 * 4 * nsets)
    alg = B * (5 * J * H * H * 2 + H * H * 4)
    return us, alg / us / 1e3
print("B=64: %.2f us %.0f GB/s | B=512: %.2f us %.0f GB/s" % (*t(64, 12), *t(512, 3)))
