"""Profiling aid (not a test): graph-timed duration of token_stack_kernel for the two token programs of a block, at batch 64 and
at 1 / 16 / 148 samples.  Run on a B200: python profiles/probe_token.py"""
import os, sys, torch
sys.path.insert(0, os.getcwd())
from keypointfusion_b200 import ops
from keypointfusion_b200.model.model import KPFusion
from keypointfusion_b200.utils import synth
dev = "cuda"
B, J = 64, 21
net = KPFusion(joint_num=J); synth.fill_state_dict(net, 0); net = net.to(dev).eval()
k = net.block1.kc()
g = torch.Generator(device=dev).manual_seed(1)
r = lambda *s: torch.randn(*s, device=dev, generator=g)
desa, jf, x, y, r3d = r(B, 3, J, 128), r(B, J, 128), r(B, J, 128), r(B, J, 128), r(B, J, 3)
def t(fn, n=10):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        for _ in range(n): fn()
    gr.replay(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5): gr.replay()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (5 * n)
for name, kw in (("tok_init", dict(desa=desa, jf=jf)), ("tok_final", dict(x=x, y=y, r3d=r3d, want_tokens=False))):
    pk = k[name]
    print(name, "L", pk.L, "F", pk.F, "cross", pk.cross, "pre", pk.pre, "ring entries", pk.n_weights)
    print("  us per launch (graph of 10)    : %.1f" % t(lambda: ops.token_stack(pk, **kw)))
    for Bs in (1, 16, 148):
        kw2 = {kk: (v[:Bs] if Bs <= B else v.repeat((Bs + B - 1) // B, *[1] * (v.dim() - 1))[:Bs]) if torch.is_tensor(v) else v for kk, v in kw.items()}
        print("     B=%d: %.1f us" % (Bs, t(lambda: ops.token_stack(pk, **kw2))))
