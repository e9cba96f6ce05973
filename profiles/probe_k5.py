"""Profiling aid: K5 (spatial_aggregate_tc) alone at the benchmark shape, graph-timed.
profiles/srcstalls.sh spatial_aggregate r2_k5 profiles/probe_k5.py"""
import os, sys, torch
sys.path.insert(0, os.getcwd())
from keypointfusion_b200 import ops
from keypointfusion_b200.model.model import KPFusion
from keypointfusion_b200.utils import synth
dev = "cuda"
B = 64
net = KPFusion(joint_num=21); synth.fill_state_dict(net, 0); net = net.to(dev).eval()
b = net.block1; k = b.kc()
inp = synth.make_inputs(B, 128, 21, 128, seed=5)
c = {kk: v.to(dev) for kk, v in inp.items()}
rgb = c["img_feat_rgb"].bfloat16()
r3d = (torch.rand(B, 21, 3, device=dev) - 0.5)
fn = lambda: ops.spatial_aggregate_tc(rgb, r3d, c["img"][:, :, ::4, ::4], c["center"], c["M"], c["cube"], c["cam"], k["wa_packed"], b.atten_spatial.bias,
                                      b.weight_dis, b.fc_spatial2joint_feature.weight, b.fc_spatial2joint_feature.bias)
for _ in range(10): fn()
torch.cuda.synchronize()
g = torch.cuda.CUDAGraph()
with torch.cuda.graph(g):
    for _ in range(10): fn()
g.replay(); torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(5): g.replay()
e1.record(); torch.cuda.synchronize()
print("K5 us per launch: %.1f" % (e0.elapsed_time(e1) * 1e3 / 50))
