"""Profiling aid (not a test): graph-timed point stage (plain, storing and loading staged tiles) and DESA at batch 64.
Run on a B200: python profiles/probe_kernels.py"""
import os, sys, torch, numpy as np
sys.path.insert(0, os.getcwd())
from keypointfusion_b200 import ops
from keypointfusion_b200.model.model import KPFusion
from keypointfusion_b200.utils import synth
dev = "cuda"
B = 64
net = KPFusion(joint_num=21); synth.fill_state_dict(net, 0); net = net.to(dev).eval()
blk = net.block1; k = blk.kc()
inp = synth.make_inputs(B, 128, 21, 128, seed=5)
c = {kk: v.to(dev) for kk, v in inp.items()}
pcl, _ = ops.getpcl(c["img"], c["center"], c["cube"], c["M"], c["cam"], seed=2)
order = ops.spatial_order(pcl, c["center"], c["M"], c["cube"], c["cam"], 128, 32)
close, _, idx = ops.img2pcl_index(pcl, c["img"], c["center"], c["M"], c["cube"], c["cam"], 128, 4, fs=32, want_i64=False, want_i32=True, order=order)
joint = pcl[:, ::48][:, :21].contiguous() + 0.01
featT = ops.repack_features(c["img_feat"].bfloat16(), c["img_feat_rgb"].bfloat16(), c["img_offset"][:, 84:].bfloat16())
def t(fn, n=10):
    """us per call, timed as a CUDA graph of n calls (no host launch overhead inside the timed region)"""
    for _ in range(3): fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(n): fn()
    g.replay(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5): g.replay()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (5 * n)
e, acc, ms = ops.point_embed(featT, idx, close, pcl, joint, k["pe_wmat"], k["pe_wvec"], 0.8, order=order)
print("point_embed us", t(lambda: ops.point_embed(featT, idx, close, pcl, joint, k["pe_wmat"], k["pe_wvec"], 0.8, order=order)))
stage = ops.point_embed_stage(B, pcl.shape[1], dev)
print("point_embed + stage_out us", t(lambda: ops.point_embed(featT, idx, close, pcl, joint, k["pe_wmat"], k["pe_wvec"], 0.8, order=order, stage_out=stage)))
print("point_embed from stage_in us", t(lambda: ops.point_embed(featT, idx, close, pcl, joint, k["pe_wmat"], k["pe_wvec"], 0.8, order=order, stage_in=stage)))
print("desa us", t(lambda: ops.desa_fused(e, acc, ms, pcl, joint, k["ds_wmat"], k["ds_wvec"], blk.FA.radius, 64)))
