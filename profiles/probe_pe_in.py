"""Profiling aid: the point stage loading staged tiles (block 2's launch), for profiles/srcstalls.sh point_embed <tag> profiles/probe_pe_in.py"""
import os, sys, torch
sys.path.insert(0, os.getcwd())
exec(open("profiles/probe_kernels.py").read().split("def t(fn")[0])
stage = ops.point_embed_stage(B, pcl.shape[1], dev)
ops.point_embed(featT, idx, close, pcl, joint, k["pe_wmat"], k["pe_wvec"], 0.8, order=order, stage_out=stage)
for _ in range(12):
    ops.point_embed(featT, idx, close, pcl, joint, k["pe_wmat"], k["pe_wvec"], 0.8, order=order, stage_in=stage)
torch.cuda.synchronize()
