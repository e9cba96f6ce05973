"""Profiling aid: throughput when consecutive STEPS (independent batches of 64) are kept in flight on several streams.
Prints us per step for 1, 2 and 3 streams."""
import os, sys, torch
sys.path.insert(0, os.getcwd())
from keypointfusion_b200.dataloader.loader import loader
from keypointfusion_b200.model.model import KPFusion
from keypointfusion_b200.runtime import GraphedFusionPath
from keypointfusion_b200.utils import synth
dev = "cuda"
net = KPFusion(joint_num=21); synth.fill_state_dict(net, 0); net = net.to(dev).eval()
sets = []
for s in range(4):
    inp = synth.make_inputs(64, 128, 21, 128, seed=20 + s, depth_noise=0.35)
    d = {kk: inp[kk].to(dev) for kk in GraphedFusionPath.KEYS}
    for kk in ("img_feat", "img_feat_rgb", "img_offset"): d[kk] = d[kk].bfloat16()
    sets.append(d)
L = loader(img_size=128)
graphs = [GraphedFusionPath(net, L, d, bind=True) for d in sets]
for nstream in (1, 2, 3):
    streams = [torch.cuda.Stream() for _ in range(nstream)]
    def run(n):
        for i in range(n):
            with torch.cuda.stream(streams[i % nstream]):
                graphs[i % 4].graph.replay()
    run(8); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in streams: s.wait_event(e0)
    run(40)
    for s in streams: torch.cuda.current_stream().wait_stream(s)
    e1.record(); torch.cuda.synchronize()
    print(f"streams {nstream}: {e0.elapsed_time(e1) * 1e3 / 40:7.1f} us per step", flush=True)
