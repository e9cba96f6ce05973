"""What evaluating on the device costs, on one GPU at batch 64 (21 joints, the five joint sets of the fusion path: offset, r3d_1,
r2d_1, r3d_2, r2d_2; PCK thresholds 0..50 mm).

  1. ms per step with six steps in flight (OverlappedSteps, one graph bound to each of six resident input sets, ops.K5_SPLIT = 1
     as bench.py sets it): GraphedEvalPath (fusion path + stage joints + kpf_eval_accumulate in the same graph) against
     GraphedFusionPath, alternated in the same process, `--repeats` times each.
  2. kpf_eval_accumulate alone at S = 5, B = 64: CUDA events around a captured graph of 50 launches (device time per launch), and
     around 200 eager launches (host launch cost included); for comparison kpf_eval_errors on the five sets, one after the other
     (a captured graph of 10 x 5 launches).
  3. The reference's way for comparison (train.py:330-396): per step and joint set, eval_errors, .cpu() of the [B,J] errors, a numpy
     accumulation of sums and a histogram; host clock, samples/s.
Both paths compute the same joints (checked).  The six input sets (~300 MB) exceed the 126 MB L2.

    python profiles/bench_eval.py --out profiles/bench_eval.json
prints one JSON line and writes it to --out."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

B, J, N_SETS, S_OV = 64, 21, 6, 6


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as ex:
        q = f"unavailable ({type(ex).__name__})"
    return {"gpu": name, "power_limit_and_max_sm_clock": q}


def inputs(seed):
    from keypointfusion_b200.utils import synth
    inp = synth.make_inputs(B, 128, J, 128, seed=seed, depth_noise=0.35)
    for k in ("img_feat", "img_feat_rgb", "img_offset"):
        inp[k] = inp[k].bfloat16()
    inp.pop("img_rgb")
    rs = np.random.RandomState(seed)
    inp["gt"] = torch.from_numpy(rs.uniform(-0.5, 0.5, (B, J, 3)).astype(np.float32))
    inp["valid"] = torch.ones(B, dtype=torch.uint8)
    return {k: v.cuda() for k, v in inp.items()}


def overlapped_ms(ov, steps, warmup):
    for _ in range(warmup):
        ov.submit()
    ov.join()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ov.fork()
    for _ in range(steps):
        ov.submit()
    ov.join()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=120)
    ap.add_argument("--warmup", type=int, default=24)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_eval.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_eval.py needs a CUDA device"
    from keypointfusion_b200 import ops
    from keypointfusion_b200.dataloader.loader import loader
    from keypointfusion_b200.evaluation import DEFAULT_STAGES, Evaluator
    from keypointfusion_b200.model.model import KPFusion
    from keypointfusion_b200.runtime import GraphedEvalPath, GraphedFusionPath, OverlappedSteps
    from keypointfusion_b200.utils import synth

    net = KPFusion(joint_num=J)
    synth.fill_state_dict(net, seed=0)
    net = net.cuda().eval()
    ldr = loader(img_size=128)
    ops.K5_SPLIT = 1
    sets = [inputs(2000 + s) for s in range(N_SETS)]
    ev = Evaluator(J)
    plain = OverlappedSteps([GraphedFusionPath(net, ldr, d, bind=True) for d in sets], S_OV)
    evald = OverlappedSteps([GraphedEvalPath(net, ldr, d, evaluator=ev, bind=True) for d in sets], S_OV)
    for p, q in zip(plain.paths, evald.paths):
        p.graph.replay()
        q.graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(p.out["joints"], q.out["joints"]), "the evaluated path must compute the same joints"

    # 1. alternating A/B, six steps in flight
    ms = {"GraphedFusionPath": [], "GraphedEvalPath": []}
    with torch.no_grad():
        for _ in range(a.repeats):
            ms["GraphedFusionPath"].append(overlapped_ms(plain, a.steps, a.warmup))
            ms["GraphedEvalPath"].append(overlapped_ms(evald, a.steps, a.warmup))
    med = {k: float(np.median(v)) for k, v in ms.items()}

    # 2. the accumulate kernel alone
    rs = np.random.RandomState(7)
    gt = torch.from_numpy(rs.uniform(-0.5, 0.5, (B, J, 3)).astype(np.float32)).cuda()
    pred = (gt[None] + torch.from_numpy(rs.normal(0, 0.02, (5, B, J, 3)).astype(np.float32)).cuda()).contiguous()
    cube = torch.full((B, 3), 250.0, device="cuda")
    valid = torch.ones(B, dtype=torch.uint8, device="cuda")
    acc_ev = Evaluator(J, device="cuda")
    thr = list(acc_ev.thresholds)
    for _ in range(3):
        ops.eval_accumulate(acc_ev.acc, pred, gt, cube, valid, thr)
    torch.cuda.synchronize()
    n_graph = 50
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s), torch.cuda.graph(g, stream=s):
        for _ in range(n_graph):
            ops.eval_accumulate(acc_ev.acc, pred, gt, cube, valid, thr)
    torch.cuda.current_stream().wait_stream(s)
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 20
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    kernel_us = e0.elapsed_time(e1) * 1e3 / (reps * n_graph)
    g_err = torch.cuda.CUDAGraph()   # the same per-sample code without accumulation: kpf_eval_errors on each of the five sets
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            [ops.eval_errors(pred[k], gt, cube) for k in range(5)]
        with torch.cuda.graph(g_err, stream=s):
            for _ in range(10):
                [ops.eval_errors(pred[k], gt, cube) for k in range(5)]
    torch.cuda.current_stream().wait_stream(s)
    g_err.replay()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        g_err.replay()
    e1.record()
    torch.cuda.synchronize()
    errors_us = e0.elapsed_time(e1) * 1e3 / (reps * 10)
    n_eager = 200
    e0.record()
    for _ in range(n_eager):
        ops.eval_accumulate(acc_ev.acc, pred, gt, cube, valid, thr)
    e1.record()
    torch.cuda.synchronize()
    eager_us = e0.elapsed_time(e1) * 1e3 / n_eager

    # 3. the reference-style loop on the same joint sets: per set eval_errors, .cpu(), numpy sums and histogram
    thr_np = np.asarray(thr, np.float32)
    sums = np.zeros((5, 2, J))
    hist = np.zeros((5, 2, len(thr) + 1), np.int64)

    def host_step():
        for k in range(5):
            err, pa = ops.eval_errors(pred[k], gt, cube)
            e, p = err.cpu().numpy(), pa.cpu().numpy()
            for i, x in enumerate((e, p)):
                sums[k, i] += x.sum(0)
                hist[k, i] += np.bincount(np.searchsorted(thr_np, x.ravel(), side="left"), minlength=len(thr) + 1)
    for _ in range(5):
        host_step()
    n_host = 200
    t0 = time.perf_counter()
    for _ in range(n_host):
        host_step()
    host_s = (time.perf_counter() - t0) / n_host

    line = {
        "what": "device evaluation cost at batch 64, 21 joints, 5 joint sets, 51 PCK thresholds",
        **gpu_info(),
        "ms_per_step_6_in_flight": {k: [round(x, 4) for x in v] for k, v in ms.items()},
        "median_ms_per_step": {k: round(v, 4) for k, v in med.items()},
        "eval_overhead_pct": round(100.0 * (med["GraphedEvalPath"] / med["GraphedFusionPath"] - 1.0), 2),
        "samples_per_s": {k: round(B / (v / 1e3), 1) for k, v in med.items()},
        "eval_accumulate_us": {"device_per_launch_in_graph": round(kernel_us, 2), "eager_per_call": round(eager_us, 2), "S": 5, "B": B},
        "eval_accumulate_samples_per_s_in_graph": round(B / (kernel_us / 1e6), 1),
        "eval_errors_us_5_sets_in_graph": round(errors_us, 2),
        "reference_style_loop": {"ms_per_step": round(host_s * 1e3, 3), "samples_per_s": round(B / host_s, 1),
                                 "per_step": "5 x (eval_errors + .cpu() of err and pa + numpy sums and histogram)"},
        "stages": list(DEFAULT_STAGES), "steps": a.steps, "warmup": a.warmup, "repeats": a.repeats, "steps_in_flight": S_OV,
    }
    print(json.dumps(line))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(line, indent=1) + "\n")


if __name__ == "__main__":
    main()
