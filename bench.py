#!/usr/bin/env python
"""bench.py -- fusion-path throughput (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--batch B] [--no-cpu-baseline] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic RGB-D crops: depth crop -> point cloud (K1) ->
initial joints (K4a) -> nearest-cell indices (K2) -> 2 x Block_KPFusion -> final joints, fed with bf16 backbone feature
maps of the default config (BASELINE.json configs[1]: fusion path only, batch 64, bf16, 1 x B200).  With N > 1 every
rank runs its own batch (weak scaling; the path shards by sample) and the per-sample joints are all-gathered over NCCL,
the one exchange step the path has (SURVEY.md 8e).

Prints ONE JSON line.  `--impl reference` times the reference algorithm's CPU implementation (the oracle port: the
Python reference itself cannot travel to the GPU box) on the host cores for the same metric.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from keypointfusion_b200.utils import synth  # noqa: E402

J, C, S, N_PTS = 21, 128, 128, 1024
H = S // 4
# SURVEY.md 8d: algorithmic bytes / FLOPs per sample of the whole fusion path (bf16 features)
PATH_BYTES_PER_SAMPLE = (2 * C + 5 * J) * H * H * 2 + S * S * 4 + 76 + 4 * J * 12 + 2 * J * H * H * 4 + 2 * J * C * 4
PATH_FLOPS_PER_SAMPLE = 871.5e6


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def build_net(device):
    from keypointfusion_b200.model.model import KPFusion
    net = KPFusion(joint_num=J)
    synth.fill_state_dict(net, seed=0)
    return net.to(device).eval()


DEPTH_NOISE = float(os.environ.get("KPF_DEPTH_NOISE", "0.35"))   # synthetic depth noise (normalised; x125 mm), see utils/synth.py


def host_inputs(B, seed):
    inp = synth.make_inputs(B, S, J, C, seed=seed, depth_noise=DEPTH_NOISE)
    for k in ("img_feat", "img_feat_rgb", "img_offset"):
        inp[k] = inp[k].bfloat16()
    inp.pop("img_rgb")
    return inp


def run_step(net, loader, d, seed):
    """One pass of the hot path; returns what runtime.GraphedFusionPath returns: the final joints [B,J,3] (normalised xyz) as
    "joints", forward_path's results and spatial weights, the sampled point cloud."""
    from keypointfusion_b200 import ops
    pcl, _ = ops.getpcl(d["img"], d["center"], d["cube"], d["M"], d["cam"], N_PTS, seed=seed)
    res, sw, _ = net.forward_path(d["img_offset"], d["img_feat"], None, d["img_feat_rgb"], d["img"], pcl, loader, d["center"], d["M"],
                                  d["cube"], d["cam"], 0.8)
    return dict(joints=res[-1], result=res, spatial_weight=sw, pcl=pcl)


DUMP_LIMIT = 64 * 10**6   # bytes --dump-outputs writes at most


def dump_outputs(out, directory):
    """Write what one step of the path returned (a run_step / GraphedFusionPath dict) as DIR/<name>.npy in float32: the joints of
    every block (r3d_<k>, r2d_<k>; r2d of the last block are the final joints), their spatial weights and the sampled point cloud,
    all [B, ...].  Above DUMP_LIMIT only a fixed, seeded subset of the samples is written, the same samples for every array."""
    parts = out["chains"] if "chains" in out else [(out["result"], out["spatial_weight"], out["pcl"])]
    arrays = {}
    for res, sw, pcl in parts:   # chains > 1: contiguous slices of the batch, in order
        named = [(("r3d_%d" if j % 2 == 0 else "r2d_%d") % (j // 2 + 1), t) for j, t in enumerate(res[2:])]
        named += [("spatial_weight_%d" % (j + 1), t) for j, t in enumerate(sw)] + [("pcl", pcl)]
        for name, t in named:
            arrays.setdefault(name, []).append(t.float().cpu().numpy())
    arrays = {k: np.concatenate(v) for k, v in arrays.items()}
    B = arrays["pcl"].shape[0]
    total = sum(v.nbytes for v in arrays.values())
    header = 128 * len(arrays)   # .npy header per file
    if total + header > DUMP_LIMIT:
        keep = np.sort(np.random.RandomState(0).choice(B, max(1, B * (DUMP_LIMIT - header) // total), replace=False))
        arrays = {k: v[keep] for k, v in arrays.items()}
        print(f"[bench] --dump-outputs: {len(keep)} of {B} samples (RandomState(0))", file=sys.stderr)
    os.makedirs(directory, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(directory, k + ".npy"), v)


def joint_error_mm(net, ldr, host, n):
    """mean joint error (mm) of the four joint sets on the first n samples of a timed input set vs the oracle (checker only)."""
    from oracle import kpf_oracle as O
    from keypointfusion_b200 import ops
    from keypointfusion_b200.model.model import KPFusion
    dev = next(net.parameters()).device
    d = {k: v[:n].to(dev) for k, v in host.items()}
    with torch.no_grad():
        pcl, _ = ops.getpcl(d["img"], d["center"], d["cube"], d["M"], d["cam"], N_PTS, seed=0)
        res, _, _ = net.forward_path(d["img_offset"], d["img_feat"], None, d["img_feat_rgb"], d["img"], pcl, ldr, d["center"], d["M"],
                                     d["cube"], d["cam"], 0.8)
        p = synth.fill_state_dict(KPFusion(joint_num=J), seed=0)
        g = [host[k][:n].numpy() for k in ("center", "M", "cube", "cam")]
        ores, _, _ = O.fusion_path(p, host["img"][:n], pcl.cpu(), host["img_offset"][:n].float(), host["img_feat"][:n].float(),
                                   host["img_feat_rgb"][:n].float(), *g)
    return [round(float(np.linalg.norm((res[2 + i].float().cpu().numpy() - ores[i].numpy()) * 125.0, axis=-1).mean()), 5) for i in range(4)]


def cpu_reference_leg(B, iters, warm=1):
    """The reference algorithm on the host cores (oracle port), whole fusion path incl. getpcl. -> samples/s."""
    from oracle import kpf_oracle as O  # cpu_baseline leg only
    from keypointfusion_b200.model.model import KPFusion
    torch.set_num_threads(os.cpu_count() or 1)
    net = KPFusion(joint_num=J)
    p = synth.fill_state_dict(net, seed=0)
    inp = synth.make_inputs(B, S, J, C, seed=100)
    g = [inp[k].numpy() for k in ("center", "M", "cube", "cam")]

    def once():
        pcl = np.stack([O.getpcl_sample(inp["img"][b, 0].numpy(), g[0][b], g[2][b], g[1][b], g[3][b], seed=0, b=b)[0] for b in range(B)])
        with torch.no_grad():
            O.fusion_path(p, inp["img"], torch.from_numpy(pcl), inp["img_offset"], inp["img_feat"], inp["img_feat_rgb"], *g)
    for _ in range(warm):
        once()
    t0 = time.perf_counter()
    for _ in range(iters):
        once()
    dt = time.perf_counter() - t0
    return B * iters / dt, dt / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="kpf_b200")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of the captured CUDA graph")
    ap.add_argument("--chains", type=int, default=1, help="sub-batch kernel chains captured on parallel streams inside the graph")
    ap.add_argument("--breakdown", action="store_true", help="also print per-stage CUDA-event times to stderr")
    ap.add_argument("--config", default="path", choices=["path", "sweep", "full", "demo"],
                    help="path: BASELINE configs[1] (default, the headline line); sweep: config 4; full: config 3; demo: config 5")
    ap.add_argument("--no-eager-baseline", action="store_true", help="skip the eager-PyTorch-on-this-GPU leg")
    ap.add_argument("--overlap", type=int, default=6, help="consecutive steps kept in flight on this many streams (1 = strictly serial; measured at batch 64 earlier in round 2: 1 / 2 / 3 / 4 / 6 / 8 -> 0.736 / 0.604 / 0.543 / 0.505 / 0.497 / 0.512 ms per step; final build, one K5 CTA per sample: 4 / 5 / 6 / 8 -> 0.473 / 0.466 / 0.464 / 0.466, profiles/ab_overlap_r2.txt)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy "
                    "(rank 0; the inputs depend only on the arguments, so two builds can be compared output for output)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "kpf_b200" or a.config != "path"):
        ap.error("--dump-outputs applies to the fusion path (--impl kpf_b200 --config path)")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    B = a.batch
    config = {"workload": "fusion path only (getpcl + offset2joint + img2pcl_index + 2 x Block_KPFusion), batch 64 synthetic RGB-D crops "
                          "128x128, 21 joints, 1024 points, bf16 feature maps [BASELINE.json configs[1]]",
              "batch_per_gpu": B, "parallelism": f"batch-sharded x{world}",
              "launch": "one CUDA graph replay per step; each resident input set has its own graph captured over it (no staging copies); the e2e leg uploads pinned host inputs into the graphs' static buffers every step"}

    if a.impl == "reference":
        if rank != 0:
            return
        sample_B = 16
        iters = a.steps
        v, s_it = cpu_reference_leg(sample_B, iters, warm=min(a.warmup, 1))
        cores = os.cpu_count()
        line = {"impl": "reference", "metric": "fusion-path RGB-D samples/sec", "value": v, "unit": "samples/s", "n_gpus": a.gpus,
                "steps": iters, "warmup": min(a.warmup, 1), "ms_per_step": s_it * 1e3, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": v, "unit": "samples/s", "cores": cores, "kind": "port",
                                 "sample": f"{iters} passes over a {sample_B}-crop slice of the batch-64 workload, torch threads={cores}"},
                "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (the fusion path has no CPU fallback)"
    torch.cuda.set_device(local)
    if a.config != "path":
        return other_configs(a, rank, world, local)
    try:   # pin this rank to the CPUs next to its GPU before any pinned host buffer is first touched (8 ranks feed 8 PCIe links)
        import pynvml
        pynvml.nvmlInit()
        props = torch.cuda.get_device_properties(local)
        bus = "%08x:%02x:%02x.0" % (getattr(props, "pci_domain_id", 0), props.pci_bus_id, props.pci_device_id) if hasattr(props, "pci_bus_id") else None
        handle = pynvml.nvmlDeviceGetHandleByPciBusId(bus) if bus else pynvml.nvmlDeviceGetHandleByIndex(local)
        pynvml.nvmlDeviceSetCpuAffinity(handle)
    except Exception:
        pass
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from keypointfusion_b200 import ops
    from keypointfusion_b200.dataloader.loader import loader as Loader
    sampler = ClockSampler(local)   # runs from before the warm-up to after the last timed region (the timed regions are ~0.1 s each)
    sampler.start()
    net = build_net(dev)
    ldr = Loader(img_size=S)
    S_OV = 1 if a.no_graph else max(1, a.overlap)
    if world > 1 and os.environ.get("KPF_EXCHANGE", "peer") == "nccl":
        S_OV = 1   # the host-issued all-gather fallback follows every step on the current stream: steps are not overlapped
    if S_OV > 1:
        ops.K5_SPLIT = 1   # steps in flight: SM-time, not the latency of one launch, is what counts (ops.spatial_aggregate_tc)
    NSETS = S_OV * ((4 + S_OV - 1) // S_OV)   # >= 4 resident input sets (> L2 together), a multiple of the steps in flight
    config["l2"] = f"inputs rotate over {NSETS} resident sets (~{NSETS * 51} MB) > 126 MB L2; no flush kernel inside the timed region"
    hosts = [host_inputs(B, seed=1000 * rank + s) for s in range(NSETS)]
    sets = [{k: v.to(dev) for k, v in h.items()} for h in hosts]
    pinned = [{k: v.pin_memory() for k, v in h.items()} for h in hosts]
    gathered = torch.empty(world * B, J, 3, device=dev) if world > 1 else None

    from keypointfusion_b200.runtime import GraphedFusionPath, OverlappedSteps, PeerExchange
    # the exchange step: fused into the last kernel of the path (peer stores over NVLink + arrival counter, runtime.PeerExchange),
    # captured inside the graph; KPF_EXCHANGE=nccl falls back to a per-step ncclAllGather issued from the host
    comm = "none"
    px = None
    pxs = []          # one exchange per in-flight stream (a PeerExchange's step counter lives on one stream)
    if world > 1 and not a.no_graph and os.environ.get("KPF_EXCHANGE", "peer") == "peer":
        try:
            pxs = [PeerExchange(B, J, dev) for _ in range(S_OV)]
            px = pxs[0]
            comm = "fused peer stores into symmetric memory (no NCCL call on the data path; NCCL_DEBUG logs stay empty)"
        except Exception as ex:   # no peer access / symmetric memory on this box
            print(f"[bench] PeerExchange unavailable ({type(ex).__name__}: {ex}); using ncclAllGather", file=sys.stderr)
    no_exchange = os.environ.get("KPF_EXCHANGE") == "off"   # diagnosis only: N independent replicas, no exchange step at all
    if world > 1 and px is None:
        comm = "DIAGNOSTIC: exchange step switched off (independent replicas)" if no_exchange else "ncclAllGather of [B_local,21,3] per step, issued from the host"
    graphed = None if a.no_graph else GraphedFusionPath(net, ldr, sets[0], sample_num=N_PTS, kernel=0.8, seed=0, chains=a.chains, exchange=px)
    # device-resident leg: one graph captured directly over each resident input set (no staging copies in the timed region)
    bound = {} if a.no_graph else {id(d): GraphedFusionPath(net, ldr, d, sample_num=N_PTS, kernel=0.8, seed=0, chains=a.chains, bind=True,
                                                            exchange=pxs[j % S_OV] if pxs else None) for j, d in enumerate(sets)}
    overlapped = None if a.no_graph else OverlappedSteps([bound[id(d)] for d in sets], S_OV)
    config["overlap"] = f"{S_OV} consecutive steps in flight (step i on stream i % {S_OV}); every step is a full, independent batch"

    def step(i, d):
        """d: a dict of device tensors (resident inputs) or of pinned host tensors (e2e).  Returns the path's output dict."""
        if id(d) in bound:
            out = bound[id(d)]()                     # replay the graph bound to this resident set
        elif graphed is not None:
            out = graphed(d)                         # copies the step's inputs into the graph's static buffers, replays
        else:
            if not d["img"].is_cuda:
                d = {k: v.to(dev, non_blocking=True) for k, v in d.items()}
            out = run_step(net, ldr, d, seed=i)
        if world > 1 and px is None and not no_exchange:
            dist.all_gather_into_tensor(gathered, out["joints"].contiguous())  # the path's one exchange step (NCCL fallback)
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def flush_exchanges(streams=None):
        for k, x in enumerate(pxs):
            if streams is not None:
                with torch.cuda.stream(streams[k]):
                    x.flush()
            else:
                x.flush()

    def timed(fn, steps, warmup, ov=None):
        """ov: an OverlappedSteps whose streams carry the steps (fork at the start event, join before the end event)"""
        with torch.no_grad():
            for i in range(warmup):
                fn(i)
            flush_exchanges(ov.streams if ov else None)
            if ov:
                ov.join()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            if ov:
                ov.fork()
            for i in range(steps):
                fn(warmup + i)
            flush_exchanges(ov.streams if ov else None)   # the last steps' gathers complete inside the timed region
            if ov:
                ov.join()
            e1.record()
            barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            every = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(every, t)
            rank_ms[:] = [float(x) / steps for x in every]   # evidence for the scaling run: the job's time is the slowest rank's
            ms = max(float(x) for x in every)
        return ms

    rank_ms = []

    W = max(a.warmup, 3)
    if os.environ.get("KPF_PROFILE"):  # `ncu --profile-from-start off`: capture exactly two warm steps, nothing else
        with torch.no_grad():
            for i in range(3):
                step(i, sets[i % NSETS])
            torch.cuda.synchronize()
            torch.cuda.profiler.start()
            for i in range(2):
                step(i, sets[i % NSETS])
            torch.cuda.synchronize()
            torch.cuda.profiler.stop()
        return
    if os.environ.get("KPF_TRACE"):  # CUPTI timeline of warm graph replays: in-step kernel durations and the gaps between them
        from torch.profiler import profile, ProfilerActivity
        with torch.no_grad():
            for i in range(4):
                step(i, sets[i % NSETS])
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for i in range(4):
                    step(i, sets[i % NSETS])
                torch.cuda.synchronize()
        evs = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                     key=lambda e: e.time_range.start)
        os.makedirs(os.path.dirname(os.path.abspath(os.environ["KPF_TRACE"])), exist_ok=True)
        with open(os.environ["KPF_TRACE"], "w") as f:
            prev_end = None
            for e in evs:
                s, t = e.time_range.start, e.time_range.end
                gap = 0.0 if prev_end is None else s - prev_end
                f.write(f"{s - evs[0].time_range.start:10.1f} us  dur {t - s:8.1f}  gap {gap:7.1f}  {e.name[:70]}\n")
                prev_end = t
        return
    n0 = ops.launch_count()
    last = {}   # the output dict of the latest step

    if overlapped is not None and S_OV > 1:
        def resident_step(i):
            last["out"] = overlapped.submit()
        ms = timed(resident_step, a.steps, W, ov=overlapped)
    else:
        def resident_step(i):
            last["out"] = step(i, sets[i % NSETS])
        ms = timed(resident_step, a.steps, W)
    if a.dump_outputs and rank == 0:
        dump_outputs(last["out"], a.dump_outputs)   # before any later step replays the same graph over its output buffers
    device_rank_ms = list(rank_ms)   # per-rank ms per step of the device-resident leg (world > 1)
    if graphed is not None:
        launches = graphed.launches_per_replay * a.steps   # kernels of ours replayed by the graph inside the K timed steps
    else:
        launches = (ops.launch_count() - n0) * a.steps // (a.steps + W)

    # end to end through the public API: pinned host buffers -> H2D -> path -> D2H joints, every step
    h2d = sum(v.numel() * v.element_size() for v in hosts[0].values())
    out_host = torch.empty(B, J, 3).pin_memory()

    def e2e_step(i):
        out_host.copy_(step(i, pinned[i % NSETS])["joints"], non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the caller reads the joints on the host every step
    if graphed is None:
        ms_e2e = timed(e2e_step, a.steps, W)
    else:
        # public serving API: double-buffered graphs, H2D of step i+1 overlaps compute of step i, host reads step i-1's joints
        from keypointfusion_b200.runtime import PipelinedRunner
        runner = PipelinedRunner(net, ldr, sets[0], sample_num=N_PTS, kernel=0.8, seed=0, exchange=px)
        # the caller's host buffers: pinned arenas handed out by the runner (one upload per step), filled with the same data
        host_sets = []
        for h in hosts:
            d = runner.new_host_inputs()
            for k, v in h.items():
                d[k].copy_(v)
            host_sets.append(d)
        h2d = host_sets[0]["_arena"].numel()
        pending = []

        def pipe_step(i):
            pending.append(runner.submit(host_sets[i % NSETS]))
            if world > 1 and px is None:
                dist.all_gather_into_tensor(gathered, runner.paths[pending[-1]].out["joints"].contiguous())
            if len(pending) > 1:
                runner.fetch(pending.pop(0))       # host-side read of the previous step's result
        with torch.no_grad():
            for i in range(W):
                pipe_step(i)
            while pending:
                runner.fetch(pending.pop(0))
            if px is not None:
                px.flush()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(a.steps):
                pipe_step(W + i)
            while pending:
                runner.fetch(pending.pop(0))       # the last result is read inside the timed region too
            if px is not None:
                px.flush()
            e1.record()
            barrier()
        ms_e2e = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms_e2e], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_e2e = float(t)
    value = world * B * a.steps / (ms / 1e3)
    e2e = world * B * a.steps / (ms_e2e / 1e3)
    hbm, tfl, which = load_peaks()

    # dominant kernel of the step: measured live, CUDA events on the launching stream
    roof = dominant_kernel_roofline(net, ldr, sets, hbm, tfl, which, a.breakdown and rank == 0)
    # keep the GPU under the same load until nvidia-smi has delivered a few samples (its first sample takes ~1 s to appear)
    t_end = time.time() + 3.0
    with torch.no_grad():
        while len(sampler.rows) < 8 and time.time() < t_end:
            for i in range(20):
                step(i, sets[i % NSETS])
            torch.cuda.synchronize()
    clocks = sampler.stop()

    line = {"metric": "fusion-path RGB-D samples/sec", "value": value, "unit": "samples/s", "n_gpus": world, "steps": a.steps, "warmup": W,
            "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": config, "clocks": clocks,
            "e2e": {"value": e2e, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": B * J * 3 * 4,
                    "h2d_gb_per_s": round(h2d * (e2e / world / B) / 1e9, 1),
                    "note": "upload-bound: one pinned-arena cudaMemcpyAsync per step, overlapped with compute (profiles/h2d_ceiling.py measures the link)"},
            "gpu_launches": launches, "comm": comm, "roofline": roof,
            "path_roofline": {"hbm_frac": value / world * PATH_BYTES_PER_SAMPLE / (hbm * 1e9),
                              "tensor_frac": value / world * PATH_FLOPS_PER_SAMPLE / (tfl * 1e12), "peaks": which}}
    if world > 1:
        line["rank_ms_per_step"] = [round(x, 4) for x in device_rank_ms]
    if rank == 0 and world == 1:
        # parity of the exact configuration that was timed: a 4-sample slice of resident set 0 against the CPU oracle (the kernels are
        # batch invariant, tests/test_modules_gpu.py)
        line["joint_err_mm"] = joint_error_mm(net, ldr, hosts[0], 4)
        if not a.no_eager_baseline:
            import bench_extra as X
            line["cuda_eager_baseline"] = X.cuda_eager_leg(dev, hosts[0])
    if rank == 0:
        if world == 1 and not a.no_cpu_baseline:
            sample_B, iters = 16, 3
            v, s_it = cpu_reference_leg(sample_B, iters)
            line["cpu_baseline"] = {"value": v, "unit": "samples/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": f"{iters} passes over a {sample_B}-crop slice of the workload, torch threads={os.cpu_count()}"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def other_configs(a, rank, world, local):
    """BASELINE.json configs 3, 4, 5 (bench_extra.py): one JSON line each, same keys as the headline line where they apply."""
    import bench_extra as X
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    hbm, tfl, which = load_peaks()
    sampler = ClockSampler(local)
    sampler.start()
    W = max(a.warmup, 3)
    base = {"n_gpus": world, "steps": a.steps, "warmup": W, "higher_is_better": True, "vs_baseline": None, "data": "synthetic"}
    if a.config == "sweep":
        assert world == 1, "the kernel sweep is a single-GPU configuration"
        rows = X.sweep(dev, hbm)
        # the same kernels at config 3's batch (512 crops per GPU): at batch 64 a launch moves 2-15 MB, i.e. 0.3-2 us of HBM time --
        # below the duration of ANY kernel launch -- so the batch-64 rows measure latency, these measure bandwidth
        rows += X.sweep(dev, hbm, B=512, sizes=(128,), k7=False)
        k1 = next(r for r in rows if r["kernel"].startswith("backproject") and r["S"] == 128)
        line = dict(base, metric="kernel sweep: back-projection + keypoint gather GB/s over crop sizes 64-256 and 21-42 joints",
                    value=k1["GBs"], unit="GB/s (K1 at S=128; all rows in `sweep`)", scaling="weak", dtype="f32/bf16",
                    config={"workload": "BASELINE.json configs[3]: K1, K2, K3, K4a, K4d over S in {64,96,128,192,256}, J in {21,42}, K7 at the ResNet-18 "
                                        "stage shapes; batch 64, and batch 512 (config 3's) at S=128; inputs rotate over resident sets (> L2 where the working set allows)"},
                    sweep=rows, roofline={"bound": "hbm", "achieved": k1["GBs"], "peak": hbm, "unit": "GB/s", "frac": k1["GBs"] / hbm,
                                          "traffic": None, "kernel": "backproject_kernel", "peaks": which})
    else:
        fn = X.full_model if a.config == "full" else X.demo
        r = fn(dev, world, rank, a.steps, W, barrier=barrier)
        ms = torch.tensor([r["ms_per_step"]], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            r["value"] = world * r["batch_per_gpu"] / (float(ms) / 1e3)
            r["ms_per_step"] = float(ms)
        wl = ("BASELINE.json configs[2]: full model inference = 2 x stock-PyTorch ConvNeXt-T UNet stand-in backbones (bf16, channels_last; out "
              "of scope, utils/standin_backbone.py) + the fusion path, batch 512 sharded over the ranks") if a.config == "full" else \
             ("BASELINE.json configs[4]: 640x480 uint16 depth + uint8 BGR frames -> bbox centre, crops (crop.cu), back-projection (K1), stand-in "
              "backbones, fusion path; batch 128 sharded over the ranks")
        line = dict(base, metric="full-model RGB-D samples/sec" if a.config == "full" else "in-the-wild RGB-D frames/sec",
                    unit="samples/s", scaling="strong", dtype="bf16", config={"workload": wl, "batch_per_gpu": r["batch_per_gpu"],
                                                                             "parallelism": f"batch-sharded x{world}"}, **r)
    line["clocks"] = sampler.stop()
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def dominant_kernel_roofline(net, ldr, sets, hbm, tfl, which, verbose):
    """Time every kernel of the step ALONE with CUDA events on the launching stream (inputs rotate over resident sets so they
    come from HBM, not L2), weight by launches per step, and report the roofline of the kernel with the largest share.
    ALGORITHMIC bytes / FLOPs per launch follow SURVEY.md 8d x the units one launch processes (DESIGN.md section 4)."""
    from keypointfusion_b200 import ops
    d0 = sets[0]
    B = d0["img"].shape[0]
    blk = net.block1
    k = blk.kc()
    with torch.no_grad():
        pcl, _ = ops.getpcl(d0["img"], d0["center"], d0["cube"], d0["M"], d0["cam"], N_PTS, seed=0)
        order = ops.spatial_order(pcl, d0["center"], d0["M"], d0["cube"], d0["cam"], S, H)
        close, _, idx = ops.img2pcl_index(pcl, d0["img"], d0["center"], d0["M"], d0["cube"], d0["cam"], S, 4, fs=H, want_i64=False, want_i32=True,
                                          order=order)
        joints = pcl[:, ::48][:, :J].contiguous() + 0.01
        featT = ops.repack_features(d0["img_feat"], d0["img_feat_rgb"], d0["img_offset"][:, 4 * J:])
        e_, acc_, ms_ = ops.point_embed(featT, idx, close, pcl, joints, k["pe_wmat"], k["pe_wvec"], 0.8, order=order)
        part_, jf_ = ops.desa_fused(e_, acc_, ms_, pcl, joints, k["ds_wmat"], k["ds_wvec"], blk.FA.radius, blk.FA.S[0])
        tok_, r3d_, _ = ops.token_stack(k["tok_init"], desa=part_, jf=jf_)
        fj_ = torch.randn(B, J, C, device=pcl.device)
        stage_ = ops.point_embed_stage(B, N_PTS, pcl.device)
        ops.point_embed(featT, idx, close, pcl, joints, k["pe_wmat"], k["pe_wvec"], 0.8, order=order, stage_out=stage_)
        # per-set point clouds / orders for the kernels whose cost depends on the points matching the depth map they came from
        geo = {}
        for d in sets:
            p_, _ = ops.getpcl(d["img"], d["center"], d["cube"], d["M"], d["cam"], N_PTS, seed=0)
            geo[id(d)] = (p_, ops.spatial_order(p_, d["center"], d["M"], d["cube"], d["cam"], S, H))
    e = 2  # bf16 feature maps
    # name[variant] -> (callable, launches per step, algorithmic bytes per launch, algorithmic FLOPs per launch, bound); the variants
    # of a kernel (its two token programs; the point stage storing / loading the gathered tiles) are averaged by launches per step
    T_ = N_PTS // 64
    stages = {
        "token_stack_kernel[tok_init]": (lambda d: ops.token_stack(k["tok_init"], desa=part_, jf=jf_), 2,
                                         B * (4 * J * C * 4 + J * C * 4 + J * 12), B * 16.05e6, "tensor"),
        "token_stack_kernel[tok_final]": (lambda d: ops.token_stack(k["tok_final"], x=fj_, y=tok_, r3d=r3d_, want_tokens=False), 2,
                                          B * (2 * J * C * 4 + J * 12 + J * 12), B * 17.67e6, "tensor"),
        "desa_prep_kernel+desa_tile_kernel": (lambda d: ops.desa_fused(e_, acc_, ms_, pcl, joints, k["ds_wmat"], k["ds_wvec"], blk.FA.radius, blk.FA.S[0]), 2,
                              B * (3 * J * 64 * C * e + N_PTS * 12 + 4 * J * C * 4), B * 270.1e6, "tensor"),
        "point_embed_kernel[stage_out]": (lambda d: ops.point_embed(featT, idx, close, pcl, joints, k["pe_wmat"], k["pe_wvec"], 0.8, order=order,
                                                                    stage_out=stage_), 1,
                                          B * ((2 * C + J) * H * H * e + N_PTS * 4 * 8 + N_PTS * C * e * 2 + T_ * ops.PE_STAGE_BYTES_PER_TILE), B * 95.4e6, "tensor"),
        "point_embed_kernel[stage_in]": (lambda d: ops.point_embed(featT, idx, close, pcl, joints, k["pe_wmat"], k["pe_wvec"], 0.8, order=order,
                                                                   stage_in=stage_), 1,
                                         B * (T_ * ops.PE_STAGE_BYTES_PER_TILE + N_PTS * 16 + N_PTS * C * e * 2), B * 95.4e6, "tensor"),
        "spatial_aggregate_tc_kernel": (lambda d: ops.spatial_aggregate_tc(d["img_feat_rgb"], joints, d["img"][:, :, ::4, ::4], d["center"], d["M"],
                                                                          d["cube"], d["cam"], k["wa_packed"], blk.atten_spatial.bias,
                                                                          blk.weight_dis, blk.fc_spatial2joint_feature.weight,
                                                                          blk.fc_spatial2joint_feature.bias), 2,
                                        B * (C * H * H * e + J * H * H * 4 + J * C * 4), B * 12.04e6, "hbm"),
        "nearest_cells_kernel": (lambda d: ops.img2pcl_index(geo[id(d)][0], d["img"], d["center"], d["M"], d["cube"], d["cam"], S, 4, fs=H,
                                                             want_i64=False, want_i32=True, order=geo[id(d)][1]), 1, B * (N_PTS * 12 + H * H * 4 + 76 + N_PTS * 4 * 8), B * 8.39e6, "hbm"),
        "repack_bf16_kernel": (lambda d: ops.repack_features(d["img_feat"], d["img_feat_rgb"], d["img_offset"][:, 4 * J:]), 1,
                          B * ((2 * C + J) * H * H * e + 288 * H * H * 2), 0.0, "hbm"),
        "offset2joint_kernel": (lambda d: ops.offset2joint_weight(d["img_offset"], d["img"], 0.8), 1, B * (5 * J * H * H * e + H * H * 4), B * 0.3e6,
                                "hbm"),
        "spatial_order_kernel": (lambda d: ops.spatial_order(geo[id(d)][0], d["center"], d["M"], d["cube"], d["cam"], S, H), 1,
                                 B * (N_PTS * 12 + N_PTS * 4), 0.0, "hbm"),
        "backproject_kernel": (lambda d: ops.getpcl(d["img"], d["center"], d["cube"], d["M"], d["cam"], N_PTS, seed=0), 1,
                               B * (S * S * 4 + 76 + N_PTS * 12), B * 0.33e6, "hbm"),
    }
    res = {}
    for name, (fn, per_step, alg_bytes, alg_flops, bound) in stages.items():
        g = torch.cuda.CUDAGraph()   # a graph of NSETS launches: no Python / launch overhead inside the timed region
        with torch.no_grad():
            for i in range(3):
                fn(sets[i % len(sets)])
            torch.cuda.synchronize()
            with torch.cuda.graph(g):
                for i in range(len(sets)):
                    fn(sets[i])
            g.replay()
            torch.cuda.synchronize()
            reps = 5
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(reps):
                g.replay()
            e1.record()
            torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / (reps * len(sets))
        res[name] = dict(us=us, per_step=per_step, bytes=alg_bytes, flops=alg_flops, bound=bound)
        if verbose:
            print(f"[breakdown] {name:30s} x{per_step}  {us:8.1f} us  {alg_bytes / us / 1e3:8.1f} GB/s  {alg_flops / us / 1e6:8.2f} TFLOP/s (algorithmic)",
                  file=sys.stderr)
    variants = res
    res = {}
    for name, v in variants.items():   # variants of one kernel -> its per-launch average, weighted by launches per step
        a = res.setdefault(name.split("[")[0], dict(us=0.0, per_step=0, bytes=0.0, flops=0.0, bound=v["bound"]))
        for f in ("us", "bytes", "flops"):
            a[f] += v[f] * v["per_step"]
        a["per_step"] += v["per_step"]
    for a in res.values():
        for f in ("us", "bytes", "flops"):
            a[f] /= a["per_step"]
    tot = sum(r["us"] * r["per_step"] for r in res.values())
    top = max(res, key=lambda n: res[n]["us"] * res[n]["per_step"])
    r = res[top]
    traffic = None
    tp = os.path.join(ROOT, "profiles", "dram_bytes_per_launch.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get(top)
    if r["bound"] == "tensor":
        ach, peak, unit = r["flops"] / (r["us"] * 1e-6) / 1e12, tfl, "TFLOP/s"
    else:
        ach, peak, unit = r["bytes"] / (r["us"] * 1e-6) / 1e9, hbm, "GB/s"
    return {"kernel": top, "bound": r["bound"], "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak, "traffic": traffic,
            "us_per_launch": r["us"], "launches_per_step": r["per_step"], "share_of_step": r["us"] * r["per_step"] / tot,
            "algorithmic_bytes": r["bytes"], "algorithmic_flops": r["flops"], "peaks": which,
            "note": "both token programs timed (tok_init, tok_final), averaged by launches; latency-bound: one sample per CTA, ~7 dependent "
                    "MMA->epilogue steps per transformer layer, identical time for 1..148 samples (profiles/probe_token.py); see DESIGN.md section 4",
            "traffic_source": "profiles/dram_bytes_per_launch.json (ncu dram__bytes of the same kernels, profiles/collect.sh; bench.py cannot read DRAM counters itself)",
            "kernels": {n: {"us": round(v["us"], 1), "per_step": v["per_step"]} for n, v in variants.items()}}


if __name__ == "__main__":
    main()
