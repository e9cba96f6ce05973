"""Several hands per frame (frame_index) against one frame per hand, frames to keypoints on one GPU.

B = 128 hands per step, the 640x480 frames of bench_extra.demo_frames and the stand-in backbones of bench_extra.build_full_net:
  indexed      64 frames x 2 hands, frame_index = [0,0,1,1,...]: each frame uploaded and stored once;
  duplicated   128 frames x 1 hand: each hand's frame copied, today's route.  Its runner leg carries frame_index = arange(128)
               (the graphed frames path has a frame_index buffer); its front-end leg runs frame_index=None.
For each: device-resident hands/s and frames/s (CUDA-event timed replays of the captured frames graph: crop front end, backbones,
fusion path, joints_to_frame), end to end from pinned host frames through PipelinedRunner (one arena upload per step, double
buffered, host clock around `steps` steps ending in a fetch), H2D bytes per step, and the crop front end alone (captured
prepare_batch, events).  Both cases compute the same keypoints (checked).  The device-resident legs replay the same resident frames;
the front end reads only the <= 16384 pixels each crop samples, so its working set sits in L2 either way.

    python profiles/bench_frames.py --steps 30 --warmup 5 --out profiles/bench_frames.json
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

CAM = (617.0, 617.0, 312.0, 241.0)


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as ex:
        q = f"unavailable ({type(ex).__name__})"
    return {"gpu": name, "power_limit_and_max_sm_clock": q}


def events_ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def make_cases(seed):
    import bench_extra as X
    rgb, depth, bbox = X.demo_frames(np.random.RandomState(seed), 64, hands=2)
    fi = np.repeat(np.arange(64), 2).astype(np.int32)
    depth = depth.view(np.int16)        # uint16 bits, stored as int16
    indexed = dict(rgb=rgb, depth=depth, bbox=bbox, frame_index=fi)
    duplicated = dict(rgb=rgb[fi], depth=depth[fi], bbox=bbox, frame_index=np.arange(128, dtype=np.int32))
    return {k: {n: torch.from_numpy(np.ascontiguousarray(v)) for n, v in d.items()} for k, d in (("indexed", indexed), ("duplicated", duplicated))}


def run_case(name, net, sets, steps, warmup, dev):
    from keypointfusion_b200.demo_RGBD import Model_RGBD
    from keypointfusion_b200.runtime import GraphedFramePath, PipelinedRunner
    F, B = sets[0]["rgb"].shape[0], sets[0]["bbox"].shape[0]
    runner = PipelinedRunner(net, None, {k: v.to(dev) for k, v in sets[0].items()}, path_cls=GraphedFramePath, cam_para=CAM)
    hosts = []
    for s in sets:
        h = runner.new_host_inputs()
        for k in GraphedFramePath.KEYS:
            h[k].copy_(s[k])
        hosts.append(h)
    # device resident: replays of one captured frames graph on the frames already in its arena
    g = runner.paths[0].graph
    for _ in range(warmup):
        g.replay()
    torch.cuda.synchronize()
    ms_dev = events_ms(g.replay, steps)
    # end to end: pinned host frames -> one upload per step -> graph -> keypoints back in pinned memory
    outs = []

    def e2e(n, keep=False):
        slots = []
        for i in range(n):
            slots.append(runner.submit(hosts[i % len(hosts)]))
            if len(slots) > 1:
                o = runner.fetch(slots.pop(0))
                if keep:
                    outs.append(tuple(t.clone() for t in o))
        o = runner.fetch(slots.pop(0))
        if keep:
            outs.append(tuple(t.clone() for t in o))
    e2e(len(hosts), keep=True)
    e2e(warmup)
    t0 = time.perf_counter()
    e2e(steps)
    s_e2e = (time.perf_counter() - t0) / steps
    # crop front end alone (centre, both crops, back-projection), captured
    m = Model_RGBD(None, cam_para=CAM)
    d = {k: v.to(dev) for k, v in sets[0].items()}
    fi = d["frame_index"] if name == "indexed" else None
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream), torch.no_grad():
        for _ in range(3):
            m.prepare_batch(d["rgb"], d["depth"], d["bbox"], fi)
    torch.cuda.current_stream().wait_stream(stream)
    torch.cuda.synchronize()
    fg = torch.cuda.CUDAGraph()
    with torch.no_grad(), torch.cuda.graph(fg, stream=stream):
        m.prepare_batch(d["rgb"], d["depth"], d["bbox"], fi)
    fg.replay()
    torch.cuda.synchronize()
    ms_front = events_ms(fg.replay, 200)
    res = {"frames": F, "hands": B, "device_hands_per_s": round(B / (ms_dev / 1e3), 1), "device_frames_per_s": round(F / (ms_dev / 1e3), 1),
           "device_ms_per_step": round(ms_dev, 3), "e2e_hands_per_s": round(B / s_e2e, 1), "e2e_frames_per_s": round(F / s_e2e, 1),
           "e2e_ms_per_step": round(s_e2e * 1e3, 3), "h2d_bytes_per_step": runner.arenas[0].nbytes, "front_end_us": round(ms_front * 1e3, 2),
           "launches_per_replay": runner.paths[0].launches_per_replay}
    return res, outs


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_frames.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_frames.py measures on a GPU; none is visible")
    import bench_extra as X
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    net = X.build_full_net(dev)
    cases = [make_cases(900 + s) for s in range(2)]       # two frame sets per case, alternated step by step
    line = {"metric": "frames to keypoints, B = 128 hands per step: 64 frames x 2 hands (frame_index) vs 128 frames x 1 hand (duplicated)",
            "steps": a.steps, "warmup": a.warmup, **gpu_info(), "torch": torch.__version__,
            "backbones": "bench_extra.build_full_net (stock-PyTorch stand-ins, bf16 channels_last)"}
    outs = {}
    with torch.no_grad():
        for name in ("indexed", "duplicated"):
            line[name], outs[name] = run_case(name, net, [c[name] for c in cases], a.steps, a.warmup, dev)
    line["same_keypoints"] = all(torch.equal(x, y) for p, q in zip(outs["indexed"], outs["duplicated"]) for x, y in zip(p, q))
    i, d = line["indexed"], line["duplicated"]
    line["indexed_over_duplicated"] = {k: round(i[k] / d[k], 3) for k in ("device_hands_per_s", "e2e_hands_per_s", "h2d_bytes_per_step", "front_end_us")}
    s = json.dumps(line)
    print(s)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
