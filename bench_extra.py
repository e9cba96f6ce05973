"""bench.py's other configurations (BASELINE.json configs 3, 4, 5) and legs that are not the headline line:

  --config sweep   config 4: K1 back-projection, K2 nearest cells, K3 keypoint gathers, K4a / K4d joint-feature kernels and K7 RGB-D
                   fusion over crop sizes 64-256 and 21 / 42 joints, each in GB/s of ALGORITHMIC bytes against the measured HBM peak
  --config full    config 3: full model = two stock-PyTorch ConvNeXt-T UNet stand-in backbones (out of scope, utils/standin_backbone.py)
                   + the fusion path, batch 512 sharded over the ranks
  --config demo    config 5: demo_RGBD.py-style 640x480 uint16 depth + uint8 BGR frames -> crop -> back-projection -> backbones ->
                   fusion path, batch 128 sharded over the ranks, frames uploaded from pinned host memory every step (e2e)
  cuda_eager_leg   the reference's op chain as eager PyTorch on the same GPU (baseline/eager_torch_path.py): BASELINE.md section 3's
                   "number the new kernels must beat"

Every function returns a dict that bench.py prints as ONE JSON line."""
import os
import time

import numpy as np
import torch

J, C = 21, 128


def _events_ms(fn, steps, warmup, barrier=None):
    with torch.no_grad():
        for i in range(warmup):
            fn(i)
        (barrier or torch.cuda.synchronize)()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(warmup + i)
        e1.record()
        (barrier or torch.cuda.synchronize)()
    return e0.elapsed_time(e1)


def _graph_us(fn, args_sets, reps=5):
    """microseconds per call of fn(*args), timed as a CUDA graph of len(args_sets) calls over rotating argument sets (> L2)."""
    g = torch.cuda.CUDAGraph()
    with torch.no_grad():
        for a in args_sets[:2]:
            fn(*a)
        torch.cuda.synchronize()
        with torch.cuda.graph(g):
            for a in args_sets:
                fn(*a)
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (reps * len(args_sets))


# ------------------------------------------------------------------------------------------------ config 4: kernel sweep
def sweep(dev, hbm_gbs, B=64, sizes=(64, 96, 128, 192, 256), k7=True):
    """Bandwidth-bound kernels of north_star items (1) and (2) over S in {64..256}, J in {21, 42}.  Inputs rotate over enough resident
    sets to exceed the 126 MB L2 where the working set allows (stated per row as `sets`)."""
    from keypointfusion_b200 import ops
    from keypointfusion_b200.utils import synth
    rows = []

    def add(kernel, S, Jn, us, alg_bytes, sets, note=""):
        gbs = alg_bytes / us / 1e3
        rows.append({"kernel": kernel, "B": B, "S": S, "J": Jn, "us": round(us, 2), "alg_MB": round(alg_bytes / 1e6, 3), "GBs": round(gbs, 1),
                     "hbm_frac": round(gbs / hbm_gbs, 4), "sets": sets, **({"note": note} if note else {})})
    for S in sizes:
        H = S // 4
        nsets = max(2, min(16, int(140e6 / (B * (2 * C + 5 * 42) * H * H * 2)) + 1))
        base = [synth.make_inputs(B, S, 21, C, seed=10 + s) for s in range(2)]
        cu = [{k: v.to(dev) for k, v in b.items()} for b in base]
        # more resident copies of the big tensors (clones: the values do not matter for timing, the addresses do)
        imgs = [cu[i % 2]["img"].clone() for i in range(nsets)]
        g = lambda i: [cu[i % 2][k] for k in ("center", "cube", "M", "cam")]
        # K1 back-projection: S*S*4 + 76 read, 1024*3*4 written per sample
        us = _graph_us(lambda im, c, q, m, k: ops.getpcl(im, c, q, m, k, 1024, seed=1), [(imgs[i], *g(i)) for i in range(nsets)])
        add("backproject_kernel (K1)", S, 0, us, B * (S * S * 4 + 76 + 1024 * 12), nsets)
        pcl = [ops.getpcl(cu[i]["img"], *g(i), 1024, seed=1)[0] for i in range(2)]
        # K2 nearest cells (fp32-ALU bound; reported against HBM too, SURVEY 8d)
        us = _graph_us(lambda p_, im, c, q, m, k: ops.img2pcl_index(p_, im, c, m, q, k, S, 4, fs=H, want_i64=False, want_i32=True),
                       [(pcl[i % 2], imgs[i], *g(i)) for i in range(nsets)])
        add("nearest_cells_kernel (K2)", S, 0, us, B * (1024 * 12 + H * H * 4 + 76 + 1024 * 4 * 8), nsets, "fp32-ALU bound, exact op order")
        close, _, idx = ops.img2pcl_index(pcl[0], cu[0]["img"], cu[0]["center"], cu[0]["M"], cu[0]["cube"], cu[0]["cam"], S, 4, fs=H,
                                          want_i64=False, want_i32=True)
        for Jn in (21, 42):
            e = 2
            maps = [(torch.randn(B, C, H, H, device=dev).bfloat16(), torch.randn(B, C, H, H, device=dev).bfloat16(),
                     torch.randn(B, 5 * Jn, H, H, device=dev).bfloat16()) for _ in range(nsets)]
            # K3 keypoint gathers (model.py:297-306): the three maps, 4 taps
            def k3(fd, fr, fo):
                ops.gather_taps(fd, idx, close)
                ops.gather_taps(fr, idx, close)
                ops.gather_taps(fo[:, 4 * Jn:], idx, close)
            us = _graph_us(k3, maps)
            add("gather_taps_kernel (K3, 3 maps)", S, Jn, us, B * ((2 * C + Jn) * H * H * e + 1024 * 4 * 8 + (2 * C + Jn) * 1024 * e), nsets)
            # K4a offset -> joint
            us = _graph_us(lambda fo, im: ops.offset2joint_weight(fo, im, 0.8), [(maps[i][2], imgs[i]) for i in range(nsets)])
            add("offset2joint_kernel (K4a)", S, Jn, us, B * (5 * Jn * H * H * e + H * H * 4), nsets)
            # K4d dense offset target (write bound)
            jt = torch.rand(B, Jn, 3, device=dev) * 1.2 - 0.6
            us = _graph_us(lambda im: ops.joint2offset(jt, im, 0.8, H), [(imgs[i],) for i in range(nsets)])
            add("joint2offset_kernel (K4d)", S, Jn, us, B * (4 * Jn * H * H * 4 + H * H * 4), nsets)
    # K7 RGBDFusion at the four ResNet-18 stage shapes of a 128 crop (model/resnet.py:439-442)
    for Cc, h in ((64, 32), (128, 16), (256, 8), (512, 4)) if k7 else ():
        n = max(2, min(32, int(140e6 / (B * Cc * h * h * 2 * 2)) + 1))
        xs = [(torch.randn(B, Cc, h, h, device=dev).bfloat16(), torch.randn(B, Cc, h, h, device=dev).bfloat16()) for _ in range(n)]
        gw, gb = torch.randn(2, 2 * Cc, device=dev), torch.randn(2, device=dev)
        us = _graph_us(lambda r, d: ops.rgbd_fusion(r, d, gw, gb), xs)
        add(f"rgbd_fusion_kernel (K7) C={Cc} {h}x{h}", 128, 0, us, B * 5 * Cc * h * h * 2, n)
    return rows


# ------------------------------------------------------------------------------------------------ configs 3 / 5: with backbones
def build_full_net(dev, bf16=True):
    from keypointfusion_b200.model.model import KPFusion
    from keypointfusion_b200.utils import synth
    from keypointfusion_b200.utils.standin_backbone import StandInBackbone
    torch.manual_seed(0)
    net = KPFusion(joint_num=J, backbone_rgb=StandInBackbone(3, J), backbone_d=StandInBackbone(1, J))
    synth.fill_state_dict({k: v for k, v in net.state_dict().items() if k.startswith("block")}, seed=0)
    sd = net.state_dict()
    sd.update(synth.fill_state_dict({k: v.clone() for k, v in sd.items() if k.startswith("block")}, seed=0))
    net.load_state_dict(sd)
    net = net.to(dev).eval()
    if bf16:
        net.backbone_rgb.to(torch.bfloat16).to(memory_format=torch.channels_last)
        net.backbone_d.to(torch.bfloat16).to(memory_format=torch.channels_last)
    return net


def full_step(net, ldr, d):
    """d: img_rgb [B,3,S,S] f32, img [B,1,S,S] f32, pcl, center, M, cube, cam -> final joints (KPFusion.forward, model.py:395-426)."""
    dt = next(net.backbone_d.parameters()).dtype
    off, feat = net.backbone_d(d["img"].to(dt).contiguous(memory_format=torch.channels_last))
    off_rgb, feat_rgb = net.backbone_rgb(d["img_rgb"].to(dt).contiguous(memory_format=torch.channels_last))
    res, sw, _ = net.forward_path(off.detach().contiguous(), feat.contiguous(), off_rgb, feat_rgb.contiguous(), d["img"], d["pcl"], ldr,
                                  d["center"], d["M"], d["cube"], d["cam"], 0.8)
    return res[-1]


def _try_graph(fn):
    """Capture fn() into a CUDA graph (returns replay callable + output) or fall back to eager."""
    try:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s), torch.no_grad():
            for _ in range(3):
                fn()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.no_grad(), torch.cuda.graph(g, stream=s):
            out = fn()
        return (lambda: (g.replay(), out)[1]), True
    except Exception as ex:   # e.g. a cuDNN algorithm that allocates during capture
        torch.cuda.synchronize()
        print(f"[bench] graph capture failed ({type(ex).__name__}: {ex}); timing eager launches", flush=True)
        return fn, False


def full_model(dev, world, rank, steps, warmup, total_batch=512, barrier=None):
    from keypointfusion_b200 import ops
    from keypointfusion_b200.dataloader.loader import loader as Loader
    from keypointfusion_b200.utils import synth
    B = total_batch // world
    net, ldr = build_full_net(dev), Loader(img_size=128)
    sets = []
    for s in range(2):
        inp = synth.make_inputs(B, 128, J, C, seed=500 + 10 * rank + s)
        d = {k: inp[k].to(dev) for k in ("img", "img_rgb", "center", "M", "cube", "cam")}
        d["pcl"] = ops.getpcl(d["img"], d["center"], d["cube"], d["M"], d["cam"], 1024, seed=s)[0]
        sets.append(d)
    runs = [_try_graph(lambda d=d: full_step(net, ldr, d)) for d in sets]
    graphed = all(r[1] for r in runs)
    ms = _events_ms(lambda i: runs[i % 2][0](), steps, warmup, barrier)
    # split: backbones alone / path alone (eager events on one set)
    d = sets[0]
    dt = next(net.backbone_d.parameters()).dtype

    def bb(i):
        net.backbone_d(d["img"].to(dt).contiguous(memory_format=torch.channels_last))
        net.backbone_rgb(d["img_rgb"].to(dt).contiguous(memory_format=torch.channels_last))
    ms_bb = _events_ms(bb, 5, 2) / 5
    return {"ms_per_step": ms / steps, "value": world * B * steps / (ms / 1e3), "batch_per_gpu": B, "graphed": graphed,
            "backbones_ms": ms_bb, "path_ms_by_difference": ms / steps - ms_bb}


def demo_frames(rs, F, hands=1):
    """F synthetic 640x480 frames with `hands` hands each, drawn from RandomState rs -> (rgb [F,480,640,3] uint8 (random BGR),
    depth [F,480,640] uint16 (900 mm background), bbox [F*hands,4] f64 (x,y,w,h); box f*hands+h is hand h of frame f).
    A "hand" is a disc 120-170 px wide at 450-650 mm with +-20 mm relief, inside its bounding box (discs of one frame may overlap)."""
    depth = np.full((F, 480, 640), 900, np.uint16)
    yy, xx = np.mgrid[0:480, 0:640]
    bbox = np.zeros((F * hands, 4), np.float64)
    for f in range(F):
        for h in range(hands):
            cx, cy, r = rs.uniform(200, 440), rs.uniform(150, 330), rs.uniform(60, 85)
            disc = (xx - cx) ** 2 + (yy - cy) ** 2 <= r * r
            depth[f][disc] = (rs.uniform(450, 650) + 20 * np.sin(xx[disc] / 9.0) * np.cos(yy[disc] / 7.0)).astype(np.uint16)
            bbox[f * hands + h] = (cx - r - 10, cy - r - 10, 2 * r + 20, 2 * r + 20)
    rgb = rs.randint(0, 256, (F, 480, 640, 3)).astype(np.uint8)
    return rgb, depth, bbox


def demo(dev, world, rank, steps, warmup, total_batch=128, barrier=None):
    """config 5: 640x480 frames (uint16 depth + uint8 BGR) -> crop (K0) -> back-projection (K1) -> backbones -> fusion path."""
    from keypointfusion_b200.demo_RGBD import Model_RGBD
    B = total_batch // world
    net = build_full_net(dev)
    m = Model_RGBD(net, cam_para=(617.0, 617.0, 312.0, 241.0))
    rs = np.random.RandomState(40 + rank)
    frames = []
    for s in range(3):
        rgb, depth, bbox = demo_frames(rs, B)
        frames.append((torch.from_numpy(rgb).pin_memory(), torch.from_numpy(depth.view(np.int16)).pin_memory(), torch.from_numpy(bbox).pin_memory()))
    dev_frames = [tuple(t.to(dev) for t in f) for f in frames]

    def step_dev(i):
        rgb, depth, bbox = dev_frames[i % 3]
        res, _ = m.estimate_pose_RGBD(rgb, depth, bbox)
        return res[-1]
    ms = _events_ms(step_dev, steps, warmup, barrier)
    out_host = torch.empty(B, J, 3).pin_memory()

    def step_e2e(i):
        rgb, depth, bbox = (t.to(dev, non_blocking=True) for t in frames[i % 3])
        res, _ = m.estimate_pose_RGBD(rgb, depth, bbox)
        out_host.copy_(res[-1], non_blocking=True)
        torch.cuda.current_stream().synchronize()
    ms_e2e = _events_ms(step_e2e, steps, warmup, barrier)
    h2d = sum(t.numel() * t.element_size() for t in frames[0])
    # front end alone (crop + back-projection), device resident
    ms_front = _events_ms(lambda i: m.prepare_batch(*dev_frames[i % 3]), 10, 3) / 10
    return {"ms_per_step": ms / steps, "value": world * B * steps / (ms / 1e3), "batch_per_gpu": B,
            "e2e": {"value": world * B * steps / (ms_e2e / 1e3), "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": B * J * 12},
            "front_end_ms": ms_front, "front_end_frames_per_s": B / (ms_front / 1e3),
            "front_end_GBs": (B * 640 * 480 * 5 + B * (128 * 128 * 16 + 1024 * 12)) / (ms_front / 1e3) / 1e9}


# ------------------------------------------------------------------------------------------------ eager PyTorch on the same GPU
def cuda_eager_leg(dev, hosts_bf16, steps=5, warmup=2):
    """The reference's op chain as stock eager PyTorch on this GPU (cuBLAS / ATen), same inputs as the headline config (bf16 maps are
    up-cast once outside the timed region, as a reference user's fp32 backbone output would arrive).  -> samples/s."""
    from baseline import eager_torch_path as E
    from keypointfusion_b200 import ops
    from keypointfusion_b200.model.model import KPFusion
    from keypointfusion_b200.utils import synth
    net = KPFusion(joint_num=J)
    p = {k: v.to(dev) for k, v in synth.fill_state_dict(net, seed=0).items()}
    d = {k: v.to(dev) for k, v in hosts_bf16.items()}
    f = {k: d[k].float() for k in ("img_offset", "img_feat", "img_feat_rgb")}
    pcl = ops.getpcl(d["img"], d["center"], d["cube"], d["M"], d["cam"], 1024, seed=0)[0]   # (numpy on dataloader workers in the reference)
    B = d["img"].shape[0]

    def once(i):
        E.fusion_path(p, d["img"], pcl, f["img_offset"], f["img_feat"], f["img_feat_rgb"], d["center"], d["M"], d["cube"], d["cam"])
    torch.cuda.reset_peak_memory_stats(dev)
    ms = _events_ms(once, steps, warmup)
    return {"value": B * steps / (ms / 1e3), "unit": "samples/s", "ms_per_step": ms / steps, "kind": "eager PyTorch restatement of the "
            "reference's op chain (baseline/eager_torch_path.py), fp32, cuBLAS/ATen kernels, no CUDA graph", "steps": steps,
            "peak_mem_GB": round(torch.cuda.max_memory_allocated(dev) / 1e9, 2)}
