"""Stream / CUDA-graph runtime for the fusion path: one captured graph per (batch, crop) shape replays the whole
post-backbone path (K1 -> K4a -> a5 -> K2 -> 2 x Block_KPFusion) with zero per-kernel host work, and a batch-sharded
multi-GPU wrapper whose only collective is the all-gather of the per-sample joints (SURVEY.md 8e)."""
import torch

from . import ops


class _GraphedPath:
    """What the graphed paths share: the step's inputs (KEYS) in static device buffers, a warm-up of `_run` on a private stream,
    one `_run` captured on that same stream into `graph` (its outputs in `out`, the kernels of ours it launches counted in
    `launches_per_replay`), and `__call__`, which stages a step's inputs and replays."""
    KEYS = ()
    FETCH = ()   # the outputs PipelinedRunner copies back to the host

    def _warm_up(self, net, example, warmup, bind):
        """bind=True: the static buffers are the caller's own (device-resident, contiguous) `example` tensors, so a replay reads
        whatever they hold at that time; otherwise they are private copies of `example` on the network's device."""
        dev = next(net.parameters()).device
        if bind:
            assert all(example[k].is_cuda and example[k].is_contiguous() for k in self.KEYS), "bind=True needs contiguous device tensors"
            self.static = {k: example[k] for k in self.KEYS}
        else:
            self.static = {k: torch.empty_like(example[k], device=dev).copy_(example[k]) for k in self.KEYS}
        self.stream = torch.cuda.Stream(device=dev)
        self.stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(self.stream), torch.no_grad():
            for _ in range(warmup):  # packed weight caches, device constants and backbone algorithm choices are built before capture
                self._run()
        torch.cuda.current_stream(dev).wait_stream(self.stream)
        torch.cuda.synchronize(dev)

    def _capture(self):
        self.graph = torch.cuda.CUDAGraph()
        n0 = ops.launch_count()
        # captured on the warm-up stream: per-stream persistent workspaces (ops._zero_counters) already exist, so no fill node
        # lands inside the graph (it would also cut the programmatic-launch chain between two kernels)
        with torch.no_grad(), torch.cuda.graph(self.graph, stream=self.stream):
            self.out = self._run()
        self.launches_per_replay = ops.launch_count() - n0

    def __call__(self, inputs=None):
        if inputs is not None:
            for k in self.KEYS:
                self.static[k].copy_(inputs[k], non_blocking=True)
        self.graph.replay()
        return self.out


class GraphedFusionPath(_GraphedPath):
    """Capture `getpcl + KPFusion.forward_path` once; `__call__` copies a step's inputs into the static buffers (device to
    device, or pinned host to device) and replays.  Inputs: dict with img [B,1,S,S] f32, img_feat / img_feat_rgb [B,128,H,H],
    img_offset [B,5J,H,H] (bf16 or f32), center [B,3], M [B,3,3], cube [B,3], cam [B,4].  `out` holds joints (the final joints),
    result and spatial_weight (forward_path's lists) and pcl (the sampled point cloud)."""
    KEYS = ("img", "img_feat", "img_feat_rgb", "img_offset", "center", "M", "cube", "cam")
    FETCH = ("joints",)

    def __init__(self, net, loader, example, sample_num=1024, kernel=0.8, seed=0, warmup=2, chains=1, bind=False, exchange=None):
        """chains must be 1: a step is one chain of kernels on one stream.  Batches share the GPU by keeping several steps in
        flight (OverlappedSteps).  bind=True: capture directly over the caller's (device-resident) `example` tensors instead of
        private static buffers; `__call__()` then replays with no staging copy and reads whatever those tensors hold at replay time."""
        if chains != 1:
            raise ValueError(f"chains={chains}: a step is one kernel chain; keep several steps in flight with OverlappedSteps instead")
        self.net, self.loader, self.sample_num, self.kernel, self.seed = net, loader, sample_num, kernel, seed
        self.exchange = exchange    # a PeerExchange: the fused all-gather of the joints is part of the captured graph
        self._warm_up(net, example, warmup, bind)
        if exchange is not None:
            with torch.cuda.stream(self.stream):
                exchange.flush()    # complete the last warm-up step's gather
            exchange.sync_ranks()   # every rank has finished the same number of (exchanging) warm-up steps before anyone captures
        self._capture()

    def _run(self):
        s = self.static
        if self.exchange is not None:
            self.exchange.begin_step()   # completes the PREVIOUS step's gather (normally already there) and opens this one
        pcl, _ = ops.getpcl(s["img"], s["center"], s["cube"], s["M"], s["cam"], self.sample_num, seed=self.seed)
        res, sw, _ = self.net.forward_path(s["img_offset"], s["img_feat"], None, s["img_feat_rgb"], s["img"], pcl, self.loader, s["center"],
                                           s["M"], s["cube"], s["cam"], self.kernel, exchange=self.exchange)
        return dict(joints=res[-1], result=res, spatial_weight=sw, pcl=pcl)


class GraphedFramePath(_GraphedPath):
    """Frames to keypoints as one captured graph: the crop front end (demo_RGBD.Model_RGBD.prepare_batch), the two stock-PyTorch
    backbones, KPFusion.forward_path and joints_to_frame, over static buffers rgb [F,Hf,Wf,3] uint8, depth [F,Hf,Wf] uint16 (or
    int16 with the same bits), bbox [B,4] f64 and frame_index [B] int32 (box b is in frame frame_index[b]).  `out` holds joints
    (normalised), joints_uvd_frame (frame pixels, depth mm), joints_xyz_cam (camera mm) and the full result list.

    A step has a fixed (F, B) shape.  A caller with fewer hands in a step repeats a box (any valid frame / box pair) and ignores
    the extra rows.  frame_index lives on the device, so it is not range-checked per step: an index outside [0,F) gives NaN
    keypoints for that hand only (include/kpf_b200.h)."""
    KEYS = ("rgb", "depth", "bbox", "frame_index")
    FETCH = ("joints_uvd_frame", "joints_xyz_cam")

    def __init__(self, net, loader, example, cam_para=(617.0, 617.0, 312.0, 241.0), cube=(250, 250, 250), img_size=128, sample_num=1024,
                 seed=0, warmup=2, bind=False):
        """net: KPFusion with backbones; loader: the geometry helper passed to the network (None: a loader(img_size)).
        bind=True: capture over the caller's device tensors `example` (as GraphedFusionPath)."""
        from .demo_RGBD import Model_RGBD
        assert example["frame_index"].dtype == torch.int32, "frame_index must be int32"
        self.model = Model_RGBD(net, cam_para=cam_para, cube=cube, img_size=img_size, sample_num=sample_num, seed=seed)
        if loader is not None:
            self.model.depthloader = loader
        self._warm_up(net, example, warmup, bind)
        self._capture()

    def _run(self):
        s = self.static
        res, b = self.model.estimate_pose_RGBD(s["rgb"], s["depth"], s["bbox"], s["frame_index"])
        return dict(joints=res[-1], joints_uvd_frame=b["joints_uvd_frame"], joints_xyz_cam=b["joints_xyz_cam"], result=res)


class OverlappedSteps:
    """Keep `n_streams` consecutive steps (independent batches) in flight: step i is replayed on stream i % n_streams.  The path is a
    long dependent chain of latency-bound kernels, several of which use only part of the machine (a token stack is one CTA per
    sample: 64 of 148 SMs at batch 64), so a second step's kernels fill the idle SMs: +13-15 % samples/s at batch 64 (measured,
    profiles/probe_overlap_steps.py).  `paths`: GraphedFusionPath objects captured with bind=True; path j must always run on the
    same stream (len(paths) % n_streams == 0), which also keeps a PeerExchange bound to one stream."""

    def __init__(self, paths, n_streams=2):
        assert len(paths) % n_streams == 0
        self.paths, self.n = list(paths), n_streams
        dev = paths[0].static["img"].device
        self.streams = [torch.cuda.Stream(device=dev) for _ in range(n_streams)]
        self.i = 0

    def fork(self):
        """the streams start after everything already enqueued on the current stream"""
        ev = torch.cuda.Event()
        ev.record()
        for s in self.streams:
            s.wait_event(ev)

    def submit(self):
        p = self.paths[self.i % len(self.paths)]
        with torch.cuda.stream(self.streams[self.i % self.n]):
            p.graph.replay()
        self.i += 1
        return p.out

    def join(self):
        """the current stream continues after every step submitted so far"""
        cur = torch.cuda.current_stream()
        for s in self.streams:
            cur.wait_stream(s)


def all_gather_joints(joints, out=None):
    """The path's one exchange step: [B_local,J,3] per rank -> [world*B_local,J,3] on every rank (NCCL over NVLink)."""
    import torch.distributed as dist
    if not dist.is_initialized() or dist.get_world_size() == 1:
        return joints
    joints = joints.contiguous()
    if out is None:
        out = joints.new_empty((dist.get_world_size() * joints.shape[0],) + tuple(joints.shape[1:]))
    dist.all_gather_into_tensor(out, joints)
    return out


class PeerExchange:
    """The path's one exchange step without NCCL: every rank's final kernel stores its [B_local,J,3] joints straight into EVERY rank's
    gathered tensor over NVLink (peer stores into symmetric memory) and counts the samples as arrived; `wait()` enqueues the one-thread
    kernel that holds the stream until all `world * B_local` samples of the step are there (include/kpf_b200.h: kpf_exchange_wait).
    The gathered tensor is double buffered by step parity, so a fast rank's next step never overwrites what a slow rank still reads.

    Symmetric memory comes from torch.distributed._symmetric_memory (CUDA IPC / fabric handles over NVLink on one node); all ranks
    must construct this collectively and run the same number of steps."""
    HEADER_FLOATS = 16

    def __init__(self, b_local, joints, device, group=None):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        self.group = group if group is not None else dist.group.WORLD
        self.world, self.rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        self.b_local, self.J = int(b_local), int(joints)
        self.rows_total, self.row0 = self.world * self.b_local, self.rank * self.b_local
        half = self.rows_total * self.J * 3
        self.buf = symm.empty(self.HEADER_FLOATS + 2 * half, dtype=torch.float32, device=device)
        self.buf.zero_()
        self.handle = symm.rendezvous(self.buf, self.group)
        self.peer_ptrs = torch.tensor([int(p_) for p_ in self.handle.buffer_ptrs], dtype=torch.int64, device=device)
        self.xstep = torch.zeros(1, dtype=torch.int32, device=device)      # steps completed (device side: graph replays advance it)
        self.inflight = torch.zeros(1, dtype=torch.int32, device=device)   # a step's joints are on their way
        self.halves = [self.buf[self.HEADER_FLOATS + h * half:self.HEADER_FLOATS + (h + 1) * half].view(self.rows_total, self.J, 3) for h in (0, 1)]
        torch.cuda.synchronize(device)
        self.sync_ranks()

    def sync_ranks(self):
        import torch.distributed as dist
        torch.cuda.synchronize(self.buf.device)
        dist.barrier(self.group)

    def begin_step(self):
        """Enqueue at the START of a step: completes the previous step's gather if one is in flight (the other ranks finished it long
        ago, so this normally does not stall) and opens the new step."""
        ops.exchange_wait(self.buf, self.xstep, self.rows_total, self.inflight)

    def flush(self):
        """Complete the step in flight (end of a run, or before the gathered tensor is read)."""
        ops.exchange_wait(self.buf, self.xstep, self.rows_total, self.inflight, flush=True)

    def gathered(self):
        """[world * B_local, J, 3] joints of the most recently COMPLETED step (call flush() first to complete the one in flight);
        reads the device step counter (one host sync)."""
        done = int(self.xstep.item())
        return self.halves[(done - 1) & 1]


def shard_batch(n_items, rank, world):
    """Contiguous per-rank slice [lo, hi) of a global batch (sample r*B/G .. (r+1)*B/G, SURVEY.md 8e); remainders go to low ranks."""
    base, rem = divmod(n_items, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class InputArena:
    """One contiguous byte buffer holding every input of a step at fixed 256-byte aligned offsets, with typed views per key.
    A pinned host arena and a device arena of the same layout turn the per-step upload into ONE cudaMemcpyAsync (55 GB/s on
    this box; the same bytes as eight separate copies reach 43-52 GB/s)."""

    def __init__(self, example, keys, device=None, pinned=False):
        self.layout, off = {}, 0
        for k in keys:
            t = example[k]
            n = t.numel() * t.element_size()
            self.layout[k] = (off, n, t.dtype, tuple(t.shape))
            off = (off + n + 255) // 256 * 256
        self.nbytes = off
        self.buf = torch.empty(off, dtype=torch.uint8, device=device) if device is not None else torch.empty(off, dtype=torch.uint8)
        if pinned:
            self.buf = self.buf.pin_memory()
        self.views = {k: self.buf[o:o + n].view(dt).view(shape) for k, (o, n, dt, shape) in self.layout.items()}


class PipelinedRunner:
    """Host-fed serving loop: two captured graphs, each bound to its own device input arena; while graph[i % 2] computes step i
    on the compute stream, a copy stream uploads step i+1's pinned host inputs into the other arena, and the host reads step
    i-1's results from pinned memory.  Every step still does its own H2D of all inputs and its own D2H of the result.
    `new_host_inputs()` hands the caller a dict of pinned views (one arena): filling those and passing the dict to `submit`
    uploads a step with a single copy; any other dict of host tensors is uploaded tensor by tensor.

    path_cls: GraphedFusionPath (crops + backbone maps in, normalised joints out) or GraphedFramePath (frames, boxes and
    frame_index in, keypoints in frame pixels and camera mm out); `example` holds that class's KEYS and `kw` go to it."""

    def __init__(self, net, loader, example, path_cls=GraphedFusionPath, **kw):
        dev = next(net.parameters()).device
        self.dev = dev
        self.keys = keys = path_cls.KEYS
        self.arenas = [InputArena(example, keys, device=dev) for _ in range(2)]
        for a in self.arenas:
            for k in keys:
                a.views[k].copy_(example[k])
        self.paths = [path_cls(net, loader, a.views, bind=True, **kw) for a in self.arenas]
        self._example = {k: example[k] for k in keys}
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.copied = [torch.cuda.Event() for _ in range(2)]
        self.done = [torch.cuda.Event() for _ in range(2)]
        self.fetch_keys = path_cls.FETCH
        outs = self.paths[0].out
        self.host_out = [[torch.empty(outs[k].shape, dtype=outs[k].dtype).pin_memory() for k in self.fetch_keys] for _ in range(2)]
        self.step = 0
        for e in self.done:
            e.record(torch.cuda.current_stream(dev))

    def new_host_inputs(self):
        """A dict of pinned host tensors (views of one arena laid out like the device arenas) for the caller to fill."""
        a = InputArena(self._example, self.keys, pinned=True)
        d = dict(a.views)
        d["_arena"] = a.buf
        return d

    def submit(self, host_inputs):
        """Enqueue one step (returns immediately); `fetch()` later returns results in submission order."""
        s = self.step % 2
        path = self.paths[s]
        main = torch.cuda.current_stream(self.dev)
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.done[s])          # the previous user of this buffer set has finished
            arena = host_inputs.get("_arena")
            if arena is not None and arena.numel() == self.arenas[s].nbytes:
                self.arenas[s].buf.copy_(arena, non_blocking=True)    # one upload for the whole step
            else:
                for k in path.KEYS:
                    path.static[k].copy_(host_inputs[k], non_blocking=True)
            self.copied[s].record(self.copy_stream)
        main.wait_event(self.copied[s])
        path.graph.replay()
        for h, k in zip(self.host_out[s], self.fetch_keys):
            h.copy_(path.out[k], non_blocking=True)
        self.done[s].record(main)
        self.step += 1
        return s

    def fetch(self, slot):
        """Block until the step submitted into `slot` is complete; returns its result (pinned host memory): the joints for
        GraphedFusionPath, the tuple (joints_uvd_frame, joints_xyz_cam) for GraphedFramePath."""
        self.done[slot].synchronize()
        h = self.host_out[slot]
        return h[0] if len(h) == 1 else tuple(h)
