"""GPU: evaluation accumulated on the device (kpf_eval_accumulate, evaluation.Evaluator, runtime.GraphedEvalPath).  The accumulator is
exactly what the documented fixed-point conversion of kpf_eval_errors' outputs gives, independent of batch order and split, graph
capture, steps in flight and ranks; its means and PCK agree with the oracle's xyz2error / rigid_align."""
import os

import numpy as np
import pytest
import torch

from keypointfusion_b200.utils import synth
from oracle import kpf_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
THR = tuple(float(x) for x in range(51))


@pytest.fixture(scope="module")
def ops():
    from keypointfusion_b200 import ops as _ops
    return _ops


def cu(x):
    return (x if torch.is_tensor(x) else torch.from_numpy(np.asarray(x))).to(DEV)


def expected_acc(ops, errs, valid, thr, J):
    """The accumulator from eval_errors outputs: errs = [(err [B,J], pa [B,J]) f32 numpy per joint set], valid [B] bool."""
    T = len(thr)
    thr32 = np.asarray(thr, np.float32)
    acc = np.zeros((len(errs), ops.eval_row_length(J, T)), np.int64)
    for s, pair in enumerate(errs):
        acc[s, 0] = int(valid.sum())
        for k, e in enumerate(pair):
            e = e[valid]
            fin = np.isfinite(e)
            q = np.rint(np.minimum(np.where(fin, e, 0).astype(np.float64), 2.0 ** 20) * 2.0 ** 20).astype(np.int64)
            acc[s, 1 + k * J:1 + (k + 1) * J] = q.sum(0)
            acc[s, 1 + (2 + k) * J:1 + (3 + k) * J] = (~fin).sum(0)
            bins = np.where(fin, np.searchsorted(thr32, np.where(fin, e, 0).astype(np.float32), side="left"), T)
            acc[s, 1 + 4 * J + k * (T + 1):1 + 4 * J + (k + 1) * (T + 1)] = np.bincount(bins.ravel(), minlength=T + 1)
    return torch.from_numpy(acc)


def device_errors(ops, sets, gt, cube):
    out = []
    for p in sets:
        err, pa = ops.eval_errors(p, gt, cube)
        out.append((err.cpu().numpy(), pa.cpu().numpy()))
    return out


def random_batch(B, J, S, seed):
    rs = np.random.RandomState(seed)
    gt = rs.uniform(-0.8, 0.8, (B, J, 3)).astype(np.float32)
    sets = [(gt + rs.normal(0, 0.02 * (s + 1), (B, J, 3))).astype(np.float32) for s in range(S)]
    cube = rs.uniform(200, 300, (B, 3)).astype(np.float32)
    return sets, gt, cube


def test_accumulator_equals_documented_conversion_of_eval_errors(ops, golden):
    # random sets S = 3, B = 37 with masked rows, and the reference's rigid_align fixture (it includes a reflected sample)
    sets, gt, cube = random_batch(37, 21, 3, seed=5)
    valid = np.ones(37, bool)
    valid[[0, 9, 36]] = False
    A, Bt = golden["f4_A"], golden["f4_B"]
    n = A.shape[0]
    gsets = [A, Bt, (A + 0.01).astype(np.float32)]
    gvalid = np.array([True, True, False, True, True, True][:n])
    for sets_, gt_, cube_, valid_ in ((sets, gt, cube, valid), (gsets, Bt, np.full((n, 3), 250.0, np.float32), gvalid)):
        J = gt_.shape[1]
        dsets = [cu(p) for p in sets_]
        acc = torch.zeros(len(dsets), ops.eval_row_length(J, len(THR)), dtype=torch.int64, device=DEV)
        ops.eval_accumulate(acc, dsets, cu(gt_), cu(cube_), cu(valid_.astype(np.uint8)), THR)
        ref = expected_acc(ops, device_errors(ops, dsets, cu(gt_), cu(cube_)), valid_, THR, J)
        assert torch.equal(acc.cpu(), ref)
        assert int(acc[0, 0]) == int(valid_.sum())
        ops.eval_accumulate(acc, torch.stack(dsets), cu(gt_), cu(cube_), cu(valid_.astype(np.uint8)), THR)   # it adds
        assert torch.equal(acc.cpu(), 2 * ref)
        acc.zero_()
        ops.eval_accumulate(acc, dsets, cu(gt_), cu(cube_), None, THR)                                        # NULL mask: all valid
        assert torch.equal(acc.cpu(), expected_acc(ops, device_errors(ops, dsets, cu(gt_), cu(cube_)), np.ones(len(gt_), bool), THR, J))


def test_nonfinite_rows_and_clamp(ops):
    from keypointfusion_b200.evaluation import Evaluator
    B, J = 8, 21
    sets, gt, cube = random_batch(B, J, 2, seed=11)
    sets[0][2] = np.nan            # a whole NaN row: what an out-of-range frame_index gives the frame path (include/kpf_b200.h)
    sets[1][5, 4] = np.nan         # one NaN joint: its plain error, and every aligned error of that sample
    sets[1][6, 7, 0] = gt[6, 7, 0] + 8.0e4   # 8e4 normalised * 125 mm: a 10 km error, clamped to 2^20 mm in the sums
    cube[6] = 250.0
    ev = Evaluator(J, stage_names=("a", "b"), thresholds_mm=THR)
    ev.update([cu(p) for p in sets], cu(gt), cu(cube), None)
    acc = ev.acc.cpu()
    errs = device_errors(ops, [cu(p) for p in sets], cu(gt), cu(cube))
    assert torch.equal(acc, expected_acc(ops, errs, np.ones(B, bool), THR, J))
    T, R0 = len(THR), 1 + 4 * J
    nf = lambda s, k: acc[s, 1 + (2 + k) * J:1 + (3 + k) * J]
    hist = lambda s, k: acc[s, R0 + k * (T + 1):R0 + (k + 1) * (T + 1)]
    assert torch.equal(nf(0, 0), torch.ones(J, dtype=torch.int64)) and torch.equal(nf(0, 1), torch.ones(J, dtype=torch.int64))
    assert int(nf(1, 0).sum()) == 1 and int(nf(1, 0)[4]) == 1 and torch.equal(nf(1, 1), torch.ones(J, dtype=torch.int64))
    assert int(hist(0, 0)[T]) >= J and int(hist(1, 0)[T]) >= 2          # NaN joints and the 10 km joint are in bin T
    assert int(hist(0, 0).sum()) == B * J and int(hist(1, 1).sum()) == B * J
    assert float(errs[1][0][6, 7]) > 2.0 ** 20
    finite_sum_b7 = int(np.rint(errs[1][0][:, 7].astype(np.float64) * 2 ** 20)[[0, 1, 2, 3, 4, 5, 7]].sum())
    assert int(acc[1, 1 + 7]) == finite_sum_b7 + 2 ** 40                 # the clamped joint adds exactly 2^20 mm
    st = ev.summary()
    assert st["a"]["nonfinite"] == J and st["b"]["nonfinite"] == 1 and st["b"]["pa_nonfinite"] == J
    assert np.isfinite(st["a"]["mean_error_mm"]) and np.isfinite(st["b"]["pa_mean_error_mm"])


def test_totals_do_not_depend_on_batch_order_split_or_padding(ops):
    from keypointfusion_b200.evaluation import Evaluator
    B, J, S = 64, 21, 5
    sets, gt, cube = random_batch(B, J, S, seed=23)
    one = Evaluator(J)
    one.update(cu(np.stack(sets)), cu(gt), cu(cube))
    split = Evaluator(J)
    perm = np.random.RandomState(1).permutation(B)
    P = np.stack(sets)
    for lo, hi in ((0, 7), (7, 27), (27, 28), (28, 44), (44, 64)):
        idx = perm[lo:hi]
        pad = 5                                               # padding rows: garbage (NaN included) masked out through valid
        p = np.concatenate([P[:, idx], np.full((S, pad, J, 3), np.nan, np.float32)], axis=1)
        g = np.concatenate([gt[idx], np.zeros((pad, J, 3), np.float32)])
        c = np.concatenate([cube[idx], np.ones((pad, 3), np.float32)])
        v = np.concatenate([np.ones(len(idx), np.uint8), np.zeros(pad, np.uint8)])
        split.update(cu(p), cu(g), cu(c), cu(v))
    assert torch.equal(one.acc, split.acc)


def test_summary_agrees_with_the_oracle(ops):
    from keypointfusion_b200.evaluation import Evaluator
    B, J = 64, 21
    sets, gt, cube = random_batch(B, J, 2, seed=31)
    center = np.zeros((B, 3))
    oracle = []
    for p in sets:
        e = O.xyz2error(p, gt, center, cube)
        pa = O.xyz2error(np.stack([O.rigid_align(p[b].astype(np.float64), gt[b].astype(np.float64)) for b in range(B)]), gt, center, cube)
        oracle.append((e, pa))
    # samples with an error within 1e-3 mm of a threshold are masked out: there fp32 and fp64 may fall on either side
    near = np.zeros(B, bool)
    for e, pa in oracle:
        for x in (e, pa):
            near |= (np.abs(x[..., None] - np.asarray(THR)) <= 1e-3).any(axis=(1, 2))
    valid = ~near
    assert valid.sum() > B // 2
    ev = Evaluator(J, stage_names=("a", "b"), thresholds_mm=THR)
    ev.update([cu(p) for p in sets], cu(gt), cu(cube), cu(valid.astype(np.uint8)))
    st = ev.summary()
    for name, (e, pa) in zip(("a", "b"), oracle):
        e, pa = e[valid], pa[valid]
        assert abs(st[name]["mean_error_mm"] - e.mean()) <= 1e-4
        assert abs(st[name]["pa_mean_error_mm"] - pa.mean()) <= 1e-3
        np.testing.assert_allclose(st[name]["per_joint_error_mm"], e.mean(0), atol=1e-4, rtol=0)
        np.testing.assert_array_equal(st[name]["pck"], (e[..., None] <= np.asarray(THR)).mean(axis=(0, 1)))
        np.testing.assert_array_equal(st[name]["pa_pck"], (pa[..., None] <= np.asarray(THR)).mean(axis=(0, 1)))
        assert st[name]["samples"] == int(valid.sum())


# ------------------------------------------------------------------------------------------------ graphs
@pytest.fixture(scope="module")
def net(path_params):
    from keypointfusion_b200.model.model import KPFusion
    n = KPFusion(joint_num=21)
    n.load_state_dict(path_params, strict=False)
    return n.to(DEV).eval()


def make(B, seed):
    inp = synth.make_inputs(B, 128, 21, 128, seed=seed)
    for k in ("img_feat", "img_feat_rgb", "img_offset"):
        inp[k] = inp[k].bfloat16()
    inp.pop("img_rgb")
    rs = np.random.RandomState(seed)
    inp["gt"] = torch.from_numpy(rs.uniform(-0.3, 0.3, (B, 21, 3)).astype(np.float32))
    valid = np.ones(B, np.uint8)
    valid[rs.randint(B)] = 0
    inp["valid"] = torch.from_numpy(valid)
    return inp


def eager_update(net, ev, d):
    from keypointfusion_b200 import ops
    from keypointfusion_b200.dataloader.loader import loader
    from keypointfusion_b200.evaluation import stage_joints
    L = loader(img_size=128)
    with torch.no_grad():
        pcl, _ = ops.getpcl(d["img"], d["center"], d["cube"], d["M"], d["cam"], 1024, seed=0)
        res, _, _ = net.forward_path(d["img_offset"], d["img_feat"], None, d["img_feat_rgb"], d["img"], pcl, L, d["center"], d["M"], d["cube"],
                                     d["cam"], 0.8)
        sets = stage_joints(res, d["img"], d["center"], d["M"], d["cube"], d["cam"], L)
        ev.update(sets, d["gt"], d["cube"], d["valid"])
    return res, sets


def test_graphed_eval_path_overlapped_and_pipelined_match_eager(net):
    from keypointfusion_b200.dataloader.loader import loader
    from keypointfusion_b200.evaluation import Evaluator
    from keypointfusion_b200.runtime import GraphedEvalPath, OverlappedSteps, PipelinedRunner
    B = 6
    hosts = [make(B, 900 + i) for i in range(3)]
    devs = [{k: v.to(DEV) for k, v in h.items()} for h in hosts]
    ldr = loader(img_size=128)
    ref = Evaluator(21)
    for d in devs:
        eager_update(net, ref, d)
    # three replays of one graph (static buffers); construction (warm-up steps) leaves the accumulator as it was
    ev = Evaluator(21)
    g = GraphedEvalPath(net, ldr, devs[0], evaluator=ev, sample_num=1024, kernel=0.8, seed=0)
    assert int(ev.acc.abs().sum()) == 0
    for d in devs:
        g(d)
    assert torch.equal(ev.acc, ref.acc)
    # two steps in flight on two streams, both graphs adding into one accumulator
    ev2 = Evaluator(21)
    paths = [GraphedEvalPath(net, ldr, {k: v.clone() for k, v in d.items()}, evaluator=ev2, bind=True) for d in devs[:2]]
    ov = OverlappedSteps(paths, n_streams=2)
    ov.fork()
    for _ in range(4):
        ov.submit()
    ov.join()
    serial = Evaluator(21)
    for d in devs[:2] * 2:
        eager_update(net, serial, d)
    assert torch.equal(ev2.acc, serial.acc)
    # the host-fed pipelined runner, two graphs sharing one evaluator
    ev3 = Evaluator(21)
    runner = PipelinedRunner(net, ldr, devs[0], path_cls=GraphedEvalPath, evaluator=ev3, sample_num=1024, kernel=0.8, seed=0)
    slots = [runner.submit({k: v.pin_memory() for k, v in h.items()}) for h in hosts[:2]]
    runner.fetch(slots[0]), runner.fetch(slots[1])
    runner.fetch(runner.submit({k: v.pin_memory() for k, v in hosts[2].items()}))
    assert torch.equal(ev3.acc, ref.acc)
    a, b = ev3.summary(), ref.summary()
    for stage in a:
        for k in a[stage]:
            np.testing.assert_array_equal(a[stage][k], b[stage][k])


def test_stage_joints_offset_stage_is_the_networks_conversion(net, ops):
    from keypointfusion_b200.dataloader.loader import loader
    from keypointfusion_b200.evaluation import Evaluator
    d = {k: v.to(DEV) for k, v in make(4, 77).items()}
    res, sets = eager_update(net, Evaluator(21), d)
    L = loader(img_size=128)
    direct = ops.uvd2xyz(ops.offset2joint_weight(d["img_offset"], d["img"], 0.8), d["center"], d["M"], d["cube"], d["cam"], L.img_size, L.flip)
    assert torch.equal(sets[0], direct)
    assert all(s is r for s, r in zip(sets[1:], res[2:]))


def test_opcheck_eval_accumulate(ops):
    from torch.library import opcheck
    sets, gt, cube = random_batch(9, 21, 3, seed=3)
    acc = torch.zeros(3, ops.eval_row_length(21, len(THR)), dtype=torch.int64, device=DEV)
    valid = cu(np.array([1, 1, 0, 1, 1, 1, 1, 0, 1], np.uint8))
    opcheck(torch.ops.kpf.eval_accumulate.default, (acc, cu(np.stack(sets)), cu(gt), cu(cube), valid, list(THR)),
            test_utils=("test_schema", "test_faketensor"))


# ------------------------------------------------------------------------------------------------ two ranks
def _worker(rank, world, port, q):
    import torch.distributed as dist
    from keypointfusion_b200.evaluation import Evaluator
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world, device_id=dev)
    try:
        B, J = 64, 21
        sets, gt, cube = random_batch(B, J, 5, seed=41)
        P = torch.from_numpy(np.stack(sets)).to(dev)
        g, c = torch.from_numpy(gt).to(dev), torch.from_numpy(cube).to(dev)
        lo, hi = rank * B // world, (rank + 1) * B // world
        mine = Evaluator(J, device=dev)
        mine.update(P[:, lo:hi], g[lo:hi], c[lo:hi])
        alone = Evaluator(J, device=dev)
        alone.update(P, g, c)
        a, b = mine.summary(dist.group.WORLD), alone.summary()
        ok = all(np.array_equal(np.asarray(a[s][k]), np.asarray(b[s][k]), equal_nan=True) for s in a for k in a[s])
        q.put((rank, bool(ok)))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_ranks_sum_to_one_rank():
    import torch.multiprocessing as mp
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() + 7) % 1000
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(600)
    res = sorted(q.get(timeout=10) for _ in range(world))
    assert res == [(0, True), (1, True)], res
