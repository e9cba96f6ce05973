"""GPU: several hands per frame through frame_index, and keypoints returned in frame pixels and camera millimetres.

An indexed batch must equal, bit for bit, the route that duplicates each hand's frame (frame_index=None on depth[frame_index]);
joints_to_frame must equal the CPU restatement (tests/frames_oracle.py) bit for bit and agree with xyz2uvd / uvd2xyz; the graphed
frames path and the pipelined runner must reproduce the eager call."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)
import frames_oracle as FO  # noqa: E402

G = os.path.join(HERE, "golden", "golden_crop.npz")
DEV = "cuda"


@pytest.fixture(scope="module")
def gc():
    return dict(np.load(G))


def u16(a):
    """uint16 depth as int16 with the same bits (the front end reads either; int16 has full indexing support)"""
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int16)).to(DEV)


def syn_frames(gc):
    """The three synthetic 640x480 frames with 2-3 boxes each (the fixture's box plus shifted / resized copies) and a
    non-monotonic frame_index."""
    fi = [1, 0, 1, 2, 0, 2, 1]
    shift = {0: (0, 0, 0, 0), 1: (-30, 12, 10, 6), 2: (25, -18, -8, 4)}
    seen, boxes = {}, []
    for f in fi:
        k = seen.get(f, 0)
        seen[f] = k + 1
        boxes.append(gc["syn_bbox"][f] + np.array(shift[k]))
    rgb = torch.from_numpy(gc["syn_rgb"]).to(DEV)
    return rgb, u16(gc["syn_depth"]), torch.from_numpy(np.stack(boxes)).to(DEV), fi


def golden_frame(gc):
    """The real frame of golden_crop.npz with its box and a second box on the same frame."""
    rgb = torch.from_numpy(gc["box_rgb"][None]).to(DEV)
    bbox = np.stack([gc["box_bbox"], gc["box_bbox"] + np.array([60.0, -40.0, -20.0, 10.0])])
    return rgb, u16(gc["box_depth"][None]), torch.from_numpy(bbox).to(DEV), [0, 0]


def assert_batches_equal(a, b):
    for k in ("center_uvd", "img", "M", "center", "img_rgb", "pcl", "cube", "cam_para"):
        assert torch.equal(a[k], b[k]), k


@pytest.mark.parametrize("frames", ["golden", "synthetic"])
def test_indexed_equals_duplicated_bit_for_bit(gc, frames):
    from keypointfusion_b200.demo_RGBD import Model_RGBD
    rgb, depth, bbox, fi = golden_frame(gc) if frames == "golden" else syn_frames(gc)
    cam = tuple(gc["box_cam"] if frames == "golden" else gc["syn_cam"])
    fe = Model_RGBD(None, cam_para=cam, seed=3)
    idx = torch.tensor(fi, device=DEV)
    dup = fe.prepare_batch(rgb[idx].contiguous(), depth[idx].contiguous(), bbox)
    assert dup["frame_index"] is None
    for given in (fi, np.array(fi), torch.tensor(fi), torch.tensor(fi, dtype=torch.int32, device=DEV)):
        got = fe.prepare_batch(rgb, depth, bbox, frame_index=given)
        assert got["frame_index"].dtype == torch.int32 and got["frame_index"].is_cuda
        assert_batches_equal(got, dup)
    if frames == "golden":   # the fixture's own box, read through the index, still gives the reference's crops exactly
        from keypointfusion_b200 import ops
        c = torch.from_numpy(np.stack([gc["box_center"]] * 2))
        img, _, _, _ = ops.crop_depth(depth, c, [250, 250, 250], gc["box_cam"], frame_index=fi)
        r = ops.crop_rgb(rgb, c, [250, 250, 250], gc["box_cam"], frame_index=fi)
        assert np.array_equal(img[0, 0].cpu().numpy(), gc["box_crop_d"])
        assert np.array_equal(r[0].cpu().numpy(), gc["box_crop_rgb"])


def test_out_of_range_device_index_gives_nan_for_that_box_only(gc):
    from keypointfusion_b200 import ops
    rgb, depth, bbox, _ = syn_frames(gc)
    bbox = bbox[:4]
    good = [2, 0, 1, 1]
    cube, cam = [250, 250, 250], gc["syn_cam"]
    ref_c = ops.center_from_bbox(depth, bbox, frame_index=good)
    ref = ops.crop_depth(depth, ref_c, cube, cam, frame_index=good)
    ref_rgb = ops.crop_rgb(rgb, ref_c, cube, cam, frame_index=good)
    for bad_value in (3, -1, 1 << 30):
        fi = torch.tensor([2, bad_value, 1, 1], dtype=torch.int32, device=DEV)
        c = ops.center_from_bbox(depth, bbox, frame_index=fi)
        img, M, com3d, _ = ops.crop_depth(depth, ref_c, cube, cam, frame_index=fi)
        r = ops.crop_rgb(rgb, ref_c, cube, cam, frame_index=fi)
        for got, want in ((c, ref_c), (img, ref[0]), (M, ref[1]), (com3d, ref[2]), (r, ref_rgb)):
            assert bool(torch.isnan(got[1]).all())
            keep = [0, 2, 3]
            assert torch.equal(got[keep], want[keep])
    torch.cuda.synchronize()   # no fault from the launches above


def test_host_index_out_of_range_raises_before_any_launch(gc):
    from keypointfusion_b200 import ops
    rgb, depth, bbox, _ = syn_frames(gc)
    n0 = ops.launch_count()
    for bad in ([0, 1, 3, 0, 0, 0, 0], [0, -1, 1, 0, 0, 0, 0], torch.tensor([0, 1, 2, 3, 0, 0, 0])):
        with pytest.raises(ValueError):
            ops.center_from_bbox(depth, bbox, frame_index=bad)
        with pytest.raises(ValueError):
            ops.crop_rgb(rgb, torch.zeros(7, 3, dtype=torch.float64, device=DEV), [250, 250, 250], gc["syn_cam"], frame_index=bad)
    with pytest.raises(ValueError):   # no index: one frame per box
        ops.center_from_bbox(depth, bbox)
    assert ops.launch_count() == n0


def _frame_inputs(gc):
    from keypointfusion_b200.demo_RGBD import Model_RGBD
    rgb, depth, bbox, fi = syn_frames(gc)
    return Model_RGBD(None, cam_para=tuple(gc["syn_cam"]), seed=1).prepare_batch(rgb, depth, bbox, frame_index=fi)


@pytest.mark.parametrize("flip", [1.0, -1.0])
def test_joints_to_frame_matches_restatement_and_crop_geometry(gc, flip):
    from keypointfusion_b200 import ops
    b = _frame_inputs(gc)
    B = b["center"].shape[0]
    joints = (torch.rand(B, 21, 3, generator=torch.Generator().manual_seed(5)) * 1.6 - 0.8).to(DEV)
    uvd, xyz = ops.joints_to_frame(joints, b["center"], b["cube"], b["cam_para"], flip)
    ruvd, rxyz = FO.joints_to_frame(joints.cpu().numpy(), b["center"].cpu().numpy(), b["cube"].cpu().numpy(), b["cam_para"].cpu().numpy(), flip)
    assert np.array_equal(uvd.cpu().numpy(), ruvd) and np.array_equal(xyz.cpu().numpy(), rxyz)
    K = torch.ops.kpf
    cuvd, cxyz = K.joints_to_frame(joints, b["center"], b["cube"], b["cam_para"], flip)
    assert torch.equal(cuvd, uvd) and torch.equal(cxyz, xyz)
    # M . [u, v, 1] lands on the crop pixel (uvd_nl + 1) * S / 2 of xyz2uvd
    S = 128
    uvd_nl = ops.xyz2uvd(joints, b["center"], b["M"], b["cube"], b["cam_para"], S, flip)
    hom = torch.cat([uvd[..., :2], torch.ones_like(uvd[..., :1])], -1).double()
    crop_px = torch.einsum("bij,bpj->bpi", b["M"].double(), hom)[..., :2]
    assert float((crop_px - (uvd_nl[..., :2].double() + 1) * S / 2).abs().max()) <= 1e-3
    # ... and uvd2xyz brings the joints back
    back = ops.uvd2xyz(uvd_nl, b["center"], b["M"], b["cube"], b["cam_para"], S, flip)
    assert float((back - joints).abs().max()) <= 1e-4


def test_estimate_pose_indexed_equals_duplicated(gc):
    import bench_extra
    from keypointfusion_b200.demo_RGBD import Model_RGBD
    rgb, depth, bbox, fi = syn_frames(gc)
    m = Model_RGBD(bench_extra.build_full_net(DEV), cam_para=tuple(gc["syn_cam"]))
    idx = torch.tensor(fi, device=DEV)
    res_d, bd = m.estimate_pose_RGBD(rgb[idx].contiguous(), depth[idx].contiguous(), bbox)
    res_i, bi = m.estimate_pose_RGBD(rgb, depth, bbox, frame_index=fi)
    assert len(res_i) == len(res_d)
    for a, c in zip(res_i, res_d):
        assert torch.equal(a, c)
    for k in ("joints_uvd_frame", "joints_xyz_cam"):
        assert torch.equal(bi[k], bd[k]), k
    assert torch.equal(bi["joints_uvd_frame"], m.to_frame(res_i[-1], bi)[0])


def test_graphed_frame_path_and_runner_match_eager(gc):
    import bench_extra
    from keypointfusion_b200.demo_RGBD import Model_RGBD
    from keypointfusion_b200.runtime import GraphedFramePath, PipelinedRunner
    net = bench_extra.build_full_net(DEV)
    cam = tuple(gc["syn_cam"])
    rgb, depth, bbox, fi = syn_frames(gc)
    sets = []
    for s in range(2):   # two different frame sets of the same (F, B) shape
        flip_rows = torch.flip(rgb, [1]) if s else rgb
        sets.append(dict(rgb=flip_rows.contiguous(), depth=torch.roll(depth, 7 * s, 2).contiguous(), bbox=bbox + 3.0 * s,
                         frame_index=torch.tensor(fi if s == 0 else fi[::-1], dtype=torch.int32, device=DEV)))
    m = Model_RGBD(net, cam_para=cam)
    ref = []
    for d in sets:
        _, b = m.estimate_pose_RGBD(d["rgb"], d["depth"], d["bbox"], d["frame_index"])
        ref.append((b["joints_uvd_frame"].clone(), b["joints_xyz_cam"].clone()))
    g = GraphedFramePath(net, None, sets[0], cam_para=cam)
    for d, r in zip(sets, ref):
        out = g(d)
        assert torch.equal(out["joints_uvd_frame"], r[0]) and torch.equal(out["joints_xyz_cam"], r[1])
    runner = PipelinedRunner(net, None, sets[0], path_cls=GraphedFramePath, cam_para=cam)
    hosts = []
    for d in sets:
        h = runner.new_host_inputs()
        for k in GraphedFramePath.KEYS:
            h[k].copy_(d[k])
        hosts.append(h)
    order = [0, 1, 1, 0]
    slots, outs = [], []
    for i in order:
        slots.append(runner.submit(hosts[i]))
        if len(slots) > 1:
            outs.append(tuple(t.clone() for t in runner.fetch(slots.pop(0))))
    outs.append(tuple(t.clone() for t in runner.fetch(slots.pop(0))))
    for i, (uvd, xyz) in zip(order, outs):
        assert torch.equal(uvd, ref[i][0].cpu()) and torch.equal(xyz, ref[i][1].cpu()), i


def test_opcheck_frame_ops(gc):
    from torch.library import opcheck
    K = torch.ops.kpf
    tests = ("test_schema", "test_faketensor")
    rgb, depth, bbox, fi = syn_frames(gc)
    fi = torch.tensor(fi, dtype=torch.int32, device=DEV)
    cube = torch.full((bbox.shape[0], 3), 250.0, device=DEV)
    cam64 = torch.tensor(gc["syn_cam"], device=DEV).expand(bbox.shape[0], 4).contiguous()
    for index in (fi, None):
        d, r = (depth, rgb) if index is not None else (depth[fi.long()].contiguous(), rgb[fi.long()].contiguous())
        opcheck(K.center_from_bbox, (d, bbox, 1500, 171, index), test_utils=tests)
        c = K.center_from_bbox(d, bbox, 1500, 171, index)
        opcheck(K.crop_depth, (d, c, cube, cam64, 128, index), test_utils=tests)
        opcheck(K.crop_rgb, (r, c, cube, cam64, 128, index), test_utils=tests)
    _, _, com3d = K.crop_depth(depth, c, cube, cam64, 128, fi)
    joints = torch.zeros(bbox.shape[0], 21, 3, device=DEV)
    opcheck(K.joints_to_frame, (joints, com3d, cube, cam64.float(), 1.0), test_utils=tests)
