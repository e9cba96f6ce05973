"""CPU: the frame front end's host layer -- custom-op registration and fake shapes, frame_index checks made before any launch, and
the frame-space restatement (tests/frames_oracle.py) against the oracle's xyz_nl2uvdnl."""
import os
import sys

import numpy as np
import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

from keypointfusion_b200 import custom_ops, ops
from oracle import kpf_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)
import frames_oracle as FO  # noqa: E402

FRONT_END = ("center_from_bbox", "crop_depth", "crop_rgb", "joints_to_frame")


def test_frame_ops_are_registered_with_optional_frame_index():
    assert set(FRONT_END) <= set(custom_ops.REGISTERED)
    for n in FRONT_END[:3]:
        assert "Tensor? frame_index=None" in str(getattr(torch.ops.kpf, n).default._schema)


def test_frame_ops_shape_propagate_under_fake_tensors():
    K = torch.ops.kpf
    with FakeTensorMode(allow_non_fake_inputs=True):
        F, B, dev = 3, 5, "cuda"
        depth = torch.empty(F, 480, 640, device=dev, dtype=torch.uint16)
        rgb = torch.empty(F, 480, 640, 3, device=dev, dtype=torch.uint8)
        bbox = torch.empty(B, 4, device=dev, dtype=torch.float64)
        fi = torch.empty(B, device=dev, dtype=torch.int32)
        cube = torch.empty(B, 3, device=dev)
        cam64 = torch.empty(B, 4, device=dev, dtype=torch.float64)
        c = K.center_from_bbox(depth, bbox, 1500, 171, fi)
        img, M, com3d = K.crop_depth(depth, c, cube, cam64, 96, fi)
        r = K.crop_rgb(rgb, c, cube, cam64, 96, fi)
        uvd, xyz = K.joints_to_frame(torch.empty(B, 21, 3, device=dev), com3d, cube, torch.empty(B, 4, device=dev), 1.0)
    assert (tuple(c.shape), c.dtype) == ((B, 3), torch.float64)
    assert [tuple(t.shape) for t in (img, M, com3d, r)] == [(B, 1, 96, 96), (B, 3, 3), (B, 3), (B, 3, 96, 96)]
    assert [tuple(t.shape) for t in (uvd, xyz)] == [(B, 21, 3)] * 2
    assert all(t.dtype == torch.float32 and t.device.type == "cuda" for t in (img, M, com3d, r, uvd, xyz))


@pytest.mark.parametrize("fn", ["center", "depth", "rgb"])
@pytest.mark.parametrize("bad", [[0, 2, 1], [-1, 0, 1], np.array([0, 1]), torch.tensor([0.0, 1.0, 1.0]), None])
def test_host_frame_index_rejected_without_a_gpu(fn, bad):
    """Two frames, three boxes: each index set is refused on the host (ValueError) before the CUDA check or any launch --
    out of range, negative, wrong length, not integers, or None (which needs F == B)."""
    F, B = 2, 3
    depth = torch.zeros(F, 8, 8, dtype=torch.uint16)
    rgb = torch.zeros(F, 8, 8, 3, dtype=torch.uint8)
    center, cube, cam = torch.zeros(B, 3, dtype=torch.float64), [250, 250, 250], (617.0, 617.0, 4.0, 4.0)
    n0 = ops.launch_count()
    with pytest.raises(ValueError):
        if fn == "center":
            ops.center_from_bbox(depth, torch.zeros(B, 4, dtype=torch.float64), frame_index=bad)
        elif fn == "depth":
            ops.crop_depth(depth, center, cube, cam, frame_index=bad)
        else:
            ops.crop_rgb(rgb, center, cube, cam, frame_index=bad)
    assert ops.launch_count() == n0


def test_valid_host_frame_index_still_needs_cuda():
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.center_from_bbox(torch.zeros(2, 8, 8, dtype=torch.uint16), torch.zeros(3, 4, dtype=torch.float64), frame_index=[1, 0, 1])


def test_frame_restatement_composes_to_xyz_nl2uvdnl():
    rs = np.random.RandomState(7)
    B, P = 4, 21
    xyz = rs.uniform(-1, 1, (B, P, 3)).astype(np.float32)
    center = np.stack([rs.uniform(-80, 80, B), rs.uniform(-60, 60, B), rs.uniform(400, 900, B)], -1).astype(np.float32)
    cube = np.full((B, 3), 250, np.float32)
    cam = np.tile(np.array([617.0, 617.0, 312.0, 241.0], np.float32), (B, 1))
    M = np.zeros((B, 3, 3), np.float32)
    M[:, 0, 0] = M[:, 1, 1] = rs.uniform(0.5, 1.5, B)
    M[:, 0, 2], M[:, 1, 2], M[:, 2, 2] = rs.uniform(-300, 0, B), rs.uniform(-200, 0, B), 1
    for flip in (1.0, -1.0):
        uvd, xyz_cam = FO.joints_to_frame(xyz, center, cube, cam, flip)
        assert np.array_equal(FO.crop_from_frame(uvd, center, M, cube, 128), O.xyz_nl2uvdnl(xyz, center, M, cube, cam, 128, flip))
        assert np.array_equal(xyz_cam, xyz * cube[:, None] / np.float32(2) + center[:, None])
        assert np.array_equal(uvd[..., 2], xyz_cam[..., 2])
