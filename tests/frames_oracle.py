"""CPU restatement of the frame-space half of the a5 transform (test infrastructure, like oracle/kpf_oracle.py).

joints_to_frame is xyz_nl2uvdnl (oracle/kpf_oracle.py, loader.py:821-834) stopped after points3DToImg (loader.py:277-288), in the
same fp32 operations and order; crop_from_frame is the rest of xyz_nl2uvdnl.  tests/test_frames_cpu.py checks that the two
composed are bit-identical to the oracle's xyz_nl2uvdnl."""
import numpy as np

f32 = np.float32


def joints_to_frame(xyz, center, cube, cam, flip=1.0):
    """[B,P,3] normalised xyz -> (uvd_frame [B,P,3]: frame pixels u, v and depth mm, xyz_cam [B,P,3]: camera mm)."""
    xyz = np.asarray(xyz, f32)
    B = xyz.shape[0]
    center = np.asarray(center, f32).reshape(B, 1, 3)
    cube = np.asarray(cube, f32).reshape(B, 1, 3)
    cam = np.asarray(cam, f32).reshape(B, 1, 4)
    p = xyz * cube / f32(2.0) + center
    pu = p[..., 0] * cam[..., 0] / (p[..., 2] + f32(1e-8)) + cam[..., 2]
    pv = f32(flip) * p[..., 1] * cam[..., 1] / p[..., 2] + cam[..., 3]
    return np.stack([pu, pv, p[..., 2]], -1).astype(f32), p.astype(f32)


def crop_from_frame(uvd_frame, center, M, cube, img_size):
    """The second half of xyz_nl2uvdnl: frame pixels through M into the crop, normalised to [-1, 1]."""
    uvd_frame = np.asarray(uvd_frame, f32)
    B = uvd_frame.shape[0]
    center = np.asarray(center, f32).reshape(B, 1, 3)
    cube = np.asarray(cube, f32).reshape(B, 1, 3)
    m = np.asarray(M, f32).reshape(B, 1, 9)
    pu, pv, z = uvd_frame[..., 0], uvd_frame[..., 1], uvd_frame[..., 2]
    tu = (m[..., 0] * pu + m[..., 1] * pv) + m[..., 2]
    tv = (m[..., 3] * pu + m[..., 4] * pv) + m[..., 5]
    uu = tu / f32(img_size) * f32(2.0) - f32(1)
    vv = tv / f32(img_size) * f32(2.0) - f32(1)
    dd = (z - center[..., 2]) / (cube[..., 2] / f32(2))
    return np.stack([uu, vv, dd], -1).astype(f32)
