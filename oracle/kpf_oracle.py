"""CPU ORACLE for the KeypointFusion hot path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / `--impl reference` legs may import this
module, and only as the checker / the timed CPU baseline.  Nothing under keypointfusion_b200/ imports it.

It is a restatement (numpy for integer / index / geometry work with a fixed operation order, torch-CPU fp32
for the dense float work) of the reference's algorithm for the path named in BASELINE.json.  Every function
cites the reference file:line it follows (paths relative to /root/reference).

Pinning status (tests/test_oracle_golden.py, fixtures in tests/golden/ made by tests/golden/make_golden.py by
running the UNMODIFIED reference in the build container):
  * a1-a2, a4-a8, a10-a16 (SURVEY.md 8a): pinned against reference outputs.
  * a3 (resample): the reference uses np.random.choice (loader.py:1179-1185), irreproducible on a GPU; the
    oracle DEFINES a counter-based permutation (feistel) with the same multiset semantics.  Selection given
    explicit ranks is pinned; the RNG itself is "parity unpinned" by construction.
  * DESA's ball query follows pointnet2_ops 3.0.0 (not vendored): "parity unpinned" (SURVEY.md 8c).
  * BertLayer follows transformers 4.25.1 modeling_bert; pinned against the installed transformers 5.5
    BertEncoder through the reference's own KP_Interaction_TR.

Where the reference's arithmetic order is implementation-defined (BLAS matmul, LAPACK inverse, topk ties),
the oracle fixes one: fp64 adjugate inverse rounded to fp32, left-to-right fp32 sums without FMA, ties
broken by lower index.  The CUDA kernels follow the same order so index outputs are bit-exact.
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

f32 = np.float32
f64 = np.float64


# ----------------------------------------------------------------------------------------------
# small helpers
# ----------------------------------------------------------------------------------------------
def inv3x3_f64(M):
    """Closed-form adjugate inverse in fp64 of [...,3,3] (replaces np.linalg.inv loader.py:882 and
    torch.linalg.inv loader.py:781).  Operation order is part of the contract with the CUDA kernels."""
    M = np.asarray(M, f64)
    a, b, c = M[..., 0, 0], M[..., 0, 1], M[..., 0, 2]
    d, e, f = M[..., 1, 0], M[..., 1, 1], M[..., 1, 2]
    g, h, i = M[..., 2, 0], M[..., 2, 1], M[..., 2, 2]
    A = e * i - f * h
    Bc = f * g - d * i
    C = d * h - e * g
    det = (a * A + b * Bc) + c * C
    out = np.empty(M.shape, f64)
    out[..., 0, 0] = A / det
    out[..., 0, 1] = (c * h - b * i) / det
    out[..., 0, 2] = (b * f - c * e) / det
    out[..., 1, 0] = Bc / det
    out[..., 1, 1] = (a * i - c * g) / det
    out[..., 1, 2] = (c * d - a * f) / det
    out[..., 2, 0] = C / det
    out[..., 2, 1] = (b * g - a * h) / det
    out[..., 2, 2] = (a * e - b * d) / det
    return out


def nearest_down(img, fs):
    """F.interpolate(img, [fs, fs]) default mode='nearest' (model.py:409,:471): src = floor(dst*S/fs)."""
    S = img.shape[-1]
    if S == fs:
        return img
    idx = np.floor(np.arange(fs, dtype=f32) * f32(S / fs)).astype(np.int64)
    idx = np.minimum(idx, S - 1)
    if isinstance(img, torch.Tensor):
        ti = torch.from_numpy(idx)
        return img[..., ti, :][..., :, ti]
    return img[..., idx, :][..., :, idx]


def cell_coords(fs):
    """2(i+.5)/fs-1 in fp32 (model.py:477-481).  Returns (u[fs*fs], v[fs*fs]) flat row-major: u=col, v=row."""
    t = (((np.arange(fs, dtype=f32) + f32(0.5)) * f32(2.0)) / f32(fs)) - f32(1.0)
    u = np.tile(t, fs)
    v = np.repeat(t, fs)
    return u.astype(f32), v.astype(f32)


# ----------------------------------------------------------------------------------------------
# a1-a3  back-projection  (dataloader/loader.py:843-893, :1173-1186; API util/img2pcl.py:11-40)
# ----------------------------------------------------------------------------------------------
BG_BAND = 1e-8 + 1e-5 * 1.0  # np.isclose(x, 1): atol + rtol*|1|   (loader.py:844)
ZERO_BAND = 1e-8             # np.isclose(d, 0): atol               (loader.py:880)


def valid_mask(imgD, com3D, cube):
    """[S,S] fp32 -> (valid bool [S,S], dpt fp32 [S,S]).  loader.py:844-847 then :880."""
    imgD = np.asarray(imgD, f32)
    bg = np.abs(imgD.astype(f64) - 1.0) <= BG_BAND
    dpt = (imgD * f32(f32(cube[2]) / f32(2.0)) + f32(com3D[2])).astype(f32)
    dpt = np.where(bg, f32(0), dpt)
    valid = np.abs(dpt.astype(f64)) > ZERO_BAND
    return valid, dpt


def getpcl(imgD, com3D, cube, M, cam, flip=1.0):
    """One sample.  Returns (pcl [P,3] f64 normalised, pix [P] int32 flat row-major pixel index).
    loader.py:843-853 (getpcl) + :874-893 (depthToPCL)."""
    S = imgD.shape[-1]
    valid, dpt = valid_mask(imgD, com3D, cube)
    pix = np.flatnonzero(valid.reshape(-1)).astype(np.int32)  # np.where row-major (y, x)   :880
    r = (pix // S).astype(f64)
    c = (pix % S).astype(f64)
    Mi = inv3x3_f64(M)
    u = c + 0.5
    v = r + 0.5
    qx = (Mi[0, 0] * u + Mi[0, 1] * v) + Mi[0, 2]
    qy = (Mi[1, 0] * u + Mi[1, 1] * v) + Mi[1, 2]
    qz = (Mi[2, 0] * u + Mi[2, 1] * v) + Mi[2, 2]
    qx = qx / qz
    qy = qy / qz
    depth = dpt.reshape(-1)[pix].astype(f64)
    fx, fy, fu, fv = [f64(t) for t in cam]
    x = (qx - fu) / fx * depth
    y = f64(flip) * (qy - fv) / fy * depth
    z = depth
    com = np.asarray(com3D, f64)
    half = np.asarray(cube, f64) / 2.0
    pcl = np.stack([(x - com[0]) / half[0], (y - com[1]) / half[1], (z - com[2]) / half[2]], 1)
    return pcl, pix


def _mix32(x):
    x = np.uint64(x) & np.uint64(0xFFFFFFFF)
    x ^= x >> np.uint64(16)
    x = (x * np.uint64(0x85EBCA6B)) & np.uint64(0xFFFFFFFF)
    x ^= x >> np.uint64(13)
    x = (x * np.uint64(0xC2B2AE35)) & np.uint64(0xFFFFFFFF)
    x ^= x >> np.uint64(16)
    return int(x)


def feistel_perm(i, n, key):
    """Bijection on [0,n): 4-round balanced Feistel on the next even-bit power of two, cycle-walking."""
    bits = max(2, (n - 1).bit_length())
    bits += bits & 1
    half = bits // 2
    mask = (1 << half) - 1
    x = i
    while True:
        l, r = x >> half, x & mask
        for rnd in range(4):
            l, r = r, l ^ (_mix32(r ^ key ^ ((rnd * 0x9E3779B9) & 0xFFFFFFFF)) & mask)
        x = (l << half) | r
        if x < n:
            return x


def sample_key(seed, b):
    return _mix32((seed & 0xFFFFFFFF) ^ _mix32((b + 0x85EBCA6B) & 0xFFFFFFFF))


def _mix32_v(x):
    x = x.astype(np.uint64) & np.uint64(0xFFFFFFFF)
    x ^= x >> np.uint64(16)
    x = (x * np.uint64(0x85EBCA6B)) & np.uint64(0xFFFFFFFF)
    x ^= x >> np.uint64(13)
    x = (x * np.uint64(0xC2B2AE35)) & np.uint64(0xFFFFFFFF)
    x ^= x >> np.uint64(16)
    return x


def feistel_perm_v(i, n, key):
    """Vectorised feistel_perm over an index array (same integer arithmetic)."""
    bits = max(2, (n - 1).bit_length())
    bits += bits & 1
    half = np.uint64(bits // 2)
    mask = np.uint64((1 << (bits // 2)) - 1)
    x = np.asarray(i, np.uint64).copy()
    todo = np.ones(x.shape, bool)
    while todo.any():
        l, r = x[todo] >> half, x[todo] & mask
        for rnd in range(4):
            l, r = r, l ^ (_mix32_v(r ^ np.uint64(key) ^ np.uint64((rnd * 0x9E3779B9) & 0xFFFFFFFF)) & mask)
        x[todo] = (l << half) | r
        todo &= x >= n
    return x.astype(np.int64)


def resample_ranks(P, sample_num, seed, b):
    """Deterministic stand-in for loader.py:1176-1185: a random `sample_num`-subset (P>=sample_num) or the
    multiset {each index floor(sample_num/P) times + distinct random remainder} (P<sample_num), in random order."""
    if P == 0:
        return np.zeros(sample_num, np.int32)
    key = sample_key(seed, b)
    j = np.arange(sample_num)
    if P >= sample_num:
        return feistel_perm_v(j, P, key).astype(np.int32)
    tmp = sample_num // P
    t = feistel_perm_v(j, sample_num, key ^ 0x1234567)
    out = t // tmp
    rem = t >= tmp * P
    if rem.any():
        out[rem] = feistel_perm_v(t[rem] - tmp * P, P, key)
    return out.astype(np.int32)


def getpcl_sample(imgD, com3D, cube, M, cam, sample_num=1024, ranks=None, seed=0, b=0, clamp=False, flip=1.0):
    """a1+a2+a3 for one sample -> ([sample_num,3] f32, P).  `ranks` (into the ordered valid list) overrides the
    built-in permutation; P==0 -> zeros (loader.py:1176-1177); clamp: loader.py:1399 / demo_RGBD.py:332."""
    pcl, pix = getpcl(imgD, com3D, cube, M, cam, flip)
    P = pcl.shape[0]
    if P == 0:
        return np.zeros((sample_num, 3), f32), 0
    if ranks is None:
        ranks = resample_ranks(P, sample_num, seed, b)
    ranks = np.minimum(np.asarray(ranks, np.int64), P - 1)
    out = pcl[ranks].astype(f32)
    if clamp:
        out = np.clip(out, -1, 1)
    return out, P


# ----------------------------------------------------------------------------------------------
# a5  uvd <-> xyz normalised transforms (dataloader/loader.py:775-789, :821-841, :265-288)
# ----------------------------------------------------------------------------------------------
def uvd_nl2xyznl(uvd, center, M, cube, cam, img_size, flip=1.0):
    """[B,P,3] fp32 -> [B,P,3] fp32; fixed-order fp32 arithmetic, M^-1 = fl32(fp64 adjugate)."""
    uvd = np.asarray(uvd, f32)
    B = uvd.shape[0]
    Mi = inv3x3_f64(np.asarray(M, f64)).astype(f32)
    center = np.asarray(center, f32).reshape(B, 1, 3)
    cube = np.asarray(cube, f32).reshape(B, 1, 3)
    cam = np.asarray(cam, f32).reshape(B, 1, 4)
    hs = f32(img_size / 2)
    u = (uvd[..., 0] + f32(1)) * hs
    v = (uvd[..., 1] + f32(1)) * hs
    d = uvd[..., 2] * (cube[..., 2] / f32(2.0)) + center[..., 2]
    m = Mi.reshape(B, 1, 9)
    xw = (m[..., 0] * u + m[..., 1] * v) + m[..., 2]
    yw = (m[..., 3] * u + m[..., 4] * v) + m[..., 5]
    X = (xw - cam[..., 2]) * d / cam[..., 0]
    Y = f32(flip) * (yw - cam[..., 3]) * d / cam[..., 1]
    out = np.stack([X, Y, d], -1).astype(f32)
    return ((out - center) / (cube / f32(2.0))).astype(f32)


def xyz_nl2uvdnl(xyz, center, M, cube, cam, img_size, flip=1.0):
    """Inverse of the above (loader.py:821-834; note +1e-8 only on the X divide, :282 vs :285)."""
    xyz = np.asarray(xyz, f32)
    B = xyz.shape[0]
    center = np.asarray(center, f32).reshape(B, 1, 3)
    cube = np.asarray(cube, f32).reshape(B, 1, 3)
    cam = np.asarray(cam, f32).reshape(B, 1, 4)
    m = np.asarray(M, f32).reshape(B, 1, 9)
    p = xyz * cube / f32(2.0) + center
    pu = p[..., 0] * cam[..., 0] / (p[..., 2] + f32(1e-8)) + cam[..., 2]
    pv = f32(flip) * p[..., 1] * cam[..., 1] / p[..., 2] + cam[..., 3]
    tu = (m[..., 0] * pu + m[..., 1] * pv) + m[..., 2]
    tv = (m[..., 3] * pu + m[..., 4] * pv) + m[..., 5]
    uu = tu / f32(img_size) * f32(2.0) - f32(1)
    vv = tv / f32(img_size) * f32(2.0) - f32(1)
    dd = (p[..., 2] - center[..., 2]) / (cube[..., 2] / f32(2))
    return np.stack([uu, vv, dd], -1).astype(f32)


def cell_xyz(img_down, center, M, cube, cam, img_size, flip=1.0):
    """All H*W cells of the down-sampled depth map -> normalised xyz [B,HW,3] (loader.py:948-953)."""
    img_down = np.asarray(img_down, f32)
    B, _, H, W = img_down.shape
    u, v = cell_coords(W)
    uvd = np.stack([np.broadcast_to(u, (B, H * W)), np.broadcast_to(v, (B, H * W)),
                    img_down.reshape(B, H * W)], -1)
    return uvd_nl2xyznl(uvd, center, M, cube, cam, img_size, flip)


# ----------------------------------------------------------------------------------------------
# a6  nearest-cell indices + weights (dataloader/loader.py:936-967)
# ----------------------------------------------------------------------------------------------
def img2pcl_index(pcl, img_down, center, M, cube, cam, img_size, select_num=4, flip=1.0):
    """-> closeness [B,N,K] f32, index [B,N,K] int64 (flat row*W+col), distances [B,N,K] f32.
    Squared distances: ((dx*dx + dy*dy) + dz*dz) in fp32; ties broken by lower cell index."""
    pcl = np.asarray(pcl, f32)
    cells = cell_xyz(img_down, center, M, cube, cam, img_size, flip)  # B HW 3
    B, N, _ = pcl.shape
    idx = np.empty((B, N, select_num), np.int64)
    val = np.empty((B, N, select_num), f32)
    HW = cells.shape[1]
    kc = min(HW, select_num + 8)  # candidates: exact unless > 8 cells tie at the K-th distance (then full stable sort)
    for b in range(B):
        d = pcl[b][:, None, :] - cells[b][None, :, :]
        d2 = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
        cv, ci = torch.topk(torch.from_numpy(d2), kc, dim=1, largest=False, sorted=True)
        cv, ci = cv.numpy(), ci.numpy()
        order = np.lexsort((ci, cv), axis=1)  # (distance, then lower index)
        ci = np.take_along_axis(ci, order, 1)
        cv = np.take_along_axis(cv, order, 1)
        amb = np.flatnonzero(cv[:, select_num - 1] == cv[:, kc - 1]) if kc < HW else []
        for n in amb:
            o = np.argsort(d2[n], kind="stable")[:kc]
            ci[n], cv[n] = o, d2[n][o]
        idx[b] = ci[:, :select_num]
        val[b] = cv[:, :select_num]
    c = f32(1) / (val + f32(1e-8))
    s = c[..., 0]
    for k in range(1, select_num):
        s = s + c[..., k]
    close = c / (s[..., None] + f32(1e-8))
    return close.astype(f32), idx, val


# ----------------------------------------------------------------------------------------------
# a4  offset2joint_weight (model/model.py:466-500 == util/generateFeature.py:166-195)
# ----------------------------------------------------------------------------------------------
def _kernel_vec(kernel_size, J):
    if torch.is_tensor(kernel_size):
        return kernel_size.float().view(1, J, 1)
    return torch.full((1, J, 1), float(kernel_size))


def offset2joint_weight(offset, depth, kernel_size):
    offset = offset.float()
    B, C5, fs, _ = offset.shape
    J = C5 // 5
    d = nearest_down(depth.float(), fs).reshape(B, 1, fs * fs)
    u, v = cell_coords(fs)
    coords = torch.cat([torch.from_numpy(u).view(1, 1, -1).expand(B, 1, -1),
                        torch.from_numpy(v).view(1, 1, -1).expand(B, 1, -1), d], 1)  # B 3 HW
    unit = offset[:, :3 * J].reshape(B, J, 3, -1)
    heat = offset[:, 3 * J:4 * J].reshape(B, J, -1)
    wgt = offset[:, 4 * J:].reshape(B, J, -1)
    m = (d < 0.99).float()
    w = torch.softmax(wgt.masked_fill((d > 0.99).expand(B, J, -1), -1e8), -1)
    k = _kernel_vec(kernel_size, J)
    dist = k - (heat * m) * k
    return (((unit * m.unsqueeze(1)) * dist.unsqueeze(2) + coords.unsqueeze(1)) * w.unsqueeze(2)).sum(-1)


# ----------------------------------------------------------------------------------------------
# a7  pcl_joint2offset (model/model.py:503-525 == generateFeature.py:465-488)
# ----------------------------------------------------------------------------------------------
def pcl_joint2offset(joint, pcl, kernel_size):
    B, J, _ = joint.shape
    off = joint.unsqueeze(2) - pcl.unsqueeze(1)  # B J N 3
    dis = off.pow(2).sum(-1).sqrt()
    unit = off / (dis.unsqueeze(-1) + 1e-8)
    k = _kernel_vec(kernel_size, J)
    heat = (k - dis) / k
    m = (heat >= 0).float() * (pcl[:, :, 2] < 0.99).float().unsqueeze(1)
    unit = (unit * m.unsqueeze(-1)).permute(0, 2, 1, 3).reshape(B, -1, 3 * J)  # B N (J,3) joint-major
    return torch.cat([unit, (heat * m).permute(0, 2, 1)], -1)


# ----------------------------------------------------------------------------------------------
# a8  K-tap weighted gathers (model/model.py:297-306)
# ----------------------------------------------------------------------------------------------
def gather_taps(feat, index, closeness):
    """feat [B,C,H,W] (or [B,C,HW]), index [B,N,K] int64, closeness [B,N,K] -> [B,N,C]."""
    B, C = feat.shape[:2]
    N, K = index.shape[1:]
    g = torch.gather(feat.reshape(B, C, -1).float(), 2, index.reshape(B, 1, -1).expand(B, C, -1)).view(B, C, N, K)
    return (g * closeness.unsqueeze(1)).sum(-1).permute(0, 2, 1)


# ----------------------------------------------------------------------------------------------
# a10 joint2heatmap (generateFeature.py:584-600), a11 img2anchor_dis (loader.py:791-819)
# ----------------------------------------------------------------------------------------------
def joint2heatmap(joint, std, heatmap_size, sigma=1.5):
    B, J, _ = joint.shape
    S = heatmap_size
    ar = torch.arange(S, dtype=torch.float32) + 0.5
    jx = ((joint[:, :, 0] + 1) / 2 * S).view(B, J, 1, 1)
    jy = ((joint[:, :, 1] + 1) / 2 * S).view(B, J, 1, 1)
    mx = ar.view(1, 1, 1, S)  # x varies along columns (np.meshgrid xx)
    my = ar.view(1, 1, S, 1)
    return torch.exp(-(((mx - jx) / std) ** 2 + ((my - jy) / std) ** 2) / (2 * sigma ** 2))


def img2anchor_dis(joint_uvd, img_down, center, M, cube, cam, img_size, gamma=10, flip=1.0):
    B, J, _ = joint_uvd.shape
    H, W = img_down.shape[-2:]
    jx = torch.from_numpy(uvd_nl2xyznl(joint_uvd.numpy(), center, M, cube, cam, img_size, flip))
    cx = torch.from_numpy(cell_xyz(img_down.numpy(), center, M, cube, cam, img_size, flip))
    d2 = (cx.unsqueeze(1) - jx.unsqueeze(2)).pow(2).sum(-1)
    return (1 / (gamma * d2 + 1)).view(B, J, H, W)


# ----------------------------------------------------------------------------------------------
# a16 joint2offset dense target (generateFeature.py:59-84; model.py:440-463 has no +1e-8)
# ----------------------------------------------------------------------------------------------
def joint2offset(joint, img, kernel_size, feature_size, eps=1e-8):
    B = img.shape[0]
    fs = feature_size
    joint = joint.reshape(B, -1, 3)
    J = joint.shape[1]
    d = nearest_down(img.float(), fs).reshape(B, 1, fs * fs)
    u, v = cell_coords(fs)
    coords = torch.cat([torch.from_numpy(u).view(1, 1, -1).expand(B, 1, -1),
                        torch.from_numpy(v).view(1, 1, -1).expand(B, 1, -1), d], 1)  # B 3 HW
    off = joint.unsqueeze(-1) - coords.unsqueeze(1)  # B J 3 HW
    dist = (off.pow(2).sum(2) + eps).sqrt()
    unit = off / dist.unsqueeze(2)
    k = _kernel_vec(kernel_size, J)
    heat = (k - dist) / k
    m = (heat >= 0).float() * (d < 0.99).float()
    return torch.cat([(unit * m.unsqueeze(2)).reshape(B, 3 * J, fs, fs), (heat * m).reshape(B, J, fs, fs)], 1)


# ----------------------------------------------------------------------------------------------
# a14/a15 feature-level fusion modules (model/fusion_layer.py)
# ----------------------------------------------------------------------------------------------
def rgbd_fusion(p, rgb, depth):
    """RGBDFusion.forward fusion_layer.py:56-83.  p: state_dict of the module."""
    cat = torch.cat([rgb, depth], 1)
    l = F.conv2d(cat, p["gate_rgb.weight"], p["gate_rgb.bias"])
    r = F.conv2d(cat, p["gate_depth.weight"], p["gate_depth.bias"])
    a = torch.softmax(torch.cat([l, r], 1), 1)
    merge = rgb * a[:, 0:1] + depth * a[:, 1:2]
    return [torch.relu((rgb + merge) / 2), torch.relu((depth + merge) / 2)], merge


def ac_fusion(p, rgb, depth):
    """ACFusion.forward fusion_layer.py:101-116."""
    wr = torch.sigmoid(F.conv2d(rgb.mean((2, 3), keepdim=True), p["cam_rgb.weight"], p["cam_rgb.bias"]))
    wd = torch.sigmoid(F.conv2d(depth.mean((2, 3), keepdim=True), p["cam_depth.weight"], p["cam_depth.bias"]))
    merge = wr * rgb + wd * depth
    return [torch.relu((rgb + merge) / 2), torch.relu((depth + merge) / 2)], merge


def filter_layer(p, x, prefix=""):
    """FilterLayer.forward fusion_layer.py:18-22."""
    y = x.mean((2, 3))
    y = torch.relu(F.linear(y, p[prefix + "fc.0.weight"], p[prefix + "fc.0.bias"]))
    y = torch.sigmoid(F.linear(y, p[prefix + "fc.2.weight"], p[prefix + "fc.2.bias"]))
    return y.view(y.shape[0], -1, 1, 1)


def fsp(p, guide, main, prefix=""):
    """FSP.forward fusion_layer.py:33-37."""
    return main + filter_layer(p, torch.cat([guide, main], 1), prefix + "filter.") * guide


# ----------------------------------------------------------------------------------------------
# a13 cross-attention decoder layer (model/transfusion_head.py:684-708, :132-173, :303-556)
# ----------------------------------------------------------------------------------------------
def cross_decoder_layer(p, prefix, anchor_feats, img_feats, num_heads=4):
    """One TransformerDecoderLayer(cross_only=True) -> [B,C,J].  query=anchor_feats (RGB joint feats),
    key=value=img_feats + cross_posembed (transfusion_head.py:161-163); q scaled after bias (:403,:468)."""
    B, J, C = anchor_feats.shape
    hd = C // num_heads
    q_in = anchor_feats + p[prefix + "self_posembed.weight"][:J].unsqueeze(0)
    k_in = img_feats + p[prefix + "cross_posembed.weight"][:J].unsqueeze(0)
    Wi, bi = p[prefix + "multihead_attn.in_proj_weight"], p[prefix + "multihead_attn.in_proj_bias"]
    q = F.linear(q_in, Wi[:C], bi[:C]) * (float(hd) ** -0.5)
    kv = F.linear(k_in, Wi[C:], bi[C:])
    k, v = kv[..., :C], kv[..., C:]
    q = q.view(B, J, num_heads, hd).transpose(1, 2)
    k = k.view(B, J, num_heads, hd).transpose(1, 2)
    v = v.view(B, J, num_heads, hd).transpose(1, 2)
    a = torch.softmax(q @ k.transpose(-1, -2), -1)
    o = (a @ v).transpose(1, 2).reshape(B, J, C)
    o = F.linear(o, p[prefix + "multihead_attn.out_proj.weight"], p[prefix + "multihead_attn.out_proj.bias"])
    x = F.layer_norm(anchor_feats + o, (C,), p[prefix + "norm2.weight"], p[prefix + "norm2.bias"], 1e-5)
    y = F.linear(torch.relu(F.linear(x, p[prefix + "linear1.weight"], p[prefix + "linear1.bias"])),
                 p[prefix + "linear2.weight"], p[prefix + "linear2.bias"])
    x = F.layer_norm(x + y, (C,), p[prefix + "norm3.weight"], p[prefix + "norm3.bias"], 1e-5)
    return x.permute(0, 2, 1)


def updated_decoder(p, prefix, anchor_feats, img_feats, num_layers=4, num_heads=4):
    """updatedDecoder.forward: every layer gets the SAME inputs and only the last output is returned
    (transfusion_head.py:705-708), so only layer num_layers-1 is live."""
    return cross_decoder_layer(p, f"{prefix}decoder.{num_layers - 1}.", anchor_feats, img_feats, num_heads)


# ----------------------------------------------------------------------------------------------
# 8b exports off the live path: general-shape attention (model/transfusion_head.py:16-91, :94-173, :303-556, :560-632, :711-783)
# pinned against tests/golden/golden_heads.npz (made by tests/golden/make_golden_heads.py from the unmodified reference)
# ----------------------------------------------------------------------------------------------
def mha_forward(p, prefix, query, key, value, num_heads, key_padding_mask=None, attn_mask=None):
    """multi_head_attention_forward, general branch (transfusion_head.py:303-556): query [L,N,E], key / value [S,N,E] ->
    (out [L,N,E], head-averaged weights [N,L,S])."""
    L, N, E = query.shape
    S = key.shape[0]
    hd = E // num_heads
    W, b = p[prefix + "in_proj_weight"], p[prefix + "in_proj_bias"]
    q = F.linear(query, W[:E], b[:E]) * (float(hd) ** -0.5)                    # :403, :468
    k = F.linear(key, W[E:2 * E], b[E:2 * E])
    v = F.linear(value, W[2 * E:], b[2 * E:])
    q = q.contiguous().view(L, N * num_heads, hd).transpose(0, 1)              # :497-501
    k = k.contiguous().view(S, N * num_heads, hd).transpose(0, 1)
    v = v.contiguous().view(S, N * num_heads, hd).transpose(0, 1)
    w = torch.bmm(q, k.transpose(1, 2))                                        # :524
    if attn_mask is not None:
        w = w + attn_mask.unsqueeze(0)                                         # :527-529
    if key_padding_mask is not None:                                           # :531-537
        w = w.view(N, num_heads, L, S).masked_fill(key_padding_mask.unsqueeze(1).unsqueeze(2), float("-inf")).view(N * num_heads, L, S)
    w = torch.softmax(w, dim=-1)
    o = torch.bmm(w, v).transpose(0, 1).contiguous().view(L, N, E)             # :543-545
    o = F.linear(o, p[prefix + "out_proj.weight"], p[prefix + "out_proj.bias"])
    return o, w.view(N, num_heads, L, S).sum(dim=1) / num_heads               # :551-554


def decoder_layer(p, prefix, query, key, query_pos, key_pos, num_heads=4, cross_only=True, attn_mask=None):
    """TransformerDecoderLayer.forward (transfusion_head.py:132-173) with the position embeddings given as tensors
    (query_pos [B or 1,Pq,C], key_pos [B or 1,Pk,C]; None = no embedding) -> [B,C,Pq]."""
    C = query.shape[-1]
    qp = 0 if query_pos is None else query_pos
    kp = 0 if key_pos is None else key_pos
    x = query.permute(1, 0, 2)                                                 # :154-155  [P,B,C]
    if not cross_only:                                                         # :157-161
        qq = (query + qp).permute(1, 0, 2)
        x = F.layer_norm(x + mha_forward(p, prefix + "self_attn.", qq, qq, qq, num_heads)[0], (C,), p[prefix + "norm1.weight"],
                         p[prefix + "norm1.bias"], 1e-5)
    kk = (key + kp).permute(1, 0, 2)
    qq = x + (qp.permute(1, 0, 2) if torch.is_tensor(qp) else 0)
    a = mha_forward(p, prefix + "multihead_attn.", qq, kk, kk, num_heads, attn_mask=attn_mask)[0]   # :163-165
    x = F.layer_norm(x + a, (C,), p[prefix + "norm2.weight"], p[prefix + "norm2.bias"], 1e-5)
    y = F.linear(torch.relu(F.linear(x, p[prefix + "linear1.weight"], p[prefix + "linear1.bias"])),
                 p[prefix + "linear2.weight"], p[prefix + "linear2.bias"])                          # :167-169
    x = F.layer_norm(x + y, (C,), p[prefix + "norm3.weight"], p[prefix + "norm3.bias"], 1e-5)
    return x.permute(1, 2, 0)                                                  # :172


def sine_position_embedding(mask, embedding_dim, temperature=10000, normalize=False, scale=2 * math.pi):
    """DetrSinePositionEmbedding.forward (transfusion_head.py:75-91): mask [B,H,W] -> [B, 2*embedding_dim, H, W]."""
    y_embed = mask.cumsum(1, dtype=torch.float32)
    x_embed = mask.cumsum(2, dtype=torch.float32)
    if normalize:
        y_embed = y_embed / (y_embed[:, -1:, :] + 1e-6) * scale
        x_embed = x_embed / (x_embed[:, :, -1:] + 1e-6) * scale
    dim_t = torch.arange(embedding_dim, dtype=torch.float32)
    dim_t = temperature ** (2 * torch.div(dim_t, 2, rounding_mode="floor") / embedding_dim)
    pos_x = x_embed[:, :, :, None] / dim_t
    pos_y = y_embed[:, :, :, None] / dim_t
    pos_x = torch.stack((pos_x[:, :, :, 0::2].sin(), pos_x[:, :, :, 1::2].cos()), dim=4).flatten(3)
    pos_y = torch.stack((pos_y[:, :, :, 0::2].sin(), pos_y[:, :, :, 1::2].cos()), dim=4).flatten(3)
    return torch.cat((pos_y, pos_x), dim=3).permute(0, 3, 1, 2)


def detr_decoder(p, prefix, anchor_feats, img_feats, num_layers, num_heads=4):
    """detrDecoder.forward (transfusion_head.py:605-632): joint tokens attend over the map's cells; last layer only."""
    B, C, W, H = img_feats.shape
    J = anchor_feats.shape[1]
    key_pos = sine_position_embedding(torch.ones(B, W, H), C // 2, normalize=True).flatten(2).permute(0, 2, 1)
    lp = f"{prefix}decoder.{num_layers - 1}."
    return decoder_layer(p, lp, anchor_feats, img_feats.flatten(2).permute(0, 2, 1), p[lp + "self_posembed.weight"][:J].unsqueeze(0),
                         key_pos, num_heads)


def spatial_aggregate_tr(p, prefix, img_feats, anchor_feats, num_layers, num_heads=4):
    """spatial_aggregate_TR.forward (transfusion_head.py:758-783): the map's cells attend over the joint tokens; last layer only."""
    B, C, W, H = img_feats.shape
    J = anchor_feats.shape[1]
    query_pos = sine_position_embedding(torch.ones(B, W, H), C // 2, normalize=True).flatten(2).permute(0, 2, 1)
    lp = f"{prefix}decoder.{num_layers - 1}."
    return decoder_layer(p, lp, img_feats.flatten(2).permute(0, 2, 1), anchor_feats, query_pos,
                         p[lp + "cross_posembed.weight"][:J].unsqueeze(0), num_heads)


def position_embedding_learned(p, prefix, xyz, eps=1e-5):
    """PositionEmbeddingLearned.forward (transfusion_head.py:29-32), eval-mode BatchNorm: [B,P,in] -> [B,F,P]."""
    h = F.linear(xyz, p[prefix + "0.weight"][:, :, 0], p[prefix + "0.bias"])
    h = (h - p[prefix + "1.running_mean"]) / torch.sqrt(p[prefix + "1.running_var"] + eps) * p[prefix + "1.weight"] + p[prefix + "1.bias"]
    return F.linear(torch.relu(h), p[prefix + "3.weight"][:, :, 0], p[prefix + "3.bias"]).permute(0, 2, 1)


# ----------------------------------------------------------------------------------------------
# "next" rows needed to close the block: a9 embeddings, DESA, BERT token encoders
# ----------------------------------------------------------------------------------------------
def conv_bn(p, prefix, x):
    """nn.Sequential(Conv1d(k=1), BatchNorm1d) in eval mode on [B,L,Cin] -> [B,L,Cout] (model.py:254-259)."""
    y = F.linear(x, p[prefix + "0.weight"].squeeze(-1), p[prefix + "0.bias"])
    s = p[prefix + "1.weight"] / torch.sqrt(p[prefix + "1.running_var"] + 1e-5)
    return (y - p[prefix + "1.running_mean"]) * s + p[prefix + "1.bias"]


def _bn2d(p, prefix, x):  # x [..., C]
    s = p[prefix + "weight"] / torch.sqrt(p[prefix + "running_var"] + 1e-5)
    return (x - p[prefix + "running_mean"]) * s + p[prefix + "bias"]


def ball_query(xyz, centers, radius, nsample, return_counts=False):
    """pointnet2_ops 3.0.0 ball_query: first `nsample` indices (ascending) with d2 < r*r, rest = first hit,
    zero-initialised.  d2 = ((dx*dx+dy*dy)+dz*dz) fp32, r2 = fl32(r)*fl32(r).  numpy, exact.
    return_counts: also the number of points inside each ball (before truncation to nsample), [B,J]."""
    xyz = np.asarray(xyz, f32)
    centers = np.asarray(centers, f32)
    B, N, _ = xyz.shape
    J = centers.shape[1]
    r2 = f32(radius) * f32(radius)
    idx = np.zeros((B, J, nsample), np.int32)
    counts = np.zeros((B, J), np.int64)
    for b in range(B):
        d = centers[b][:, None, :] - xyz[b][None, :, :]
        d2 = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
        for j in range(J):
            allhits = np.flatnonzero(d2[j] < r2)
            counts[b, j] = allhits.size
            hits = allhits[:nsample]
            if hits.size:
                idx[b, j, :] = hits[0]
                idx[b, j, :hits.size] = hits
    return (idx, counts) if return_counts else idx


def desa(p, prefix, pcl_feat, node_feat, pcl_xyz, node_xyz, radius=(0.1, 0.2, 0.4), nsample=(64, 64, 64)):
    """DESA.forward model.py:166-204 with the pointnet2_ops grouping restated."""
    outs = desa_scales(p, prefix, pcl_feat, node_feat, pcl_xyz, node_xyz, radius, nsample)
    outs.append(node_feat)
    cat = torch.cat(outs, -1)
    y = F.linear(cat, p[prefix + "fusion.0.weight"].squeeze(-1), p[prefix + "fusion.0.bias"])
    return torch.relu(_bn2d(p, prefix + "fusion.1.", y))


def desa_scales(p, prefix, pcl_feat, node_feat, pcl_xyz, node_xyz, radius=(0.1, 0.2, 0.4), nsample=(64, 64, 64)):
    """DESA's grouping and per-scale MLP, before the fusion conv (model.py:166-200): one max-pooled [B,J,C] tensor per radius."""
    B, J, C = node_feat.shape
    xyz = torch.cat([pcl_xyz, node_xyz], 1)
    feat = torch.cat([pcl_feat, node_feat], 1)
    outs = []
    for i, (r, ns) in enumerate(zip(radius, nsample)):
        idx = torch.from_numpy(ball_query(xyz.numpy(), node_xyz.numpy(), r, ns)).long()  # B J ns
        bi = torch.arange(B).view(B, 1, 1)
        gx = (xyz[bi, idx] - node_xyz.unsqueeze(2)) / r        # B J ns 3
        gf = feat[bi, idx] - node_feat.unsqueeze(2)            # B J ns C
        loc = _bn2d(p, f"{prefix}bn_l0_blocks.{i}.", F.linear(gx, p[f"{prefix}conv_l0_blocks.{i}.weight"].view(-1, 3),
                                                            p[f"{prefix}conv_l0_blocks.{i}.bias"]))
        ft = _bn2d(p, f"{prefix}bn_f0_blocks.{i}.", F.linear(gf, p[f"{prefix}conv_f0_blocks.{i}.weight"].view(-1, C),
                                                           p[f"{prefix}conv_f0_blocks.{i}.bias"]))
        g = torch.relu(loc + ft)
        n_extra = len([k for k in p if k.startswith(f"{prefix}conv_blocks.{i}.") and k.endswith("weight")])
        for j in range(n_extra):
            w = p[f"{prefix}conv_blocks.{i}.{j}.weight"]
            g = torch.relu(_bn2d(p, f"{prefix}bn_blocks.{i}.{j}.",
                                 F.linear(g, w.view(w.shape[0], -1), p[f"{prefix}conv_blocks.{i}.{j}.bias"])))
        outs.append(g.max(2)[0])  # B J C
    return outs


def bert_layer(p, prefix, h, num_heads=4, eps=1e-12):
    """transformers 4.25.1 BertLayer (self-attention, post-LN, erf-gelu), no mask, eval."""
    B, L, C = h.shape
    hd = C // num_heads

    def lin(name, x):
        return F.linear(x, p[prefix + name + ".weight"], p[prefix + name + ".bias"])
    q = lin("attention.self.query", h).view(B, L, num_heads, hd).transpose(1, 2)
    k = lin("attention.self.key", h).view(B, L, num_heads, hd).transpose(1, 2)
    v = lin("attention.self.value", h).view(B, L, num_heads, hd).transpose(1, 2)
    a = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(hd), -1)
    ctx = (a @ v).transpose(1, 2).reshape(B, L, C)
    x = F.layer_norm(lin("attention.output.dense", ctx) + h, (C,), p[prefix + "attention.output.LayerNorm.weight"],
                     p[prefix + "attention.output.LayerNorm.bias"], eps)
    y = lin("output.dense", F.gelu(lin("intermediate.dense", x)))
    return F.layer_norm(y + x, (C,), p[prefix + "output.LayerNorm.weight"], p[prefix + "output.LayerNorm.bias"], eps)


def kp_interaction_tr(p, prefix, x, num_layers=4, num_heads=4):
    """KP_Interaction_TR.forward model.py:116-126 (+ TR_Encoder.forward :45-103) -> (tokens, pred[B,J,3])."""
    B, L, _ = x.shape
    h = p[prefix + "bert.position_embeddings.weight"][:L].unsqueeze(0) + \
        F.linear(x, p[prefix + "bert.img_embedding.weight"], p[prefix + "bert.img_embedding.bias"])
    for i in range(num_layers):
        h = bert_layer(p, f"{prefix}bert.encoder.layer.{i}.", h, num_heads)
    pred = F.linear(h, p[prefix + "cls_head.weight"], p[prefix + "cls_head.bias"]) + \
        F.linear(x, p[prefix + "residual.weight"], p[prefix + "residual.bias"])
    return h, pred


# ----------------------------------------------------------------------------------------------
# a12 spatial attention + aggregation (model/model.py:334-344)
# ----------------------------------------------------------------------------------------------
def spatial_aggregate(p, prefix, img_feature_rgb, hm, gam, prev=None):
    """-> (spatial_weight_loss [B,J,H,W], img_feat_j [B,J,C]); literal (materialises [B,J,C,HW])."""
    B, C, H, W = img_feature_rgb.shape
    J = hm.shape[1]
    sw = torch.sigmoid(F.conv2d(torch.cat([img_feature_rgb, hm], 1), p[prefix + "atten_spatial.weight"],
                                p[prefix + "atten_spatial.bias"]))
    s = torch.sigmoid(p[prefix + "weight_dis"])
    w = s * gam + (1 - s) * sw                                                 # B J H W
    prod = torch.relu(w.unsqueeze(2) * img_feature_rgb.unsqueeze(1)).view(B, J, C, H * W)
    fj = F.linear(prod, p[prefix + "fc_spatial2joint_feature.weight"], p[prefix + "fc_spatial2joint_feature.bias"])
    fj = fj.view(B, J, C)
    if prev is not None:
        fj = torch.relu((fj + prev) / 2)
    return sw, fj


# ----------------------------------------------------------------------------------------------
# a9 + block + a17: the whole fusion path
# ----------------------------------------------------------------------------------------------
def block_kpfusion(p, prefix, img_feat, img_feature_rgb, pcl, joint_xyz, closeness, index, img_offset,
                   prev_2d_feature, img_down, center, M, cube, cam, img_size, J=21, taps=None):
    """Block_KPFusion.forward model.py:287-351.  Returns the 5-tuple plus a dict of intermediates."""
    B, N, _ = pcl.shape
    C, H = img_feat.shape[1], img_feat.shape[2]
    t = {}
    pcl_offset = pcl_joint2offset(joint_xyz, pcl, 0.8)                                   # :295
    pcl_feat = gather_taps(img_feat, index, closeness)                                   # :297-299
    pcl_feat_rgb = gather_taps(img_feature_rgb, index, closeness)                        # :300-301
    pcl_weight = gather_taps(img_offset[:, 4 * J:], index, closeness)                    # :304-306
    t.update(pcl_offset=pcl_offset, pcl_feat_raw=pcl_feat, pcl_feat_rgb_raw=pcl_feat_rgb, pcl_weight=pcl_weight)
    e = conv_bn(p, prefix + "pcl_feat_emb.", pcl_feat) + conv_bn(p, prefix + "pcl_xyz_emb.", pcl) + \
        conv_bn(p, prefix + "pcl_pose_emb.", torch.cat([pcl_weight, pcl_offset], -1))    # :312-314
    e = torch.relu(e)
    e = torch.relu(e + conv_bn(p, prefix + "pcl_feat_emb_RGB.", pcl_feat_rgb))           # :317
    att = torch.softmax(pcl_weight.permute(0, 2, 1), -1)                                 # :319
    jf = att @ e                                                                         # :320
    t["joint_agg"] = jf
    jf = torch.relu(conv_bn(p, prefix + "joint_feat_emb.", jf) + conv_bn(p, prefix + "joint_xyz_emb.", joint_xyz))
    t.update(pcl_emb=e, joint_feat_pre=jf)
    jf = desa(p, prefix + "FA.", e, jf, pcl, joint_xyz)                                  # :327
    t["joint_feat_desa"] = jf
    tok, r3d = kp_interaction_tr(p, prefix + "init_TR.", jf)                             # :330
    hm = joint2heatmap(r3d[:, :, :2], 0.8, H, sigma=1)                                   # :334
    gam = img2anchor_dis(r3d, img_down, center, M, cube, cam, img_size)                  # :335
    sw, fj = spatial_aggregate(p, prefix, img_feature_rgb, hm, gam, prev_2d_feature)     # :336-344
    t.update(tok_init=tok, hm=hm, gam=gam)
    rj = updated_decoder(p, prefix + "crossTR.", fj, tok).permute(0, 2, 1)               # :347
    t["cross"] = rj
    _, r2d = kp_interaction_tr(p, prefix + "final_TR.", torch.cat([r3d, rj], 2))         # :348-349
    return (r3d, r2d, fj, sw, None), t


def fusion_path(p, img, pcl, img_offset, img_feat, img_feat_rgb, center, M, cube, cam, img_size=128, kernel=0.8,
                J=21, num_stages=2):
    """KPFusion.forward after the backbones, model.py:399-426.  p: KPFusion state_dict (block1.*, block2.*).
    -> (result[2:] = [r3d_1, r2d_1, r3d_2, r2d_2], spatial_weight[2], extras)."""
    H = img_feat.shape[2]
    joint_uvd = offset2joint_weight(img_offset, img, kernel)                             # :399
    img_down = nearest_down(img, H)                                                      # :409
    joint_xyz = torch.from_numpy(uvd_nl2xyznl(joint_uvd.numpy(), center, M, cube, cam, img_size))   # :410
    close, index, _ = img2pcl_index(pcl.numpy(), img_down.numpy(), center, M, cube, cam, img_size, 4)  # :411
    close, index = torch.from_numpy(close), torch.from_numpy(index)
    res, sws, prev = [], [], None
    extras = dict(joint_uvd=joint_uvd, joint_xyz0=joint_xyz, closeness=close, index=index)
    for i in range(num_stages):
        (r3d, r2d, prev, sw, _), t = block_kpfusion(p, f"block{i + 1}.", img_feat, img_feat_rgb, pcl, joint_xyz, close,
                                                    index, img_offset, prev, img_down, center, M, cube, cam, img_size, J)
        extras[f"block{i + 1}"] = t
        res += [r3d, r2d]
        sws.append(sw)
        joint_xyz = r2d                                                                  # :424
    return res, sws, extras


# ----------------------------------------------------------------------------------------------
# SURVEY 8f-3: crop + normalise front end of demo_RGBD.py (in-the-wild frames, BASELINE config 5)
#   get_center_from_bbx :253-276, comToBounds :519-529, getCrop :531-569, Crop_Image_deep_pp :410-462,
#   Crop_Image_deep_pp_RGB :464-517, normalize_img :378-385, jointImgTo3D :387-.  numpy only (cv2's INTER_NEAREST restated).
# ----------------------------------------------------------------------------------------------
def center_from_bbox(depth, bbx, upper=1500, lower=171):
    """depth [Hf,Wf] uint16, bbx (x,y,w,h) -> centre (u, v, d_mm) float64.  demo_RGBD.py:253-276."""
    c = np.array([0.0, 0.0, 300.0])
    x0, x1, y0, y1 = int(bbx[0]), int(bbx[0] + bbx[2]), int(bbx[1]), int(bbx[1] + bbx[3])
    img = depth[y0:y1, x0:x1]
    flag = np.logical_and(img <= upper, img >= lower)
    if flag.any():
        h, w = img.shape
        xs = np.linspace(0, w, w)
        ys = np.linspace(0, h, h)
        rr, cc = np.nonzero(flag)
        c[0] = xs[cc].mean()
        c[1] = ys[rr].mean()
        c[2] = img[flag].mean()
        if c[2] <= 0:
            c[2] = 300.0
    else:
        c[:] = (0, 0, 300.0)
    c[0] += bbx[0]
    c[1] += bbx[1]
    return c


def com_to_bounds(com, size, cam):
    """demo_RGBD.py:519-529 (float64, then floor)."""
    fx, fy, fu, fv = [float(t) for t in cam]
    zs, ze = com[2] - size[2] / 2., com[2] + size[2] / 2.
    xs = int(np.floor((com[0] * com[2] / fx - size[0] / 2.) / com[2] * fx + 0.5))
    xe = int(np.floor((com[0] * com[2] / fx + size[0] / 2.) / com[2] * fx + 0.5))
    ys = int(np.floor((com[1] * com[2] / fy - size[1] / 2.) / com[2] * fy + 0.5))
    ye = int(np.floor((com[1] * com[2] / fy + size[1] / 2.) / com[2] * fy + 0.5))
    return xs, xe, ys, ye, zs, ze


def _nearest_map(dst, src):
    """cv2.resize INTER_NEAREST source index: min(floor(x * (1 / (dst/src))), src-1) in double."""
    ifx = 1.0 / (float(dst) / float(src))
    return np.minimum(np.floor(np.arange(dst) * ifx).astype(np.int64), src - 1)


def crop_geometry(com, size, cam, dsize):
    """Bounds, resized size, paste offset and the 3x3 transform of Crop_Image_deep_pp (demo_RGBD.py:410-462)."""
    xs, xe, ys, ye, zs, ze = com_to_bounds(com, size, cam)
    wb, hb = xe - xs, ye - ys
    sz = (dsize, int(hb * dsize / wb)) if wb > hb else (int(wb * dsize / hb), dsize)   # (width, height)
    ch, cw = hb, wb                                                                    # cropped.shape after padding
    sc = sz[1] / float(ch) if ch > cw else sz[0] / float(cw)
    px = int(np.floor(dsize / 2. - sz[0] / 2.))
    py = int(np.floor(dsize / 2. - sz[1] / 2.))
    trans = np.eye(3)
    trans[0, 2], trans[1, 2] = -xs, -ys
    scale = np.eye(3) * sc
    scale[2, 2] = 1
    off = np.eye(3)
    off[0, 2], off[1, 2] = px, py
    return dict(xs=xs, xe=xe, ys=ys, ye=ye, zs=zs, ze=ze, sz=sz, px=px, py=py, M=off @ scale @ trans)


def crop_depth(depth, com, size, cam, dsize=128):
    """uint16 frame -> (normalised crop [dsize,dsize] f32, M [3,3] f64, com3D [3] f64).  process_depth demo_RGBD.py:305-316:
    Crop_Image_deep_pp on the uint16 frame (z-threshold writes are cast to uint16, like numpy does), nearest resize,
    centred paste into zeros, normalize_img (premax = crop max)."""
    g = crop_geometry(com, size, cam, dsize)
    Hf, Wf = depth.shape
    sx = _nearest_map(g["sz"][0], g["xe"] - g["xs"]) + g["xs"]       # source columns in the full frame
    sy = _nearest_map(g["sz"][1], g["ye"] - g["ys"]) + g["ys"]
    inside = ((sy >= 0) & (sy < Hf))[:, None] & ((sx >= 0) & (sx < Wf))[None, :]
    vals = np.where(inside, depth[np.clip(sy, 0, Hf - 1)][:, np.clip(sx, 0, Wf - 1)], 0).astype(depth.dtype)
    nz = vals != 0
    zs_cast = np.array(g["zs"]).astype(depth.dtype)                  # cropped[msk1] = zstart on a uint16 array
    vals = np.where(nz & (vals < g["zs"]), zs_cast, vals)
    vals = np.where(nz & (vals > g["ze"]), 0, vals).astype(depth.dtype)
    ret = np.zeros((dsize, dsize), np.float32)
    ret[g["py"]:g["py"] + g["sz"][1], g["px"]:g["px"] + g["sz"][0]] = vals
    hi, lo = com[2] + size[2] / 2., com[2] - size[2] / 2.
    premax = ret.max()
    ret[ret == premax] = hi
    ret[ret == 0] = hi
    ret[ret >= hi] = hi
    ret[ret <= lo] = lo
    ret -= com[2]
    ret /= (size[2] / 2.)
    fx, fy, fu, fv = [float(t) for t in cam]
    com3d = np.array([(com[0] - fu) * com[2] / fx, (com[1] - fv) * com[2] / fy, com[2]]).astype(np.float32)  # jointImgTo3D returns f32
    return ret, g["M"], com3d


def crop_rgb(rgb, com, size, cam, dsize=128):
    """uint8 HWC (BGR as cv2 gives it) -> [3,dsize,dsize] f32 in [0,1].  Crop_Image_deep_pp_RGB :464-517 + ToTensor()/255 (:87)."""
    g = crop_geometry(com, size, cam, dsize)
    Hf, Wf = rgb.shape[:2]
    sx = _nearest_map(g["sz"][0], g["xe"] - g["xs"]) + g["xs"]
    sy = _nearest_map(g["sz"][1], g["ye"] - g["ys"]) + g["ys"]
    inside = ((sy >= 0) & (sy < Hf))[:, None] & ((sx >= 0) & (sx < Wf))[None, :]
    vals = np.where(inside[..., None], rgb[np.clip(sy, 0, Hf - 1)][:, np.clip(sx, 0, Wf - 1)], 0)
    ret = np.zeros((dsize, dsize, 3), np.float32)
    ret[g["py"]:g["py"] + g["sz"][1], g["px"]:g["px"] + g["sz"][0]] = vals
    return (ret.transpose(2, 0, 1) / np.float32(255.)).astype(np.float32)


# ----------------------------------------------------------------------------------------------
# SURVEY 8f-4: evaluation tail (train.py:470-488 xyz2error; util/generateFeature.py:681-703 rigid_align)
# ----------------------------------------------------------------------------------------------
def xyz2error(output, joint, center, cube):
    """[B,J,3] normalised -> per-joint error in mm [B,J].  train.py:470-488."""
    output, joint = np.asarray(output, f64), np.asarray(joint, f64)
    c = np.asarray(center, f64)[:, None, :]
    h = np.asarray(cube, f64)[:, None, :] / 2
    d = (output * h + c) - (joint * h + c)
    return np.sqrt((d * d).sum(-1))


def rigid_align(A, B):
    """Similarity (Umeyama) alignment of A onto B, both [J,3].  generateFeature.py:681-703."""
    n = A.shape[0]
    ca, cb = A.mean(0), B.mean(0)
    H = (A - ca).T @ (B - cb) / n
    U, s, V = np.linalg.svd(H)
    R = V.T @ U.T
    if np.linalg.det(R) < 0:
        s[-1] = -s[-1]
        V[2] = -V[2]
        R = V.T @ U.T
    c = 1 / np.var(A, axis=0).sum() * np.sum(s)
    t = -(c * R) @ ca + cb
    return (c * R @ A.T).T + t
