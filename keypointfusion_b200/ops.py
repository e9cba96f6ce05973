"""Tensor-level wrappers over the C ABI (include/kpf_b200.h); `custom_ops.py` registers them with `torch.library`.

Each function validates shapes/dtypes/devices in Python, allocates outputs with torch (PyTorch owns all memory) and
launches the kernel on `torch.cuda.current_stream()`.  There is NO fallback: non-CUDA tensors raise.
"""
import ctypes
import os

import torch

from . import _lib

F32, BF16 = 0, 1
_DT = {torch.float32: F32, torch.bfloat16: BF16}


_arg_devices = set()   # devices of the tensors whose pointers were taken since the last launch


def _p(t):
    if t is None:
        return None
    _arg_devices.add(t.device)
    return ctypes.c_void_p(t.data_ptr())


def _spatial_numel(t):
    """elements per (batch, channel) plane of an NC... tensor; valid for empty batches too"""
    n = 1
    for d in t.shape[2:]:
        n *= int(d)
    return n


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("keypointfusion_b200 kernels need CUDA tensors (no CPU fallback exists for this path)")


def _f32(t):
    _need_cuda(t)
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _feat(t):
    _need_cuda(t)
    if t.dtype not in _DT:
        t = t.float()
    return t.contiguous()


_launches = 0


def launch_count():
    """Number of kernel-launching C-ABI calls made so far by this process (bench.py's `gpu_launches` evidence)."""
    return _launches


_KERNELS_PER_CALL = {"kpf_desa_fused": 2, "kpf_gather_taps": 2}   # entry points that launch more than one kernel


def _call(name, *args):
    """Launch on the device the ARGUMENTS live on (not the thread's current device): `net.to('cuda:1')` without a
    `torch.cuda.set_device(1)` must work like every stock torch op; tensors on different devices are an error."""
    global _launches
    devs = set(_arg_devices)
    _arg_devices.clear()
    if len(devs) > 1:
        raise RuntimeError(f"{name}: arguments live on different devices {sorted(str(d) for d in devs)}")
    dev = devs.pop() if devs else torch.device("cuda", torch.cuda.current_device())
    if dev.type != "cuda":
        raise RuntimeError("keypointfusion_b200 kernels need CUDA tensors (no CPU fallback exists for this path)")
    with torch.cuda.device(dev):
        rc = getattr(_lib.lib(), name)(*args, ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    _lib.check(rc, name)
    _launches += _KERNELS_PER_CALL.get(name, 1)


_kvec_cache = {}


def kernel_vec(kernel_size, J, device):
    """float or per-joint tensor (generateFeature.py:76-80, :188-192) -> device [J] f32."""
    if torch.is_tensor(kernel_size):
        return kernel_size.to(device=device, dtype=torch.float32).reshape(-1).expand(J).contiguous()
    key = (float(kernel_size), J, str(device))
    v = _kvec_cache.get(key)
    if v is None:
        v = _kvec_cache[key] = torch.full((J,), float(kernel_size), device=device, dtype=torch.float32)
    return v


def _depth_view(img, fs=None):
    """[B,1,S,S] -> (tensor, batch stride, row stride, col stride, fs) addressing the nearest-down-sampled map
    (model.py:409) without copying when S/fs is an integer."""
    _need_cuda(img)
    if img.dtype != torch.float32:
        img = img.float()
    B, _, S, S2 = img.shape
    fs = S if fs is None else fs
    if S != fs:
        if S % fs == 0:
            img = img[:, :, ::S // fs, ::S // fs]
        else:
            img = torch.nn.functional.interpolate(img, [fs, fs])
    return img, img.stride(0), img.stride(2), img.stride(3), fs


# ------------------------------------------------------------------------------------------------ a1-a3
def getpcl(img, com3D, cube, M, cam, sample_num=1024, ranks=None, seed=0, clamp=False, flip=1.0):
    img, com3D, cube, M, cam = _f32(img), _f32(com3D), _f32(cube), _f32(M), _f32(cam)
    B, S = img.shape[0], img.shape[-1]
    pcl = torch.empty(B, sample_num, 3, device=img.device, dtype=torch.float32)
    count = torch.empty(B, device=img.device, dtype=torch.int32)
    if ranks is not None:
        _need_cuda(ranks)
        ranks = ranks.to(torch.int32).contiguous()
    _call("kpf_getpcl", _p(img), _p(com3D), _p(cube), _p(M), _p(cam), B, S, sample_num, _p(ranks), int(seed) & 0xFFFFFFFF,
          int(bool(clamp)), float(flip), _p(pcl), _p(count))
    return pcl, count


def backproject_all(img, com3D, cube, M, cam, flip=1.0):
    img, com3D, cube, M, cam = _f32(img), _f32(com3D), _f32(cube), _f32(M), _f32(cam)
    B, S = img.shape[0], img.shape[-1]
    xyz = torch.empty(B, S * S, 3, device=img.device, dtype=torch.float32)
    pix = torch.empty(B, S * S, device=img.device, dtype=torch.int32)
    count = torch.empty(B, device=img.device, dtype=torch.int32)
    _call("kpf_backproject_all", _p(img), _p(com3D), _p(cube), _p(M), _p(cam), B, S, float(flip), _p(xyz), _p(pix), _p(count))
    return xyz, pix, count


# ------------------------------------------------------------------------------------------------ a5
def uvd2xyz(uvd, center, M, cube, cam, img_size, flip=1.0):
    uvd, center, M, cube, cam = _f32(uvd), _f32(center), _f32(M), _f32(cube), _f32(cam)
    B, P, _ = uvd.shape
    out = torch.empty_like(uvd)
    _call("kpf_uvd2xyz", _p(uvd), _p(center), _p(M), _p(cube), _p(cam), B, P, float(img_size), float(flip), _p(out))
    return out


def xyz2uvd(xyz, center, M, cube, cam, img_size, flip=1.0):
    xyz, center, M, cube, cam = _f32(xyz), _f32(center), _f32(M), _f32(cube), _f32(cam)
    B, P, _ = xyz.shape
    out = torch.empty_like(xyz)
    _call("kpf_xyz2uvd", _p(xyz), _p(center), _p(M), _p(cube), _p(cam), B, P, float(img_size), float(flip), _p(out))
    return out


# ------------------------------------------------------------------------------------------------ a6
def spatial_order(pcl, center, M, cube, cam, img_size, fs, flip=1.0):
    """[B,N] i32 permutation sorting each sample's points by the fs x fs cell they project to (scheduling aid for
    img2pcl_index / point_embed; results do not depend on it)."""
    pcl, center, M, cube, cam = _f32(pcl), _f32(center), _f32(M), _f32(cube), _f32(cam)
    B, N, _ = pcl.shape
    order = torch.empty(B, N, device=pcl.device, dtype=torch.int32)
    _call("kpf_spatial_order", _p(pcl), _p(center), _p(M), _p(cube), _p(cam), B, N, int(fs), float(img_size), float(flip), _p(order))
    return order


def img2pcl_index(pcl, img, center, M, cube, cam, img_size, select_num=9, flip=1.0, fs=None, want_i64=True, want_i32=False, order=None):
    pcl, center, M, cube, cam = _f32(pcl), _f32(center), _f32(M), _f32(cube), _f32(cam)
    d, bs, rs, cs, fs = _depth_view(img, fs)
    B, N, _ = pcl.shape
    close = torch.empty(B, N, select_num, device=pcl.device, dtype=torch.float32)
    i64 = torch.empty(B, N, select_num, device=pcl.device, dtype=torch.int64) if want_i64 else None
    i32 = torch.empty(B, N, select_num, device=pcl.device, dtype=torch.int32) if want_i32 else None
    _call("kpf_img2pcl_index", _p(pcl), _p(d), bs, rs, cs, _p(center), _p(M), _p(cube), _p(cam), B, N, fs, float(img_size),
          float(flip), select_num, _p(order), _p(close), _p(i64), _p(i32))
    return close, i64, i32


# ------------------------------------------------------------------------------------------------ a4
def offset2joint_weight(offset, depth, kernel_size):
    offset, depth = _feat(offset), _f32(depth)
    B, C5, fs, _ = offset.shape
    J = C5 // 5
    out = torch.empty(B, J, 3, device=offset.device, dtype=torch.float32)
    kv = kernel_vec(kernel_size, J, offset.device)
    _call("kpf_offset2joint_weight", _p(offset), _DT[offset.dtype], _p(depth), B, J, fs, depth.shape[-1], _p(kv), _p(out))
    return out


# ------------------------------------------------------------------------------------------------ a7
def pcl_joint2offset(joint, pcl, kernel_size):
    joint, pcl = _f32(joint), _f32(pcl)
    B, J, _ = joint.shape
    N = pcl.shape[1]
    out = torch.empty(B, N, 4 * J, device=pcl.device, dtype=torch.float32)
    kv = kernel_vec(kernel_size, J, pcl.device)
    _call("kpf_pcl_joint2offset", _p(joint), _p(pcl), _p(kv), B, J, N, _p(out))
    return out


# ------------------------------------------------------------------------------------------------ a8
def gather_taps(feat, index, closeness, out=None, out_c0=0):
    """feat [B,C,H,W] or [B,C,HW] (a channel slice of a contiguous map is fine) -> [B,N,C] in feat's dtype."""
    _need_cuda(feat, index, closeness)
    if feat.dtype not in _DT:
        feat = feat.float()
    B, C = feat.shape[:2]
    HW = _spatial_numel(feat)
    inner_ok = feat[0].is_contiguous() if feat.dim() == 3 else feat[0].reshape(C, HW).is_contiguous()
    if not inner_ok:
        feat = feat.contiguous()
    bs = feat.stride(0)
    closeness = _f32(closeness)
    N, K = index.shape[1:]
    if index.dtype not in (torch.int64, torch.int32):
        index = index.long()
    index = index.contiguous()
    if out is None:
        out = torch.empty(B, N, C, device=feat.device, dtype=feat.dtype)
        out_c0 = 0
    assert out.dtype == feat.dtype and out.is_contiguous()
    # maps whose 16-byte-row slab fits shared memory take the one-kernel path (csrc/gather.cu); larger ones need a channels-last workspace
    rows = torch.empty(B, HW, (C + 7) // 8 * 8, device=feat.device, dtype=feat.dtype) if HW * 16 > 96 * 1024 else None
    _call("kpf_gather_taps", _p(feat), _DT[feat.dtype], bs, B, C, HW, _p(index), int(index.dtype == torch.int64), _p(closeness), N, K,
          _p(out), out.shape[-1], out_c0, _p(rows))
    return out


# ------------------------------------------------------------------------------------------------ a10, a11, a16
def joint2heatmap(joint, std, heatmap_size, sigma=1.5):
    joint = _f32(joint)
    B, J, D = joint.shape
    out = torch.empty(B, J, heatmap_size, heatmap_size, device=joint.device, dtype=torch.float32)
    _call("kpf_joint2heatmap", _p(joint), D, B, J, heatmap_size, float(std), float(sigma), _p(out))
    return out


def img2anchor_dis(joint_uvd, img, center, M, cube, cam, img_size, gamma=10, flip=1.0, fs=None):
    joint_uvd, center, M, cube, cam = _f32(joint_uvd), _f32(center), _f32(M), _f32(cube), _f32(cam)
    d, bs, rs, cs, fs = _depth_view(img, fs)
    B, J, _ = joint_uvd.shape
    out = torch.empty(B, J, fs, fs, device=joint_uvd.device, dtype=torch.float32)
    _call("kpf_img2anchor_dis", _p(joint_uvd), _p(d), bs, rs, cs, _p(center), _p(M), _p(cube), _p(cam), B, J, fs, float(img_size),
          float(flip), float(gamma), _p(out))
    return out


def joint2offset(joint, img, kernel_size, feature_size, eps=1e-8):
    img = _f32(img)
    B, S = img.shape[0], img.shape[-1]
    joint = _f32(joint.reshape(B, -1, 3))
    J = joint.shape[1]
    out = torch.empty(B, 4 * J, feature_size, feature_size, device=img.device, dtype=torch.float32)
    kv = kernel_vec(kernel_size, J, img.device)
    _call("kpf_joint2offset", _p(joint), _p(img), B, J, S, feature_size, _p(kv), float(eps), _p(out))
    return out


# ------------------------------------------------------------------------------------------------ a12
def spatial_aggregate(feat_rgb, joints, img, center, M, cube, cam, Wa, ba, weight_dis, fc_w, fc_b, prev=None, img_size=128,
                      flip=1.0, hm_std=0.8, hm_sigma=1.0, gamma=10.0, want_maps=False):
    feat_rgb = _feat(feat_rgb)
    B, C, fs, _ = feat_rgb.shape
    joints, center, M, cube, cam = _f32(joints), _f32(center), _f32(M), _f32(cube), _f32(cam)
    J = joints.shape[1]
    d, bs, rs, cs, fs = _depth_view(img, fs)
    Wa, ba, weight_dis, fc_w, fc_b = _f32(Wa.reshape(J, C + J)), _f32(ba), _f32(weight_dis), _f32(fc_w.reshape(-1)), _f32(fc_b)
    if fc_w.numel() != fs * fs or Wa.shape != (J, C + J):
        raise ValueError(f"atten_spatial / fc_spatial2joint_feature shapes {tuple(Wa.shape)}, {fc_w.numel()} do not match a {C}-channel {fs}x{fs} map")
    prev = _f32(prev) if prev is not None else None
    dev = feat_rgb.device
    sw = torch.empty(B, J, fs, fs, device=dev, dtype=torch.float32)
    fj = torch.empty(B, J, C, device=dev, dtype=torch.float32)
    hm = torch.empty_like(sw) if want_maps else None
    gam = torch.empty_like(sw) if want_maps else None
    _call("kpf_spatial_aggregate", _p(feat_rgb), _DT[feat_rgb.dtype], _p(joints), _p(d), bs, rs, cs, _p(center), _p(M), _p(cube),
          _p(cam), _p(Wa), _p(ba), _p(weight_dis), _p(fc_w), _p(fc_b), _p(prev), B, C, J, fs, float(img_size), float(flip),
          float(hm_std), float(hm_sigma), float(gamma), _p(sw), _p(fj), _p(hm), _p(gam))
    return (sw, fj, hm, gam) if want_maps else (sw, fj)


# ------------------------------------------------------------------------------------------------ a13
def pack_decoder_layer(sd, prefix, J, C):
    """state_dict of one TransformerDecoderLayer -> the f32 blob kpf_cross_decoder_layer expects (kpf_b200.h)."""
    g = lambda k: sd[prefix + k].detach().float()
    Wi, bi = g("multihead_attn.in_proj_weight"), g("multihead_attn.in_proj_bias")
    parts = [g("self_posembed.weight")[:J], g("cross_posembed.weight")[:J], Wi[:C].t(), bi[:C], Wi[C:].t(), bi[C:],
             g("multihead_attn.out_proj.weight").t(), g("multihead_attn.out_proj.bias"), g("norm2.weight"), g("norm2.bias"),
             g("linear1.weight").t(), g("linear1.bias"), g("linear2.weight").t(), g("linear2.bias"), g("norm3.weight"),
             g("norm3.bias")]
    return torch.cat([p.contiguous().reshape(-1) for p in parts]).contiguous()


def cross_decoder_layer(anchor, tokens, wpack, heads, ffn, out_jc=None, out_jc_c0=0, want_cj=True):
    anchor, tokens, wpack = _f32(anchor), _f32(tokens), _f32(wpack)
    B, J, C = anchor.shape
    out_cj = torch.empty(B, C, J, device=anchor.device, dtype=torch.float32) if want_cj else None
    stride = out_jc.shape[-1] if out_jc is not None else 0
    _call("kpf_cross_decoder_layer", _p(anchor), _p(tokens), _p(wpack), B, J, C, ffn, heads, _p(out_cj), _p(out_jc), stride, out_jc_c0)
    return out_cj


# ------------------------------------------------------------------------------------------------ 8b: general-shape attention
def _rows3(t, name):
    """fp32 CUDA tensor [B,P,K] with ARBITRARY strides (views such as `x.transpose(0, 1)` or `feat.flatten(2).permute(0, 2, 1)` are
    addressed in place; nothing is copied)."""
    _need_cuda(t)
    if t.dim() != 3:
        raise ValueError(f"{name}: expected a [B,P,K] tensor, got {tuple(t.shape)}")
    return t if t.dtype == torch.float32 else t.float()


ROWS_BPO, ROWS_BOP, ROWS_PBO = 0, 1, 2   # linear_rows output layouts: [B,P,O] | channel-major [B,O,P] | sequence-first [P,B,O]


def linear_rows(x, weight, bias=None, pos=None, pos_index=None, scale=1.0, relu=False, out=None, out_layout=ROWS_BPO):
    """out[b,p,:] = act(((x[b,p,:] + pos_row) @ weight.T + bias) * scale)   (csrc/attn_general.cu).
    x [B,P,K] any strides; weight [O,K]; pos None | [B or 1,P,K] any strides | an nn.Embedding table [n,K] with pos_index [B,P] i64;
    out None -> a new contiguous tensor in `out_layout` ([B,P,O]; ROWS_BOP: [B,O,P]; ROWS_PBO: [P,B,O] -- written in place through
    strides, no transposed copy), or a preallocated [B,P,O] VIEW with any strides."""
    x = _rows3(x, "linear_rows")
    B, P, K = x.shape
    weight = _f32(weight)
    O = weight.shape[0]
    if weight.shape != (O, K):
        raise ValueError(f"linear_rows: weight {tuple(weight.shape)} does not match K = {K}")
    bias = None if bias is None else _f32(bias)
    pb = pp = pk = 0
    idx = None
    if pos_index is not None:
        pos = _f32(pos)
        _need_cuda(pos_index)
        idx = pos_index.to(torch.int64).expand(B, P).contiguous()
        pp, pk = pos.stride(0), pos.stride(1)
    elif pos is not None:
        pos = _rows3(pos, "linear_rows (pos)")
        if pos.shape[1:] != (P, K) or pos.shape[0] not in (1, B):
            raise ValueError(f"linear_rows: pos {tuple(pos.shape)} does not match x {tuple(x.shape)}")
        pb, pp, pk = (0 if pos.shape[0] == 1 else pos.stride(0)), pos.stride(1), pos.stride(2)
    ret = None
    if out is None:
        if out_layout == ROWS_BOP:
            ret = torch.empty(B, O, P, device=x.device, dtype=torch.float32)
            out = ret.transpose(1, 2)
        elif out_layout == ROWS_PBO:
            ret = torch.empty(P, B, O, device=x.device, dtype=torch.float32)
            out = ret.transpose(0, 1)
        else:
            ret = out = torch.empty(B, P, O, device=x.device, dtype=torch.float32)
    elif out.shape != (B, P, O) or out.dtype != torch.float32:
        raise ValueError(f"linear_rows: out {tuple(out.shape)} / {out.dtype}, expected {(B, P, O)} float32")
    _call("kpf_linear_rows", _p(x), x.stride(0), x.stride(1), x.stride(2), _p(pos), pb, pp, pk, _p(idx), _p(weight), _p(bias), B, P, K, O,
          float(scale), int(bool(relu)), _p(out), out.stride(0), out.stride(1), out.stride(2))
    return out if ret is None else ret


def mha_core(q, k, v, num_heads, attn_mask=None, key_padding_mask=None, need_weights=False):
    """softmax(q k^T + masks) v per head.  q [B,Pq,C] (already scaled), k / v [B,Pk,C]: unit stride over C, any batch / row strides
    (e.g. the two halves of a fused [B,Pk,2C] projection).  -> (out [B,Pq,C], head-averaged weights [B,Pq,Pk] or None)."""
    q, k, v = _rows3(q, "mha_core"), _rows3(k, "mha_core"), _rows3(v, "mha_core")
    q, k, v = (t if t.stride(2) == 1 else t.contiguous() for t in (q, k, v))
    B, Pq, C = q.shape
    Pk = k.shape[1]
    if k.shape != (B, Pk, C) or v.shape != (B, Pk, C) or C % num_heads or C // num_heads > 64:
        raise ValueError(f"mha_core: q {tuple(q.shape)}, k {tuple(k.shape)}, v {tuple(v.shape)}, {num_heads} heads (head_dim <= 64)")
    if attn_mask is not None:
        _need_cuda(attn_mask)
        if attn_mask.dtype == torch.bool:   # newer torch semantics: True = not allowed
            attn_mask = torch.zeros(attn_mask.shape, device=q.device).masked_fill_(attn_mask, float("-inf"))
        attn_mask = _f32(attn_mask)
        if attn_mask.shape != (Pq, Pk):
            raise ValueError(f"mha_core: attn_mask {tuple(attn_mask.shape)}, expected {(Pq, Pk)}")
    if key_padding_mask is not None:
        _need_cuda(key_padding_mask)
        if key_padding_mask.shape != (B, Pk):
            raise ValueError(f"mha_core: key_padding_mask {tuple(key_padding_mask.shape)}, expected {(B, Pk)}")
        key_padding_mask = key_padding_mask.to(torch.uint8).contiguous()
    out = torch.empty(B, Pq, C, device=q.device, dtype=torch.float32)
    stats = torch.empty(B, Pq, num_heads, 2, device=q.device, dtype=torch.float32) if need_weights else None
    w = torch.empty(B, Pq, Pk, device=q.device, dtype=torch.float32) if need_weights else None
    _call("kpf_mha_core", _p(q), q.stride(0), q.stride(1), _p(k), k.stride(0), k.stride(1), _p(v), v.stride(0), v.stride(1), _p(attn_mask),
          _p(key_padding_mask), B, Pq, Pk, C, num_heads, _p(out), out.stride(0), out.stride(1), _p(stats), _p(w))
    return out, w


def add_layernorm_rows(x, r, gamma, beta, eps=1e-5, channel_major=False):
    """LayerNorm(x + r) over the last dimension.  x [B,P,C] (any strides), r [B,P,C] or None -> [B,P,C], or the reference's
    channel-major [B,C,P] (transfusion_head.py:172) when channel_major."""
    x = _rows3(x, "add_layernorm_rows")
    B, P, C = x.shape
    r = None if r is None else _f32(r)
    if r is not None and r.shape != (B, P, C):
        raise ValueError(f"add_layernorm_rows: r {tuple(r.shape)} != x {tuple(x.shape)}")
    gamma, beta = _f32(gamma), _f32(beta)
    if channel_major:
        y = torch.empty(B, C, P, device=x.device, dtype=torch.float32)
        ys = (C * P, 1, P)
    else:
        y = torch.empty(B, P, C, device=x.device, dtype=torch.float32)
        ys = (P * C, C, 1)
    _call("kpf_add_layernorm_rows", _p(x), x.stride(0), x.stride(1), x.stride(2), _p(r), _p(gamma), _p(beta), B, P, C, float(eps), _p(y), *ys)
    return y


def sine_posembed(dim_t, B, H, W, mask=None, normalize=False, scale=6.283185307179586):
    """DetrSinePositionEmbedding.forward (transfusion_head.py:75-91): -> [B, 2*len(dim_t), H, W] f32."""
    dim_t = _f32(dim_t)
    D = dim_t.numel()
    if mask is not None:
        mask = _f32(mask)
        if mask.shape != (B, H, W):
            raise ValueError(f"sine_posembed: mask {tuple(mask.shape)}, expected {(B, H, W)}")
    out = torch.empty(B, 2 * D, H, W, device=dim_t.device, dtype=torch.float32)
    _call("kpf_sine_posembed", _p(mask), _p(dim_t), B, H, W, D, int(bool(normalize)), float(scale), _p(out))
    return out


# ------------------------------------------------------------------------------------------------ a14, a15
def channel_mean(x):
    x = _feat(x)
    B, C = x.shape[:2]
    out = torch.empty(B, C, device=x.device, dtype=torch.float32)
    _call("kpf_channel_mean", _p(x), _DT[x.dtype], B * C, _spatial_numel(x), _p(out))
    return out


def rgbd_fusion(rgb, depth, gate_w, gate_b, want_attn_mean=False):
    rgb, depth = _feat(rgb), _feat(depth)
    if depth.dtype != rgb.dtype:
        depth = depth.to(rgb.dtype)
    B, C = rgb.shape[:2]
    HW = _spatial_numel(rgb)
    ro, do, mg = torch.empty_like(rgb), torch.empty_like(rgb), torch.empty_like(rgb)
    asum = torch.zeros(2, device=rgb.device, dtype=torch.float32) if want_attn_mean else None
    gate_w, gate_b = _f32(gate_w), _f32(gate_b)
    _call("kpf_rgbd_fusion", _p(rgb), _p(depth), _DT[rgb.dtype], _p(gate_w), _p(gate_b), B, C, HW, _p(ro), _p(do), _p(mg), _p(asum))
    return ro, do, mg, (asum / (B * HW) if want_attn_mean else None)


def ac_fusion(rgb, depth, w_rgb, b_rgb, w_depth, b_depth):
    rgb, depth = _feat(rgb), _feat(depth)
    if depth.dtype != rgb.dtype:
        depth = depth.to(rgb.dtype)
    B, C = rgb.shape[:2]
    HW = _spatial_numel(rgb)
    mr, md = channel_mean(rgb), channel_mean(depth)
    ro, do, mg = torch.empty_like(rgb), torch.empty_like(rgb), torch.empty_like(rgb)
    w_rgb, b_rgb, w_depth, b_depth = _f32(w_rgb.reshape(C, C)), _f32(b_rgb), _f32(w_depth.reshape(C, C)), _f32(b_depth)
    _call("kpf_ac_fusion", _p(rgb), _p(depth), _DT[rgb.dtype], _p(mr), _p(md), _p(w_rgb), _p(b_rgb), _p(w_depth), _p(b_depth), B, C, HW,
          _p(ro), _p(do), _p(mg))
    return ro, do, mg


def fsp(guide, main, w0, b0, w2, b2):
    guide, main = _feat(guide), _feat(main)
    if main.dtype != guide.dtype:
        main = main.to(guide.dtype)
    B, C = guide.shape[:2]
    HW = _spatial_numel(guide)
    out = torch.empty_like(main)
    mg, mm = channel_mean(guide), channel_mean(main)  # keep references alive until the launch is enqueued
    w0, b0, w2, b2 = _f32(w0), _f32(b0), _f32(w2), _f32(b2)
    _call("kpf_fsp", _p(guide), _p(main), _DT[guide.dtype], _p(mg), _p(mm), _p(w0), _p(b0), _p(w2), _p(b2), B, C, w0.shape[0], HW,
          _p(out))
    return out


# ------------------------------------------------------------------------------------------------ 8f-1 DESA
def ball_query(xyz, centers, radius, nsample):
    xyz, centers = _f32(xyz), _f32(centers)
    B, Np, _ = xyz.shape
    J = centers.shape[1]
    idx = torch.empty(B, J, nsample, device=xyz.device, dtype=torch.int32)
    _call("kpf_ball_query", _p(xyz), _p(centers), B, Np, J, float(radius), nsample, _p(idx))
    return idx


# ------------------------------------------------------------------------------------------------ split-precision operands
# fp32 weights / activations reach the tensor cores as two 16-bit planes (hi = rn16(x), lo = rn16(x - hi)), three MMAs per product
# (csrc/tcgen05.cuh).  fp16 planes carry 22 mantissa bits (results indistinguishable from an fp32 GEMM), bf16 planes 16 bits
# with the full fp32 exponent range.  KPF_SPLIT_FMT=bf16 selects the latter, e.g. for a checkpoint with |w| or |activation| > 65504.
FMT_F16, FMT_BF16 = 0, 1
SPLIT_FMT = FMT_BF16 if os.environ.get("KPF_SPLIT_FMT", "fp16").lower() in ("bf16", "1") else FMT_F16


def _fmt_dtype(fmt):
    return torch.float16 if fmt == FMT_F16 else torch.bfloat16


def split_planes(W, fmt=None):
    """fp32 tensor -> (hi, lo) 16-bit planes with hi + lo == W to ~2^-22 (fp16) / 2^-16 (bf16) relative."""
    fmt = SPLIT_FMT if fmt is None else fmt
    dt = _fmt_dtype(fmt)
    W = W.detach().float()
    if fmt == FMT_F16 and W.numel() and float(W.abs().max()) > 6.0e4:
        raise ValueError("weight magnitude exceeds the fp16 plane range; set KPF_SPLIT_FMT=bf16")
    hi = W.to(dt)
    lo = (W - hi.float()).to(dt)
    return hi, lo


def _canon16(W16):
    """[N,K] 16-bit -> SWIZZLE_NONE canonical K-major operand [K/8][N][8] (csrc/tcgen05.cuh), flattened, as raw int16 bits."""
    N, K = W16.shape
    assert K % 8 == 0
    return W16.reshape(N, K // 8, 8).permute(1, 0, 2).contiguous().reshape(-1).view(torch.int16)


def _canon(W, fmt=None):
    """[N,K] fp32 -> canonical hi plane followed by canonical lo plane (int16 bits)."""
    hi, lo = split_planes(W, fmt)
    return torch.cat([_canon16(hi), _canon16(lo)])


def _pad(v, n):
    v = v.detach().float().reshape(-1)
    return torch.cat([v, v.new_zeros(n - v.numel())]) if v.numel() < n else v


# ------------------------------------------------------------------------------------------------ tensor-core token stacks
class TokenProgram:
    """Packed weights of one kpf_token_stack launch: optional cross layer, optional DESA-fusion prologue, optional encoder."""

    def __init__(self, wmat, wseq, wvec, cross, pre, D, L, F, Fc, J, fmt):
        self.wmat, self.wseq, self.wvec = wmat, wseq, wvec
        self.cross, self.pre, self.D, self.L, self.F, self.Fc, self.J, self.fmt = cross, pre, D, L, F, Fc, J, fmt
        self.n_weights = wseq.shape[0]

    def to(self, device):
        self.wmat, self.wseq, self.wvec = self.wmat.to(device), self.wseq.to(device), self.wvec.to(device)
        return self


def pack_token_program(J, enc=None, cross=None, fusion=None, C=128, fmt=None):
    """enc = (state_dict, prefix) of a KP_Interaction_TR; cross = (state_dict, prefix) of one TransformerDecoderLayer;
    fusion = (W [128,512], b [128]) BN-folded DESA fusion conv.  Weight order = consumption order of csrc/token_stack.cu.

    wmat is a sequence of ring entries (<= 32 KB each): a [128,128] matrix is two half-K tiles, each = canonical hi plane
    [8][128] + canonical lo plane; a 16-wide FFN is one entry (W1 hi | W1 lo | W2 hi | W2 lo); the embedding's K tail one entry.
    wseq row e = (source offset, count) in 16-byte units, the layer whose per-layer vectors the producer loads in front of
    entry e (-1: none), 0."""
    fmt = SPLIT_FMT if fmt is None else fmt
    mats, seq, vecs, off = [], [], [], 0

    def add(m):
        nonlocal off
        n = m.numel() // 8
        assert n <= 2048 and m.numel() % 8 == 0
        seq.append([off, n, -1, 0])
        mats.append(m)
        off += n

    def add_mat(W):   # [128,128] (as A operand) or [N=128,K=128] (as B operand): two half-K tiles
        assert tuple(W.shape) == (C, C), W.shape
        for h in range(2):
            add(_canon(W[:, 64 * h:64 * (h + 1)], fmt))

    def add_ffn(W1, W2):
        Fh = W1.shape[0]
        if Fh == 16:
            add(torch.cat([_canon(W1, fmt), _canon(W2, fmt)]))     # [16,128] K-major B operand ; [128,16] K-major A operand
        elif Fh == C:
            add_mat(W1)
            add_mat(W2)
        else:
            raise NotImplementedError(f"FFN width {Fh}: the token-stack kernel covers 16 (BERT intermediate) and 128 (decoder layer)")
        return Fh

    layer_base = []

    def add_layer(Wq, Wk, Wv, Wo, W1, W2):
        layer_base.append(len(seq))
        for W in (Wk, Wq, Wv, Wo):   # consumption order of csrc/token_stack.cu: K first, so that V's weights can follow into K's slots
            add_mat(W)
        return add_ffn(W1, W2)
    Fc = D = L = F_ = 0
    if cross is not None:
        sd, pf = cross
        g = lambda k: sd[pf + k].detach().float()
        Wi, bi = g("multihead_attn.in_proj_weight"), g("multihead_attn.in_proj_bias")
        Fc = add_layer(Wi[:C], Wi[C:2 * C], Wi[2 * C:], g("multihead_attn.out_proj.weight"), g("linear1.weight"), g("linear2.weight"))
        vecs += [g("self_posembed.weight")[:J].reshape(-1), g("cross_posembed.weight")[:J].reshape(-1), bi[:C], bi[C:2 * C], bi[2 * C:],
                 g("multihead_attn.out_proj.bias"), g("norm2.weight"), g("norm2.bias"), _pad(g("linear1.bias"), C), g("linear2.bias"),
                 g("norm3.weight"), g("norm3.bias")]
    if fusion is not None:
        Wfu, bfu = fusion
        for s_ in range(4):
            add_mat(Wfu.detach().float()[:, C * s_:C * (s_ + 1)])
        vecs.append(bfu.detach().float())
    if enc is not None:
        sd, pf = enc
        g = lambda k: sd[pf + k].detach().float()
        Wemb = g("bert.img_embedding.weight")
        D = Wemb.shape[1]
        shift = D - C
        add_mat(Wemb[:, shift:])
        if shift > 0:
            T = Wemb.new_zeros(C, 16)
            T[:, :shift] = Wemb[:, :shift]
            add(_canon(T, fmt))   # K tail: [2][128] hi | lo
        Wres = g("residual.weight")                       # [3, D] -> 16-byte aligned rows: [3][16] lead (zero padded) | [3][128] features
        lead = Wres.new_zeros(3, 16)
        lead[:, :shift] = Wres[:, :shift]
        vecs += [g("bert.position_embeddings.weight")[:J].reshape(-1), g("bert.img_embedding.bias"), lead.reshape(-1),
                 Wres[:, shift:].reshape(-1), _pad(g("residual.bias"), 4), g("cls_head.weight").reshape(-1), _pad(g("cls_head.bias"), 4)]
        while f"{pf}bert.encoder.layer.{L}.attention.self.query.weight" in sd:
            lp = f"bert.encoder.layer.{L}."
            F_ = add_layer(*(g(lp + k_ + ".weight") for k_ in ("attention.self.query", "attention.self.key", "attention.self.value",
                                                               "attention.output.dense", "intermediate.dense", "output.dense")))
            vecs += [g(lp + "attention.self.query.bias"), g(lp + "attention.self.key.bias"), g(lp + "attention.self.value.bias"),
                     g(lp + "attention.output.dense.bias"), g(lp + "attention.output.LayerNorm.weight"),
                     g(lp + "attention.output.LayerNorm.bias"), _pad(g(lp + "intermediate.dense.bias"), C), g(lp + "output.dense.bias"),
                     g(lp + "output.LayerNorm.weight"), g(lp + "output.LayerNorm.bias")]
            L += 1
    # vector prefetch schedule: layer 0's vectors in front of the first entry, layer it+1's in front of layer it's V weights
    # (by then the ring guarantees layer it-1 has finished, so the buffer they overwrite is free: csrc/token_stack.cu)
    if layer_base:
        seq[0][2] = 0
        for it, base in enumerate(layer_base[:-1]):
            seq[base + 4][2] = it + 1
    return TokenProgram(torch.cat(mats).contiguous(), torch.tensor(seq, dtype=torch.int32).contiguous(),
                        torch.cat([v.reshape(-1) for v in vecs]).contiguous(), int(cross is not None), int(fusion is not None), D, L, F_, Fc, J,
                        fmt)


def token_stack(pk, x=None, y=None, r3d=None, desa=None, jf=None, want_tokens=True, out_jc=None, out_jc_c0=0, want_cj=False,
                exchange=None):
    """Run one packed token program.  Returns (tokens [B,J,128] | None, pred [B,J,3] | None, out_cj [B,128,J] | None).
    exchange = (peer_ptrs [world] i64 device, xstep [1] i32 device, row0, rows_total): pred is also stored into every rank's gathered
    buffer (runtime.PeerExchange)."""
    ref = x if x is not None else desa
    dev = ref.device
    B = ref.shape[0]
    J = pk.J
    x = _f32(x) if x is not None else None
    y = _f32(y) if y is not None else None
    r3d = _f32(r3d) if r3d is not None else None
    desa = _f32(desa) if desa is not None else None
    jf = _f32(jf) if jf is not None else None
    tokens = torch.empty(B, J, 128, device=dev, dtype=torch.float32) if (want_tokens and (pk.L > 0 or (pk.pre and not pk.cross))) else None
    pred = torch.empty(B, J, 3, device=dev, dtype=torch.float32) if pk.L > 0 else None
    out_cj = torch.empty(B, 128, J, device=dev, dtype=torch.float32) if (want_cj and pk.L == 0) else None
    stride = out_jc.shape[-1] if out_jc is not None else 0
    _call("kpf_token_stack", _p(x), _p(y), _p(r3d), _p(desa), _p(jf), _p(pk.wmat), _p(pk.wseq), _p(pk.wvec), pk.n_weights, pk.cross, pk.pre,
          B, J, pk.D, pk.L, pk.F, pk.Fc, pk.fmt, _p(tokens), _p(pred), _p(out_cj), _p(out_jc), stride, out_jc_c0,
          _p(exchange[0]) if exchange else None, _p(exchange[1]) if exchange else None, exchange[0].numel() if exchange else 0,
          int(exchange[2]) if exchange else 0, int(exchange[3]) if exchange else 0)
    return tokens, pred, out_cj


def exchange_wait(buf, xstep, samples_per_step, inflight, flush=False):
    """Receiving side of the fused exchange (runtime.PeerExchange; include/kpf_b200.h: kpf_exchange_wait): begin a step (completing the
    previous one if it is in flight) or, with flush=True, complete the step in flight."""
    _call("kpf_exchange_wait", _p(buf), _p(xstep), int(samples_per_step), _p(inflight), 1 if flush else 0)


# ------------------------------------------------------------------------------------------------ fused point stage
_sm_count = {}


def sm_count(device):
    """Multiprocessors of `device` (cached): the persistent kernels' grid size, and one wave for K5's split."""
    i = torch.device(device).index or 0
    if i not in _sm_count:
        _sm_count[i] = torch.cuda.get_device_properties(i).multi_processor_count
    return _sm_count[i]


def repack_features(img_feat, img_feat_rgb, weight_map):
    """NCHW maps -> channels-last bf16 rows [B,HW,288] (128 depth-branch | 128 rgb-branch | J weight channels padded to 32).
    Returns (hi, lo): bf16 maps are exact in one plane (lo = None); fp32 maps are carried as two bf16 planes hi + lo."""
    _need_cuda(img_feat, img_feat_rgb, weight_map)
    dt = img_feat.dtype if img_feat.dtype in _DT else torch.float32
    f_d, f_rgb = img_feat.to(dt).contiguous(), img_feat_rgb.to(dt).contiguous()
    w = weight_map.to(dt)
    B, C = f_d.shape[:2]
    J = w.shape[1]
    HW = _spatial_numel(f_d)
    if B == 0 or not w[0].reshape(J, HW).is_contiguous():   # a channel slice of a larger map is fine as long as each sample is dense
        w = w.contiguous()
    out = torch.empty(B, HW, 288, device=f_d.device, dtype=torch.bfloat16)
    lo = torch.empty_like(out) if dt == torch.float32 else None
    _call("kpf_repack_features", _p(f_d), _p(f_rgb), _p(w), w.stride(0), _DT[dt], B, C, J, HW, _p(out), _p(lo))
    return out, lo


def pack_point_embed(Wf, bf, Wx, bx, Wp, bp, Wr, br, J, fmt=None):
    """BN-folded point-embedding weights (pcl_feat_emb, pcl_xyz_emb, pcl_pose_emb, pcl_feat_emb_RGB) -> (wmat 16-bit planes, wvec f32).
    A1 column order: [depth feats 128 | weight map J (+pad to 32) | (unit offset xyz, closeness) per joint, xyz 3 (+pad to 96)]
    (the reference's pcl_pose_emb input is [weight J | unit offsets 3J joint-major | closeness J], model.py:312-317).
    wmat = canonical W1 [128,256] hi | lo, W2 [128,128] hi | lo (csrc/point_embed.cu keeps them in tensor memory)."""
    C = Wf.shape[0]
    W1 = Wf.new_zeros(C, 256)
    W1[:, :128] = Wf
    W1[:, 128:128 + J] = Wp[:, :J]
    for j in range(J):
        W1[:, 160 + 4 * j:160 + 4 * j + 3] = Wp[:, J + 3 * j:J + 3 * j + 3]
        W1[:, 160 + 4 * j + 3] = Wp[:, 4 * J + j]
    W1[:, 160 + 4 * J:160 + 4 * J + 3] = Wx
    wmat = torch.cat([_canon(W1, fmt), _canon(Wr, fmt)]).contiguous()
    wvec = torch.cat([(bf + bx + bp).float(), br.float()]).contiguous()
    return wmat, wvec


E_ROW = 256   # 16-bit elements per point-feature row: [hi 128 | lo 128]


PE_STAGE_BYTES_PER_TILE = 79200   # include/kpf_b200.h: KPF_POINT_EMBED_STAGE_BYTES_PER_TILE


def point_embed_stage(B, N, device):
    """workspace for point_embed(stage_out=...) -> point_embed(stage_in=...): the gathered operand image of every 64-point tile"""
    return torch.empty(int(B) * (int(N) // 64) * PE_STAGE_BYTES_PER_TILE, device=device, dtype=torch.uint8)


def point_embed(featT, idx32, clos, pcl, joint, wmat, wvec, kernel_size=0.8, order=None, fmt=None, stage_out=None, stage_in=None):
    """featT = (hi, lo | None) from repack_features.
    -> e [B,N,256] int16 (rows [hi 128 | lo 128] in the split format), part_acc [B,T,128,32] f32, part_ms [B,T,2,32] f32  (T = N/64).
    stage_out: also store the gathered (joint-independent) operand image of every tile into this point_embed_stage buffer;
    stage_in: load those images (a launch on the same maps / taps / order filled them) instead of gathering: block 2 of KPFusion."""
    fmt = SPLIT_FMT if fmt is None else fmt
    feat_hi, feat_lo = featT if isinstance(featT, (tuple, list)) else (featT, None)
    _need_cuda(feat_hi, idx32, clos, pcl, joint)
    pcl, joint, clos = _f32(pcl), _f32(joint), _f32(clos)
    idx32 = idx32.to(torch.int32).contiguous()
    B, N, _ = pcl.shape
    J = joint.shape[1]
    HW = feat_hi.shape[1]
    if N % 64 or J > 21 or feat_hi.shape[2] != 288:
        raise NotImplementedError("the point stage covers N % 64 == 0 points, J <= 21 joints and 128-channel maps (no fallback path)")
    T = N // 64
    dev = pcl.device
    # 32 spare rows per sample behind the points: kpf_desa_fused appends the joints' own feature rows there (they are members
    # N .. N+J-1 of DESA's grouped point set); the returned tensor is the [B,N,256] view of the points
    e_full = torch.empty(B, N + 32, E_ROW, device=dev, dtype=torch.int16)
    e = e_full[:, :N]
    acc = torch.empty(B, T, 128, 32, device=dev, dtype=torch.float32)
    ms = torch.empty(B, T, 2, 32, device=dev, dtype=torch.float32)
    _call("kpf_point_embed", _p(feat_hi), _p(feat_lo), _p(idx32), _p(clos), _p(pcl), _p(joint), _p(order), _p(wmat), _p(wvec), B, N, J, HW,
          float(kernel_size), fmt, _p(e), e.stride(0), _p(acc), _p(ms), _p(stage_out), _p(stage_in), sm_count(dev))
    return e, acc, ms


def e_to_float(e, fmt=None):
    """[B,N,256] int16 point-feature rows -> [B,N,128] f32 (hi + lo); test / inspection helper."""
    dt = _fmt_dtype(SPLIT_FMT if fmt is None else fmt)
    return e[..., :128].contiguous().view(dt).float() + e[..., 128:].contiguous().view(dt).float()


def e_from_float(x, fmt=None, spare_rows=32):
    """[B,N,128] f32 -> [B,N,256] int16 rows (a view of a [B,N+spare_rows,256] buffer, as kpf_desa_fused wants)."""
    hi, lo = split_planes(x, fmt)
    B, N, _ = x.shape
    full = torch.zeros(B, N + spare_rows, E_ROW, device=x.device, dtype=torch.int16)
    full[:, :N, :128] = hi.view(torch.int16)
    full[:, :N, 128:] = lo.view(torch.int16)
    return full[:, :N]


def combine_point_partials(acc, ms, J):
    """flash-style combination of the per-tile softmax partials -> joint_agg [B,J,128] (torch glue used by tests)."""
    m_t, s_t = ms[:, :, 0, :J], ms[:, :, 1, :J]                      # B T J
    m = m_t.max(dim=1, keepdim=True)[0]
    sc = torch.exp(m_t - m)                                          # B T J
    num = (acc[:, :, :, :J] * sc.unsqueeze(2)).sum(1)                # B 128 J
    den = (s_t * sc).sum(1)                                          # B J
    return (num / den.unsqueeze(1)).permute(0, 2, 1).contiguous()


# ------------------------------------------------------------------------------------------------ fused DESA
def pack_desa(Wj, bj, Wjx, bjx, scales, fmt=None):
    """Wj [128,128], Wjx [128,3] (BN-folded joint_feat_emb / joint_xyz_emb); scales: list of (Wf0, bf0, Wl0, bl0, W2, b2), all BN-folded.
    -> (wmat 16-bit canonical planes: Wj hi | lo ; per scale W1 main hi | lo, W1 tail hi | lo, W2 hi | lo ; wvec f32) for kpf_desa_fused."""
    mats = [_canon(Wj, fmt)]
    wx = Wj.new_zeros(128, 4)
    wx[:, :3] = Wjx
    vecs = [(bj + bjx).float(), wx.reshape(-1).float()]
    for Wf0, bf0, Wl0, bl0, W2, b2 in scales:
        tail = Wf0.new_zeros(128, 16)
        tail[:, :3] = Wl0
        mats += [_canon(Wf0, fmt), _canon(tail, fmt), _canon(W2, fmt)]
        vecs += [(bf0 + bl0).float(), b2.float()]
    return torch.cat(mats).contiguous(), torch.cat(vecs).contiguous()


def desa_fused(e, part_acc, part_ms, pcl, joint, wmat, wvec, radius, nsample, fmt=None, jf_in=None, keep_scratch=None):
    """e: [B,N,256] int16 rows from point_embed (or e_from_float).  jf_in [B,J,128]: the joints' features are given (no embedding)."""
    fmt = SPLIT_FMT if fmt is None else fmt
    pcl, joint = _f32(pcl), _f32(joint)
    B, N, _ = pcl.shape
    J = joint.shape[1]
    S = len(radius)
    r = list(radius) + [0.0] * (4 - S)
    part = torch.empty(B, S, J, 128, device=pcl.device, dtype=torch.float32)
    jf = torch.empty(B, J, 128, device=pcl.device, dtype=torch.float32)
    assert e.dtype == torch.int16 and e.shape[-1] == E_ROW
    if e.stride(0) < (N + J) * E_ROW or e.stride(1) != E_ROW or e.stride(2) != 1:   # not from ops.point_embed: make room for the joint rows
        e_full = torch.empty(B, N + 32, E_ROW, device=pcl.device, dtype=torch.int16)
        e_full[:, :N].copy_(e)
        e = e_full[:, :N]
    # workspace between the two kernels: W1_s jf terms fp32 [B,S,J,128], padded xyz table [B,N+32,4] f32, ball-query indices u16
    # [B,S,J,nsample], widest ball per (sample, scale) i32 [B,S]
    scratch = torch.empty(B * S * J * 128 * 4 + B * (N + 32) * 16 + B * S * J * nsample * 2 + B * S * 4, device=pcl.device, dtype=torch.uint8)
    _call("kpf_desa_fused", _p(e), e.stride(0), _p(part_acc), _p(part_ms), _p(pcl), _p(joint), _p(wmat), _p(wvec), B, N, J, S, nsample, float(r[0]),
          float(r[1]), float(r[2]), float(r[3]), fmt, _p(_f32(jf_in) if jf_in is not None else None), _p(part), _p(jf), _p(scratch),
          sm_count(pcl.device))
    if keep_scratch is not None:   # tests read the ball-query indices back out of the hand-over workspace
        keep_scratch["buf"] = scratch
    return part, jf


# ------------------------------------------------------------------------------------------------ a12 on tensor cores
_counter_cache = {}
K5_SPLIT = None   # None: spread a sample's cell tiles over as many CTAs as fit one wave (latency); 1: one CTA per sample (SM-time)


def _zero_counters(n, device):
    """Persistent zeroed int32 workspace per (device, size, stream): kernels that use it leave it zero again."""
    key = (str(device), n, torch.cuda.current_stream(device).cuda_stream)
    c = _counter_cache.get(key)
    if c is None:
        c = _counter_cache[key] = torch.zeros(n, device=device, dtype=torch.int32)
    return c


def split_planes3_bf16(W):
    """fp32 -> three bf16 planes (hi + mid + lo = W to 2^-24): the GEMM partner of a bf16 feature-map operand (both operands of an
    MMA share one format, csrc/tcgen05.cuh)."""
    W = W.detach().float()
    hi = W.bfloat16()
    r = W - hi.float()
    mid = r.bfloat16()
    lo = (r - mid.float()).bfloat16()
    return hi, mid, lo


def pack_spatial_wa(Wa, J, C=128, fmt=None):
    """atten_spatial.weight [J, C+J(,1,1)] -> canonical 16-bit B operand planes: Wa[:, :C] as [16][32][8] x 3 bf16 planes (it multiplies the
    bf16 feature map), Wa[:, C:] as [4][32][8] hi | lo in the split format (it multiplies the computed heat map)."""
    Wa = Wa.detach().float().reshape(J, C + J)
    main = Wa.new_zeros(32, C)
    main[:J] = Wa[:, :C]
    hm = Wa.new_zeros(32, 32)
    hm[:J, :J] = Wa[:, C:]
    return torch.cat([_canon16(p_) for p_ in split_planes3_bf16(main)] + [_canon(hm, fmt)]).contiguous()


def split_map(x):
    """fp32 tensor -> (hi, lo) bf16 planes of the same shape (kpf_split_planes)."""
    x = _f32(x)
    hi = torch.empty(x.shape, device=x.device, dtype=torch.bfloat16)
    lo = torch.empty_like(hi)
    n = x.numel()
    if n % 4:
        raise NotImplementedError("split_map: element count must be a multiple of 4")
    _call("kpf_split_planes", _p(x), n, _p(hi), _p(lo))
    return hi, lo


def spatial_aggregate_tc(feat_rgb, joints, img, center, M, cube, cam, wa_packed, ba, weight_dis, fc_w, fc_b, prev=None, img_size=128,
                         flip=1.0, hm_std=0.8, hm_sigma=1.0, gamma=10.0, fmt=None):
    """feat_rgb: bf16 [B,128,fs,fs], or a (hi, lo) pair of bf16 planes (split_map of an fp32 map)."""
    fmt = SPLIT_FMT if fmt is None else fmt
    feat_rgb, feat_lo = feat_rgb if isinstance(feat_rgb, (tuple, list)) else (feat_rgb, None)
    _need_cuda(feat_rgb)
    assert feat_rgb.dtype == torch.bfloat16 and (feat_lo is None or feat_lo.dtype == torch.bfloat16)
    feat_rgb = feat_rgb.contiguous()
    feat_lo = feat_lo.contiguous() if feat_lo is not None else None
    B, C, fs, _ = feat_rgb.shape
    joints, center, M, cube, cam = _f32(joints), _f32(center), _f32(M), _f32(cube), _f32(cam)
    J = joints.shape[1]
    d, bs, rs, cs, fs = _depth_view(img, fs)
    ba, weight_dis, fc_w, fc_b = _f32(ba), _f32(weight_dis), _f32(fc_w.reshape(-1)), _f32(fc_b)
    if fc_w.numel() != fs * fs:
        raise ValueError(f"fc_spatial2joint_feature has {fc_w.numel()} inputs but the feature map has {fs}x{fs} cells (model.py:264 pins 32x32)")
    if C != 128 or (fs * fs) % 128 or J > 32:
        raise NotImplementedError("spatial aggregation covers 128-channel maps with fs*fs % 128 == 0 and J <= 32 (no fallback path)")
    prev = _f32(prev) if prev is not None else None
    sw = torch.empty(B, J, fs, fs, device=feat_rgb.device, dtype=torch.float32)
    fj = torch.empty(B, J, C, device=feat_rgb.device, dtype=torch.float32)
    T = fs * fs // 128
    # cell tiles of a sample spread over `split` CTAs: as many as still fit in ONE wave of one-CTA-per-SM (measured at B = 64:
    # split 1 / 2 / 4 / 8 -> 60 / 39 / 47 / 62 us)
    split = next((s_ for s_ in (8, 4, 2) if T % s_ == 0 and B * s_ <= sm_count(feat_rgb.device)), 1)
    # ... which is the LATENCY optimum of a launch that has the GPU to itself.  With several steps in flight what counts is the launch's
    # SM-time, and the per-CTA prologue (weights, tables, first tile) is paid `split` times: one CTA per sample is 60 us x 64 SMs against
    # 35 us x 128.  K5_SPLIT (set by the caller that overlaps steps, before it captures its graphs) overrides the policy: bench.py
    # at batch 64, six steps in flight, split 2 -> 1: 0.479 -> 0.464 ms per step (profiles/ab_overlap_r2.txt)
    if K5_SPLIT and T % K5_SPLIT == 0:
        split = K5_SPLIT
    scratch = torch.empty(B, split, 128, 32, device=feat_rgb.device, dtype=torch.float32) if split > 1 else None
    counters = _zero_counters(B, feat_rgb.device) if split > 1 else None
    _call("kpf_spatial_aggregate_tc", _p(feat_rgb), _p(feat_lo), _p(joints), _p(d), bs, rs, cs, _p(center), _p(M), _p(cube), _p(cam),
          _p(wa_packed), _p(ba), _p(weight_dis), _p(fc_w), _p(fc_b), _p(prev), B, C, J, fs, float(img_size), float(flip), float(hm_std),
          float(hm_sigma), float(gamma), fmt, _p(sw), _p(fj), _p(scratch), _p(counters), split)
    return sw, fj


# ------------------------------------------------------------------------------------------------ 8f-3 crop front end
def _u16(t):
    _need_cuda(t)
    if t.dtype == torch.uint16:
        return t.contiguous()
    if t.dtype == torch.int16:
        return t.contiguous()          # same bits
    return t.to(torch.int32).clamp_(0, 65535).to(torch.uint16).contiguous()


def _f64(t, device):
    if not torch.is_tensor(t):
        t = torch.as_tensor(t, dtype=torch.float64)
    return t.to(device=device, dtype=torch.float64).contiguous()


def frame_index_arg(frame_index, B, F, device):
    """frame_index of the front-end ops -> None or a [B] int32 tensor on `device`.
    None: box b reads frame b, which needs F == B.  Indices given on the host (list, numpy array, CPU tensor) are checked
    against [0, F) here, before any launch (ValueError).  A CUDA int32 tensor is passed through unchecked, so the calls can be
    captured in a CUDA graph; a box whose device index is out of range gets NaN outputs and reads no frame."""
    if frame_index is None:
        if F != B:
            raise ValueError(f"frame_index=None reads frame b for box b, but there are {F} frames and {B} boxes")
        return None
    if torch.is_tensor(frame_index) and frame_index.is_cuda:
        if frame_index.dtype != torch.int32 or tuple(frame_index.shape) != (B,):
            raise ValueError(f"a device frame_index must be an int32 tensor of shape ({B},), got {frame_index.dtype} {tuple(frame_index.shape)}")
        return frame_index.contiguous()
    fi = torch.as_tensor(frame_index)
    if fi.dtype.is_floating_point or fi.dtype.is_complex or fi.dtype == torch.bool:
        raise ValueError(f"frame_index must hold integers, got {fi.dtype}")
    fi = fi.reshape(-1)
    if fi.numel() != B:
        raise ValueError(f"frame_index has {fi.numel()} entries for {B} boxes")
    bad = (fi < 0) | (fi >= F)
    if bool(bad.any()):
        raise ValueError(f"frame_index {fi[bad].tolist()} outside [0, {F}) (F = number of frames)")
    return fi.to(device=device, dtype=torch.int32)


def center_from_bbox(depth_u16, bbox, upper=1500, lower=171, frame_index=None):
    """depth [F,Hf,Wf] uint16, bbox [B,4] (x,y,w,h) -> centre [B,3] f64 (u, v, d_mm); box b reads frame frame_index[b]."""
    F, Hf, Wf = depth_u16.shape
    B = torch.as_tensor(bbox).numel() // 4
    fi = frame_index_arg(frame_index, B, F, depth_u16.device)
    d = _u16(depth_u16)
    bbox = _f64(bbox, d.device).reshape(B, 4)
    out = torch.empty(B, 3, device=d.device, dtype=torch.float64)
    _call("kpf_center_from_bbox", _p(d), _p(bbox), _p(fi), F, B, Hf, Wf, int(upper), int(lower), _p(out))
    return out


def crop_depth(depth_u16, center, cube, cam, dsize=128, frame_index=None):
    """depth [F,Hf,Wf] uint16, center [B,3] -> (img [B,1,dsize,dsize], M [B,3,3], com3d [B,3], cube [B,3]); box b reads frame
    frame_index[b]."""
    F, Hf, Wf = depth_u16.shape
    B = torch.as_tensor(center).numel() // 3
    fi = frame_index_arg(frame_index, B, F, depth_u16.device)
    d = _u16(depth_u16)
    center, cam = _f64(center, d.device).reshape(B, 3), _f64(cam, d.device).reshape(-1, 4).expand(B, 4).contiguous()
    cube = torch.as_tensor(cube, dtype=torch.float32).to(d.device).reshape(-1, 3).expand(B, 3).contiguous()
    img = torch.empty(B, 1, dsize, dsize, device=d.device, dtype=torch.float32)
    M = torch.empty(B, 3, 3, device=d.device, dtype=torch.float32)
    com3d = torch.empty(B, 3, device=d.device, dtype=torch.float32)
    _call("kpf_crop_depth", _p(d), _p(center), _p(cube), _p(cam), _p(fi), F, B, Hf, Wf, dsize, _p(img), _p(M), _p(com3d))
    return img, M, com3d, cube


def crop_rgb(rgb_u8, center, cube, cam, dsize=128, frame_index=None):
    """rgb [F,Hf,Wf,3] uint8, center [B,3] -> [B,3,dsize,dsize] f32 in [0,1]; box b reads frame frame_index[b]."""
    F, Hf, Wf, _ = rgb_u8.shape
    B = torch.as_tensor(center).numel() // 3
    fi = frame_index_arg(frame_index, B, F, rgb_u8.device)
    _need_cuda(rgb_u8)
    r = rgb_u8.to(torch.uint8).contiguous()
    center, cam = _f64(center, r.device).reshape(B, 3), _f64(cam, r.device).reshape(-1, 4).expand(B, 4).contiguous()
    cube = torch.as_tensor(cube, dtype=torch.float32).to(r.device).reshape(-1, 3).expand(B, 3).contiguous()
    out = torch.empty(B, 3, dsize, dsize, device=r.device, dtype=torch.float32)
    _call("kpf_crop_rgb", _p(r), _p(center), _p(cube), _p(cam), _p(fi), F, B, Hf, Wf, dsize, _p(out))
    return out


def joints_to_frame(joints, center, cube, cam, flip=1.0):
    """Normalised joints [B,P,3] of crops with com3d `center` [B,3] (mm), `cube` [B,3], `cam` [B,4] (fx,fy,fu,fv) ->
    (uvd_frame [B,P,3]: frame pixels u, v and depth mm;  xyz_cam [B,P,3]: camera-space mm).  The points3DToImg half of
    xyz_nl2uvdnl_tensor (loader.py:821-834, :277-288): the same fp32 operations as xyz2uvd before it applies M."""
    joints, center, cube, cam = _f32(joints), _f32(center), _f32(cube), _f32(cam)
    B, P, _ = joints.shape
    uvd = torch.empty_like(joints)
    xyz = torch.empty_like(joints)
    _call("kpf_joints_to_frame", _p(joints), _p(center.reshape(B, 3)), _p(cube.reshape(B, 3)), _p(cam.reshape(B, 4)), B, P, float(flip),
          _p(uvd), _p(xyz))
    return uvd, xyz


# ------------------------------------------------------------------------------------------------ 8f-4 evaluation tail
def eval_errors(pred, gt, cube, aligned=True):
    """-> (err [B,J] mm, pa_err [B,J] mm | None): Trainer.xyz2error and the rigid_align'ed error of train.py:330-386."""
    pred, gt, cube = _f32(pred), _f32(gt), _f32(cube)
    B, J, _ = pred.shape
    err = torch.empty(B, J, device=pred.device, dtype=torch.float32)
    pa = torch.empty(B, J, device=pred.device, dtype=torch.float32) if aligned else None
    _call("kpf_eval_errors", _p(pred), _p(gt), _p(cube), B, J, _p(err), _p(pa))
    return err, pa
