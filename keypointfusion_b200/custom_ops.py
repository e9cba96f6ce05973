"""`torch.library` registration of the fusion-path operators: the thin custom-op layer between the drop-in nn.Modules and the C ABI.

Every operator a module calls on the hot path is a `torch.ops.kpf.*` custom op whose implementation is the ctypes launch in
`ops.py` (same validation, same allocation, same C-ABI entry) and whose `register_fake` gives the output shapes / dtypes / strides.
That is what lets the drop-ins sit next to the stock PyTorch backbones inside `torch.compile` / `torch.export` graphs:
`torch.compile(net.forward_path, fullgraph=True)` traces without a graph break (tests/test_custom_ops_gpu.py) and
`torch.library.opcheck` passes for each op.  Reference boundary these stand behind: model/model.py:11-19 (the names KPFusion imports)
and :395 (the `loader` helper object).

Conventions: optional OUTPUTS do not exist in the op schema, so an absent tensor result is returned as an empty (numel 0) tensor;
optional INPUTS are `Optional[Tensor]`.  Packed weights travel as plain tensors (+ ints).  No op aliases an input; `desa_fused`
declares that it writes into `e` (it appends the joints' rows behind the points of the same buffer).
"""
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import ops

_lib_ns = "kpf"


def _empty(dev):
    return torch.empty(0, device=dev)


def _op(name, mutates=()):
    return torch.library.custom_op(f"{_lib_ns}::{name}", mutates_args=mutates, device_types="cuda")


# ------------------------------------------------------------------------------------------------ geometry
@_op("getpcl")
def getpcl(img: Tensor, com3D: Tensor, cube: Tensor, M: Tensor, cam: Tensor, sample_num: int, seed: int, clamp: bool, flip: float,
           ranks: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    return ops.getpcl(img, com3D, cube, M, cam, sample_num, ranks=ranks, seed=seed, clamp=clamp, flip=flip)


@getpcl.register_fake
def _(img, com3D, cube, M, cam, sample_num, seed, clamp, flip, ranks=None):
    B = img.shape[0]
    return img.new_empty(B, sample_num, 3, dtype=torch.float32), img.new_empty(B, dtype=torch.int32)


@_op("offset2joint_weight")
def offset2joint_weight(offset: Tensor, depth: Tensor, kernel_size: float) -> Tensor:
    return ops.offset2joint_weight(offset, depth, kernel_size)


@offset2joint_weight.register_fake
def _(offset, depth, kernel_size):
    return offset.new_empty(offset.shape[0], offset.shape[1] // 5, 3, dtype=torch.float32)


@_op("uvd2xyz")
def uvd2xyz(uvd: Tensor, center: Tensor, M: Tensor, cube: Tensor, cam: Tensor, img_size: float, flip: float) -> Tensor:
    return ops.uvd2xyz(uvd, center, M, cube, cam, img_size, flip)


@uvd2xyz.register_fake
def _(uvd, center, M, cube, cam, img_size, flip):
    return uvd.new_empty(uvd.shape, dtype=torch.float32)


@_op("xyz2uvd")
def xyz2uvd(xyz: Tensor, center: Tensor, M: Tensor, cube: Tensor, cam: Tensor, img_size: float, flip: float) -> Tensor:
    return ops.xyz2uvd(xyz, center, M, cube, cam, img_size, flip)


@xyz2uvd.register_fake
def _(xyz, center, M, cube, cam, img_size, flip):
    return xyz.new_empty(xyz.shape, dtype=torch.float32)


@_op("spatial_order")
def spatial_order(pcl: Tensor, center: Tensor, M: Tensor, cube: Tensor, cam: Tensor, img_size: float, fs: int, flip: float) -> Tensor:
    return ops.spatial_order(pcl, center, M, cube, cam, img_size, fs, flip)


@spatial_order.register_fake
def _(pcl, center, M, cube, cam, img_size, fs, flip):
    return pcl.new_empty(pcl.shape[0], pcl.shape[1], dtype=torch.int32)


@_op("img2pcl_index")
def img2pcl_index(pcl: Tensor, img: Tensor, center: Tensor, M: Tensor, cube: Tensor, cam: Tensor, img_size: float, select_num: int,
                  flip: float, want_i64: bool, order: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    """-> (closeness [B,N,K] f32, index [B,N,K] i64 or i32).  `img` may be a strided view of the crop (fused nearest down-sample)."""
    close, i64, i32 = ops.img2pcl_index(pcl, img, center, M, cube, cam, img_size, select_num, flip, want_i64=want_i64,
                                        want_i32=not want_i64, order=order)
    return close, (i64 if want_i64 else i32)


@img2pcl_index.register_fake
def _(pcl, img, center, M, cube, cam, img_size, select_num, flip, want_i64, order=None):
    B, N = pcl.shape[:2]
    return pcl.new_empty(B, N, select_num, dtype=torch.float32), pcl.new_empty(B, N, select_num, dtype=torch.int64 if want_i64 else torch.int32)


@_op("pcl_joint2offset")
def pcl_joint2offset(joint: Tensor, pcl: Tensor, kernel_size: float) -> Tensor:
    return ops.pcl_joint2offset(joint, pcl, kernel_size)


@pcl_joint2offset.register_fake
def _(joint, pcl, kernel_size):
    return pcl.new_empty(pcl.shape[0], pcl.shape[1], 4 * joint.shape[1], dtype=torch.float32)


@_op("gather_taps")
def gather_taps(feat: Tensor, index: Tensor, closeness: Tensor) -> Tensor:
    return ops.gather_taps(feat, index, closeness)


@gather_taps.register_fake
def _(feat, index, closeness):
    dt = feat.dtype if feat.dtype in (torch.float32, torch.bfloat16) else torch.float32
    return feat.new_empty(feat.shape[0], index.shape[1], feat.shape[1], dtype=dt)


@_op("joint2heatmap")
def joint2heatmap(joint: Tensor, std: float, heatmap_size: int, sigma: float) -> Tensor:
    return ops.joint2heatmap(joint, std, heatmap_size, sigma)


@joint2heatmap.register_fake
def _(joint, std, heatmap_size, sigma):
    return joint.new_empty(joint.shape[0], joint.shape[1], heatmap_size, heatmap_size, dtype=torch.float32)


@_op("img2anchor_dis")
def img2anchor_dis(joint_uvd: Tensor, img: Tensor, center: Tensor, M: Tensor, cube: Tensor, cam: Tensor, img_size: float, gamma: float,
                   flip: float) -> Tensor:
    return ops.img2anchor_dis(joint_uvd, img, center, M, cube, cam, img_size, gamma, flip)


@img2anchor_dis.register_fake
def _(joint_uvd, img, center, M, cube, cam, img_size, gamma, flip):
    return joint_uvd.new_empty(joint_uvd.shape[0], joint_uvd.shape[1], img.shape[-2], img.shape[-1], dtype=torch.float32)


@_op("joint2offset")
def joint2offset(joint: Tensor, img: Tensor, kernel_size: float, feature_size: int, eps: float) -> Tensor:
    return ops.joint2offset(joint, img, kernel_size, feature_size, eps)


@joint2offset.register_fake
def _(joint, img, kernel_size, feature_size, eps):
    B = img.shape[0]
    J = joint.numel() // (3 * B)
    return img.new_empty(B, 4 * J, feature_size, feature_size, dtype=torch.float32)


# ------------------------------------------------------------------------------------------------ block kernels
@_op("repack_features")
def repack_features(img_feat: Tensor, img_feat_rgb: Tensor, weight_map: Tensor) -> Tuple[Tensor, Tensor]:
    """-> (hi [B,HW,288] bf16, lo): lo is the second plane of fp32 maps, EMPTY (numel 0) for bf16 maps."""
    hi, lo = ops.repack_features(img_feat, img_feat_rgb, weight_map)
    return hi, (lo if lo is not None else _empty(hi.device).to(torch.bfloat16))


@repack_features.register_fake
def _(img_feat, img_feat_rgb, weight_map):
    B = img_feat.shape[0]
    HW = img_feat.shape[2] * img_feat.shape[3] if img_feat.dim() == 4 else img_feat.shape[2]
    hi = img_feat.new_empty(B, HW, 288, dtype=torch.bfloat16)
    lo = img_feat.new_empty((0,) if img_feat.dtype == torch.bfloat16 else (B, HW, 288), dtype=torch.bfloat16)
    return hi, lo


@_op("split_map")
def split_map(x: Tensor) -> Tuple[Tensor, Tensor]:
    return ops.split_map(x)


@split_map.register_fake
def _(x):
    return x.new_empty(x.shape, dtype=torch.bfloat16), x.new_empty(x.shape, dtype=torch.bfloat16)


def _e_like(pcl):
    B, N = pcl.shape[:2]
    return torch.empty_strided((B, N, ops.E_ROW), ((N + 32) * ops.E_ROW, ops.E_ROW, 1), device=pcl.device, dtype=torch.int16)


@_op("point_embed")
def point_embed(feat_hi: Tensor, feat_lo: Tensor, idx32: Tensor, clos: Tensor, pcl: Tensor, joint: Tensor, wmat: Tensor, wvec: Tensor,
                kernel_size: float, fmt: int, order: Optional[Tensor] = None) -> Tuple[Tensor, Tensor, Tensor]:
    return ops.point_embed((feat_hi, feat_lo if feat_lo.numel() else None), idx32, clos, pcl, joint, wmat, wvec, kernel_size, order=order, fmt=fmt)


@point_embed.register_fake
def _(feat_hi, feat_lo, idx32, clos, pcl, joint, wmat, wvec, kernel_size, fmt, order=None):
    B, N = pcl.shape[:2]
    return _e_like(pcl), pcl.new_empty(B, N // 64, 128, 32, dtype=torch.float32), pcl.new_empty(B, N // 64, 2, 32, dtype=torch.float32)


@_op("point_embed_staged", mutates=("stage",))
def point_embed_staged(feat_hi: Tensor, feat_lo: Tensor, idx32: Tensor, clos: Tensor, pcl: Tensor, joint: Tensor, wmat: Tensor, wvec: Tensor,
                       kernel_size: float, fmt: int, stage: Tensor, read: bool, order: Optional[Tensor] = None) -> Tuple[Tensor, Tensor, Tensor]:
    """point_embed that also stores (read = False) or instead loads (read = True) the tiles' gathered operand images in `stage`
    (ops.point_embed_stage): the second block of KPFusion gathers the same taps as the first (model.py:297-306 per block)."""
    return ops.point_embed((feat_hi, feat_lo if feat_lo.numel() else None), idx32, clos, pcl, joint, wmat, wvec, kernel_size, order=order, fmt=fmt,
                           stage_in=stage if read else None, stage_out=None if read else stage)


@point_embed_staged.register_fake
def _(feat_hi, feat_lo, idx32, clos, pcl, joint, wmat, wvec, kernel_size, fmt, stage, read, order=None):
    B, N = pcl.shape[:2]
    return _e_like(pcl), pcl.new_empty(B, N // 64, 128, 32, dtype=torch.float32), pcl.new_empty(B, N // 64, 2, 32, dtype=torch.float32)


@_op("desa_fused", mutates=("e",))
def desa_fused(e: Tensor, part_acc: Tensor, part_ms: Tensor, pcl: Tensor, joint: Tensor, wmat: Tensor, wvec: Tensor, r0: float, r1: float,
               r2: float, nsample: int, fmt: int) -> Tuple[Tensor, Tensor]:
    return ops.desa_fused(e, part_acc, part_ms, pcl, joint, wmat, wvec, [r0, r1, r2], nsample, fmt=fmt)


@desa_fused.register_fake
def _(e, part_acc, part_ms, pcl, joint, wmat, wvec, r0, r1, r2, nsample, fmt):
    B, J = joint.shape[:2]
    return pcl.new_empty(B, 3, J, 128, dtype=torch.float32), pcl.new_empty(B, J, 128, dtype=torch.float32)


@_op("token_stack")
def token_stack(wmat: Tensor, wseq: Tensor, wvec: Tensor, cross: int, pre: int, D: int, L: int, F: int, Fc: int, J: int, fmt: int,
                want_tokens: bool, x: Optional[Tensor] = None, y: Optional[Tensor] = None, r3d: Optional[Tensor] = None,
                desa: Optional[Tensor] = None, jf: Optional[Tensor] = None, peer_ptrs: Optional[Tensor] = None,
                xstep: Optional[Tensor] = None, row0: int = 0, rows_total: int = 0) -> Tuple[Tensor, Tensor]:
    """-> (tokens [B,J,128] or EMPTY, pred [B,J,3] or EMPTY); cross-only programs: tokens = the layer output [B,J,128].
    peer_ptrs / xstep / row0 / rows_total: the fused exchange step (writes into the ranks' symmetric buffers, which are not arguments)."""
    pk = ops.TokenProgram(wmat, wseq, wvec, cross, pre, D, L, F, Fc, J, fmt)
    xch = (peer_ptrs, xstep, row0, rows_total) if peer_ptrs is not None else None
    ref = x if x is not None else desa
    if L == 0 and cross:   # cross layer alone: [B,J,128] through the strided output
        out = torch.empty(ref.shape[0], J, 128, device=ref.device, dtype=torch.float32)
        ops.token_stack(pk, x=x, y=y, out_jc=out, out_jc_c0=0)
        return out, _empty(ref.device)
    tokens, pred, _ = ops.token_stack(pk, x=x, y=y, r3d=r3d, desa=desa, jf=jf, want_tokens=want_tokens, exchange=xch)
    return (tokens if tokens is not None else _empty(ref.device)), (pred if pred is not None else _empty(ref.device))


@token_stack.register_fake
def _(wmat, wseq, wvec, cross, pre, D, L, F, Fc, J, fmt, want_tokens, x=None, y=None, r3d=None, desa=None, jf=None, peer_ptrs=None, xstep=None,
      row0=0, rows_total=0):
    ref = x if x is not None else desa
    B = ref.shape[0]
    has_tok = (L == 0 and cross) or (want_tokens and (L > 0 or (pre and not cross)))
    tok = ref.new_empty((B, J, 128) if has_tok else (0,), dtype=torch.float32)
    pred = ref.new_empty((B, J, 3) if L > 0 else (0,), dtype=torch.float32)
    return tok, pred


@_op("spatial_aggregate_tc")
def spatial_aggregate_tc(feat: Tensor, feat_lo: Tensor, joints: Tensor, img: Tensor, center: Tensor, M: Tensor, cube: Tensor, cam: Tensor,
                         wa_packed: Tensor, ba: Tensor, weight_dis: Tensor, fc_w: Tensor, fc_b: Tensor, img_size: float, flip: float,
                         hm_std: float, hm_sigma: float, gamma: float, fmt: int, prev: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    return ops.spatial_aggregate_tc((feat, feat_lo if feat_lo.numel() else None), joints, img, center, M, cube, cam, wa_packed, ba, weight_dis,
                                    fc_w, fc_b, prev=prev, img_size=img_size, flip=flip, hm_std=hm_std, hm_sigma=hm_sigma, gamma=gamma, fmt=fmt)


@spatial_aggregate_tc.register_fake
def _(feat, feat_lo, joints, img, center, M, cube, cam, wa_packed, ba, weight_dis, fc_w, fc_b, img_size, flip, hm_std, hm_sigma, gamma, fmt,
      prev=None):
    B, C, fs, _ = feat.shape
    J = joints.shape[1]
    return feat.new_empty(B, J, fs, fs, dtype=torch.float32), feat.new_empty(B, J, C, dtype=torch.float32)


@_op("cross_decoder_layer")
def cross_decoder_layer(anchor: Tensor, tokens: Tensor, wpack: Tensor, heads: int, ffn: int) -> Tensor:
    return ops.cross_decoder_layer(anchor, tokens, wpack, heads, ffn)


@cross_decoder_layer.register_fake
def _(anchor, tokens, wpack, heads, ffn):
    B, J, C = anchor.shape
    return anchor.new_empty(B, C, J, dtype=torch.float32)


# ------------------------------------------------------------------------------------------------ 8b: general-shape attention (off the live path)
@_op("linear_rows")
def linear_rows(x: Tensor, weight: Tensor, bias: Optional[Tensor], pos: Optional[Tensor], pos_index: Optional[Tensor], scale: float,
                relu: bool, out_layout: int) -> Tensor:
    return ops.linear_rows(x, weight, bias, pos=pos, pos_index=pos_index, scale=scale, relu=relu, out_layout=out_layout)


@linear_rows.register_fake
def _(x, weight, bias, pos, pos_index, scale, relu, out_layout):
    B, P, O = x.shape[0], x.shape[1], weight.shape[0]
    shape = (B, O, P) if out_layout == ops.ROWS_BOP else (P, B, O) if out_layout == ops.ROWS_PBO else (B, P, O)
    return x.new_empty(shape, dtype=torch.float32)


@_op("mha_core")
def mha_core(q: Tensor, k: Tensor, v: Tensor, num_heads: int, attn_mask: Optional[Tensor], key_padding_mask: Optional[Tensor],
             need_weights: bool) -> Tuple[Tensor, Tensor]:
    out, w = ops.mha_core(q, k, v, num_heads, attn_mask=attn_mask, key_padding_mask=key_padding_mask, need_weights=need_weights)
    return out, (w if w is not None else _empty(q.device))


@mha_core.register_fake
def _(q, k, v, num_heads, attn_mask, key_padding_mask, need_weights):
    B, Pq, C = q.shape
    return q.new_empty(B, Pq, C, dtype=torch.float32), (q.new_empty(B, Pq, k.shape[1], dtype=torch.float32) if need_weights
                                                         else q.new_empty(0, dtype=torch.float32))


@_op("add_layernorm_rows")
def add_layernorm_rows(x: Tensor, r: Optional[Tensor], gamma: Tensor, beta: Tensor, eps: float, channel_major: bool) -> Tensor:
    return ops.add_layernorm_rows(x, r, gamma, beta, eps, channel_major)


@add_layernorm_rows.register_fake
def _(x, r, gamma, beta, eps, channel_major):
    B, P, C = x.shape
    return x.new_empty((B, C, P) if channel_major else (B, P, C), dtype=torch.float32)


@_op("sine_posembed")
def sine_posembed(dim_t: Tensor, B: int, H: int, W: int, mask: Optional[Tensor], normalize: bool, scale: float) -> Tensor:
    return ops.sine_posembed(dim_t, B, H, W, mask=mask, normalize=normalize, scale=scale)


@sine_posembed.register_fake
def _(dim_t, B, H, W, mask, normalize, scale):
    return dim_t.new_empty(B, 2 * dim_t.numel(), H, W, dtype=torch.float32)


@_op("ball_query")
def ball_query(xyz: Tensor, centers: Tensor, radius: float, nsample: int) -> Tensor:
    return ops.ball_query(xyz, centers, radius, nsample)


@ball_query.register_fake
def _(xyz, centers, radius, nsample):
    return xyz.new_empty(xyz.shape[0], centers.shape[1], nsample, dtype=torch.int32)


# ------------------------------------------------------------------------------------------------ fusion-layer modules (K7)
@_op("rgbd_fusion")
def rgbd_fusion(rgb: Tensor, depth: Tensor, gate_w: Tensor, gate_b: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    ro, do, mg, _ = ops.rgbd_fusion(rgb, depth, gate_w, gate_b)
    return ro, do, mg


@rgbd_fusion.register_fake
def _(rgb, depth, gate_w, gate_b):
    dt = rgb.dtype if rgb.dtype in (torch.float32, torch.bfloat16) else torch.float32
    mk = lambda: rgb.new_empty(rgb.shape, dtype=dt)
    return mk(), mk(), mk()


@_op("ac_fusion")
def ac_fusion(rgb: Tensor, depth: Tensor, w_rgb: Tensor, b_rgb: Tensor, w_depth: Tensor, b_depth: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    return ops.ac_fusion(rgb, depth, w_rgb, b_rgb, w_depth, b_depth)


@ac_fusion.register_fake
def _(rgb, depth, w_rgb, b_rgb, w_depth, b_depth):
    dt = rgb.dtype if rgb.dtype in (torch.float32, torch.bfloat16) else torch.float32
    mk = lambda: rgb.new_empty(rgb.shape, dtype=dt)
    return mk(), mk(), mk()


@_op("fsp")
def fsp(guide: Tensor, main: Tensor, w0: Tensor, b0: Tensor, w2: Tensor, b2: Tensor) -> Tensor:
    return ops.fsp(guide, main, w0, b0, w2, b2)


@fsp.register_fake
def _(guide, main, w0, b0, w2, b2):
    dt = guide.dtype if guide.dtype in (torch.float32, torch.bfloat16) else torch.float32
    return main.new_empty(main.shape, dtype=dt)


@_op("eval_errors")
def eval_errors(pred: Tensor, gt: Tensor, cube: Tensor) -> Tuple[Tensor, Tensor]:
    return ops.eval_errors(pred, gt, cube, aligned=True)


@eval_errors.register_fake
def _(pred, gt, cube):
    B, J = pred.shape[:2]
    return pred.new_empty(B, J, dtype=torch.float32), pred.new_empty(B, J, dtype=torch.float32)


# ------------------------------------------------------------------------------------------------ 8f-3 frame front end
# frame_index: None (box b reads frame b) or a [B] int32 tensor on the device (out-of-range boxes give NaN, include/kpf_b200.h)
@_op("center_from_bbox")
def center_from_bbox(depth: Tensor, bbox: Tensor, upper: int, lower: int, frame_index: Optional[Tensor] = None) -> Tensor:
    return ops.center_from_bbox(depth, bbox, upper, lower, frame_index=frame_index)


@center_from_bbox.register_fake
def _(depth, bbox, upper, lower, frame_index=None):
    return depth.new_empty(bbox.shape[0], 3, dtype=torch.float64)


@_op("crop_depth")
def crop_depth(depth: Tensor, center: Tensor, cube: Tensor, cam: Tensor, dsize: int, frame_index: Optional[Tensor] = None) -> Tuple[Tensor, Tensor, Tensor]:
    """-> (img [B,1,dsize,dsize], M [B,3,3], com3d [B,3]) for center [B,3], cube [B,3] f32, cam [B,4] or [4] f64."""
    img, M, com3d, _ = ops.crop_depth(depth, center, cube, cam, dsize, frame_index=frame_index)
    return img, M, com3d


@crop_depth.register_fake
def _(depth, center, cube, cam, dsize, frame_index=None):
    B = center.shape[0]
    f = lambda *shape: depth.new_empty(shape, dtype=torch.float32)
    return f(B, 1, dsize, dsize), f(B, 3, 3), f(B, 3)


@_op("crop_rgb")
def crop_rgb(rgb: Tensor, center: Tensor, cube: Tensor, cam: Tensor, dsize: int, frame_index: Optional[Tensor] = None) -> Tensor:
    return ops.crop_rgb(rgb, center, cube, cam, dsize, frame_index=frame_index)


@crop_rgb.register_fake
def _(rgb, center, cube, cam, dsize, frame_index=None):
    return rgb.new_empty(center.shape[0], 3, dsize, dsize, dtype=torch.float32)


@_op("joints_to_frame")
def joints_to_frame(joints: Tensor, center: Tensor, cube: Tensor, cam: Tensor, flip: float) -> Tuple[Tensor, Tensor]:
    """-> (uvd_frame [B,P,3]: frame pixels and depth mm, xyz_cam [B,P,3]: camera-space mm)."""
    return ops.joints_to_frame(joints, center, cube, cam, flip)


@joints_to_frame.register_fake
def _(joints, center, cube, cam, flip):
    return joints.new_empty(joints.shape, dtype=torch.float32), joints.new_empty(joints.shape, dtype=torch.float32)


def run_token_program(pk, x=None, y=None, r3d=None, desa=None, jf=None, want_tokens=True, exchange=None):
    """TokenProgram (plain Python holder of three tensors + ints) -> the custom op.  Returns (tokens | None, pred | None).
    exchange: a runtime.PeerExchange (the fused exchange step) or None."""
    xa = (exchange.peer_ptrs, exchange.xstep, exchange.row0, exchange.rows_total) if exchange is not None else (None, None, 0, 0)
    tok, pred = torch.ops.kpf.token_stack(pk.wmat, pk.wseq, pk.wvec, pk.cross, pk.pre, pk.D, pk.L, pk.F, pk.Fc, pk.J, pk.fmt, want_tokens,
                                          x, y, r3d, desa, jf, *xa)
    return (tok if tok.numel() else None), (pred if pred.numel() else None)


REGISTERED = sorted(n for n, v in list(globals().items()) if isinstance(v, torch.library.CustomOpDef))
