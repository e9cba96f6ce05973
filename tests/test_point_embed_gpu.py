"""GPU: fused point stage (repack + gather + embeddings + softmax-aggregation partials) and DESA on split-precision tcgen05 GEMMs
vs the fp32 oracle: fp32-class bars (RMS relative <= TOL, two orders inside north_star's 1e-3), bit-exact ball-query indices."""
import numpy as np
import pytest
import torch

from keypointfusion_b200.utils import synth
from oracle import kpf_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"


def rms_rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).norm() / b.norm())


def _tol():
    from keypointfusion_b200 import ops
    return 2e-5 if ops.SPLIT_FMT == ops.FMT_F16 else 3e-4   # fp16 planes: 22 bits ; bf16 planes: 16 bits


def worst_rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).abs().max() / b.abs().max())


def test_repack(golden_inputs):
    from keypointfusion_b200 import ops
    i = golden_inputs
    for dt in (torch.float32, torch.bfloat16):
        out, lo = ops.repack_features(i["img_feat"].to(DEV, dt), i["img_feat_rgb"].to(DEV, dt), i["img_offset"][:, 84:].to(DEV, dt))
        ref = torch.cat([i["img_feat"], i["img_feat_rgb"], i["img_offset"][:, 84:], torch.zeros(2, 11, 32, 32)], 1)
        ref = ref.reshape(2, 288, 1024).permute(0, 2, 1).to(dt)
        assert torch.equal(out.cpu(), ref.bfloat16())
        if dt == torch.float32:   # fp32 maps: a second plane carries x - bf16(x), so hi + lo is x to 2^-16
            assert torch.equal(lo.cpu(), (ref - ref.bfloat16().float()).bfloat16())
            assert float(((out.float() + lo.float()).cpu() - ref).abs().max()) <= 2.0 ** -15 * float(ref.abs().max())
        else:
            assert lo is None


@pytest.mark.parametrize("B,maps", [(2, "bf16"), (5, "bf16"), (3, "fp32")])
def test_point_embed(golden, golden_inputs, path_params, B, maps):
    from keypointfusion_b200 import ops
    from keypointfusion_b200.model.model import Block_KPFusion
    inp = synth.make_inputs(B, 128, 21, 128, seed=50 + B, bf16_round=maps == "bf16")
    mdt = torch.bfloat16 if maps == "bf16" else torch.float32
    g = [inp[k].numpy() for k in ("center", "M", "cube", "cam")]
    c = {k: v.to(DEV) for k, v in inp.items()}
    pcl, _ = ops.getpcl(c["img"], c["center"], c["cube"], c["M"], c["cam"], seed=2)
    close, _, idx = ops.img2pcl_index(pcl, c["img"], c["center"], c["M"], c["cube"], c["cam"], 128, 4, fs=32, want_i64=False, want_i32=True)
    joint = torch.from_numpy(np.random.RandomState(B).uniform(-0.6, 0.6, (B, 21, 3)).astype(np.float32))
    blk = Block_KPFusion(21)
    blk.load_state_dict({k[len("block1."):]: v for k, v in path_params.items() if k.startswith("block1.")})
    blk = blk.to(DEV).eval()
    k = blk.kc()
    featT = ops.repack_features(c["img_feat"].to(mdt), c["img_feat_rgb"].to(mdt), c["img_offset"][:, 84:].to(mdt))
    e16, acc, ms = ops.point_embed(featT, idx, close, pcl, joint.to(DEV), k["pe_wmat"], k["pe_wvec"], 0.8)
    e = ops.e_to_float(e16)
    agg = ops.combine_point_partials(acc, ms, 21)
    # oracle on the same maps (bf16 maps are exact in one plane; fp32 maps enter as two bf16 planes = 16 mantissa bits)
    p = path_params
    pc, ix, cl = pcl.cpu(), idx.cpu().long(), close.cpu()
    off = O.pcl_joint2offset(joint, pc, 0.8)
    pf, pr = O.gather_taps(inp["img_feat"], ix, cl), O.gather_taps(inp["img_feat_rgb"], ix, cl)
    pw = O.gather_taps(inp["img_offset"][:, 84:], ix, cl)
    ee = torch.relu(O.conv_bn(p, "block1.pcl_feat_emb.", pf) + O.conv_bn(p, "block1.pcl_xyz_emb.", pc) +
                    O.conv_bn(p, "block1.pcl_pose_emb.", torch.cat([pw, off], -1)))
    ee = torch.relu(ee + O.conv_bn(p, "block1.pcl_feat_emb_RGB.", pr))
    ragg = torch.softmax(pw.permute(0, 2, 1), -1) @ ee
    tol = _tol() if maps == "bf16" else 3e-5
    print(f"[point stage] maps {maps}: e rms rel {rms_rel(e, ee):.2e} worst {worst_rel(e, ee):.2e}; aggregation rms rel {rms_rel(agg, ragg):.2e}")
    assert rms_rel(e, ee) < tol and worst_rel(e, ee) < 10 * tol, (rms_rel(e, ee), worst_rel(e, ee))
    assert rms_rel(agg, ragg) < tol and worst_rel(agg, ragg) < 10 * tol, rms_rel(agg, ragg)
    # spatial processing order (scheduling aid): K2 and the point features are bit-identical, the aggregation only regroups
    order = ops.spatial_order(pcl, c["center"], c["M"], c["cube"], c["cam"], 128, 32)
    assert torch.equal(torch.sort(order.long(), dim=1)[0].cpu(), torch.arange(pcl.shape[1]).expand(B, -1))
    close2, _, idx2 = ops.img2pcl_index(pcl, c["img"], c["center"], c["M"], c["cube"], c["cam"], 128, 4, fs=32, want_i64=False, want_i32=True,
                                        order=order)
    assert torch.equal(idx2, idx) and torch.equal(close2, close)
    e2, acc2, ms2 = ops.point_embed(featT, idx, close, pcl, joint.to(DEV), k["pe_wmat"], k["pe_wvec"], 0.8, order=order)
    assert torch.equal(e2, e16)
    agg2 = ops.combine_point_partials(acc2, ms2, 21)
    assert rms_rel(agg2, ragg) < tol and rms_rel(agg2, agg) < tol, (rms_rel(agg2, ragg), rms_rel(agg2, agg))


def _desa_setup(path_params, B, seed):
    from keypointfusion_b200 import ops
    from keypointfusion_b200.model.model import Block_KPFusion
    inp = synth.make_inputs(B, 128, 21, 128, seed=seed, bf16_round=True)
    c = {k: v.to(DEV) for k, v in inp.items()}
    pcl, _ = ops.getpcl(c["img"], c["center"], c["cube"], c["M"], c["cam"], seed=2)
    close, _, idx = ops.img2pcl_index(pcl, c["img"], c["center"], c["M"], c["cube"], c["cam"], 128, 4, fs=32, want_i64=False, want_i32=True)
    blk = Block_KPFusion(21)
    blk.load_state_dict({k[len("block1."):]: v for k, v in path_params.items() if k.startswith("block1.")})
    blk = blk.to(DEV).eval()
    return inp, c, pcl, close, idx, blk


def _joint_sets(pcl, which):
    """Centre placements that exercise the ball query's branches (pointnet2_ops semantics, model.py:158, :174)."""
    B = pcl.shape[0]
    if which == "dense":      # on the cloud: every ball well populated (> nsample hits at the large radii)
        return pcl[:, ::48][:, :21].contiguous() + 0.01
    if which == "sparse":     # just off the cloud's rim and far away: < nsample hits (padding with the first hit), and balls that
        j = pcl[:, ::48][:, :21].contiguous().clone()     # contain nothing but the centre itself
        j[:, ::3, 2] += 0.35
        j[:, 1::3, :2] += 0.3
        j[:, 20] = torch.tensor([3.0, 3.0, 3.0], device=pcl.device)
        return j
    # "edge": centres at EXACTLY radius distance (d2 == r2 must be excluded: strict <) from a cloud point along x, for each scale
    j = pcl[:, 100:121].contiguous().clone()
    for k, r in enumerate((0.1, 0.2, 0.4)):
        j[:, k::3, 0] = pcl[:, 100 + k:121:3, 0] + r
    return j


@pytest.mark.parametrize("which", ["dense", "sparse", "edge"])
def test_ball_query_indices_exact(path_params, which):
    """kpf_ball_query (stand-alone) AND the fused prep kernel's indices == the oracle's ball query, bit for bit, incl. sparse balls
    (< nsample hits -> padded with the first hit), saturated balls (> nsample hits -> the first nsample in index order), the
    d2 == r2 boundary and centres far from the cloud.  The fused kernel's indices are read back from its scratch workspace."""
    from keypointfusion_b200 import ops
    B = 3
    inp, c, pcl, close, idx, blk = _desa_setup(path_params, B, 81)
    joint = _joint_sets(pcl, which)
    N, J, NS = pcl.shape[1], 21, 64
    xyz = torch.cat([pcl, joint], 1).contiguous()
    counts = []
    for r in (0.1, 0.2, 0.4):
        got = ops.ball_query(xyz, joint, r, NS).cpu().numpy()
        ref, cnt = O.ball_query(xyz.cpu().numpy(), joint.cpu().numpy(), r, NS, return_counts=True)
        assert np.array_equal(got, ref), (which, r)
        counts.append(cnt)
    counts = np.stack(counts)
    if which == "dense":
        assert (counts[2] > NS).any()
    if which == "sparse":
        assert (counts[0] < NS).any() and (counts == 1).any()     # a ball holding only its own centre
    # fused path: same indices out of desa_prep_kernel (u16, scale-major per sample)
    k = blk.kc()
    featT = ops.repack_features(c["img_feat"].bfloat16(), c["img_feat_rgb"].bfloat16(), c["img_offset"][:, 84:].bfloat16())
    e, acc, ms = ops.point_embed(featT, idx, close, pcl, joint, k["pe_wmat"], k["pe_wvec"], 0.8)
    scratch = {}
    ops.desa_fused(e, acc, ms, pcl, joint, k["ds_wmat"], k["ds_wvec"], blk.FA.radius, NS, keep_scratch=scratch)
    torch.cuda.synchronize()
    off = B * 3 * J * 128 * 4 + B * (N + 32) * 16
    fused = scratch["buf"][off:off + B * 3 * J * NS * 2].view(torch.int16).cpu().numpy().astype(np.uint16).reshape(B, 3, J, NS)
    for s_, r in enumerate((0.1, 0.2, 0.4)):
        ref = O.ball_query(xyz.cpu().numpy(), joint.cpu().numpy(), r, NS)
        assert np.array_equal(fused[:, s_].astype(np.int64), ref.astype(np.int64)), (which, r)
    # ... and the widest ball per (sample, scale), which sets how many rows per joint the tile kernel groups (16 / 32 / nsample)
    off_gw = off + B * 3 * J * NS * 2
    gw = scratch["buf"][off_gw:off_gw + B * 3 * 4].view(torch.int32).cpu().numpy().reshape(B, 3)
    assert np.array_equal(gw, np.minimum(counts, NS).reshape(3, B, J).max(-1).T), (which, gw)
    if which == "sparse":
        assert gw[:, 0].max() <= 16      # the narrow-group path of the tile kernel is what test_desa_fused[sparse] runs


@pytest.mark.parametrize("B,which,radii", [(2, "dense", None), (3, "dense", None), (2, "sparse", None), (2, "edge", None),
                                           (3, "dense", (0.06, 0.12, 0.15)), (2, "sparse", (0.15, 0.3, 0.6))])
def test_desa_fused(path_params, B, which, radii):
    """point stage -> DESA kernel vs the oracle's joint embeddings + DESA (same ball-query membership: centres are inputs).
    The radii variants move the scales between the tile kernel's group widths (16 / 32 / nsample rows per joint)."""
    from keypointfusion_b200 import ops
    import torch.nn.functional as F
    inp, c, pcl, close, idx, blk = _desa_setup(path_params, B, 70 + B)
    joint = _joint_sets(pcl, which)
    if radii is not None:
        blk.FA.radius = list(radii)
    k = blk.kc()
    featT = ops.repack_features(c["img_feat"].bfloat16(), c["img_feat_rgb"].bfloat16(), c["img_offset"][:, 84:].bfloat16())
    e, acc, ms = ops.point_embed(featT, idx, close, pcl, joint, k["pe_wmat"], k["pe_wvec"], 0.8)
    part, jf = ops.desa_fused(e, acc, ms, pcl, joint, k["ds_wmat"], k["ds_wvec"], blk.FA.radius, blk.FA.S[0])
    # narrow groups (a scale whose widest ball holds <= 16 / 32 points is tiled 16 / 32 rows per joint) leave every bit unchanged.
    # The group width is chosen per launch, from the widest ball of any sample: a launch with one extra sample whose points and
    # joints all sit inside one 0.01 cube (every ball of every scale saturated) groups nsample rows per joint for every sample.
    N, NS, S = pcl.shape[1], blk.FA.S[0], len(blk.FA.radius)
    gen = torch.Generator(device=DEV).manual_seed(B)
    tight = lambda n: pcl[:1, :1] + 0.01 * torch.rand(1, n, 3, device=DEV, generator=gen)
    scratch = {}
    part_w, jf_w = ops.desa_fused(torch.cat([e, e[:1]]), torch.cat([acc, acc[:1]]), torch.cat([ms, ms[:1]]), torch.cat([pcl, tight(N)]),
                                  torch.cat([joint, tight(21)]), k["ds_wmat"], k["ds_wvec"], blk.FA.radius, NS, keep_scratch=scratch)
    torch.cuda.synchronize()
    off_gw = (B + 1) * (S * 21 * 128 * 4 + (N + 32) * 16 + S * 21 * NS * 2)
    gw = scratch["buf"][off_gw:off_gw + (B + 1) * S * 4].view(torch.int32).cpu().reshape(B + 1, S)
    assert (gw[B] > 32).all(), gw     # the extra sample widens every scale to nsample rows per joint
    assert torch.equal(part, part_w[:B]) and torch.equal(jf, jf_w[:B])
    fu = blk.FA.kc()["fusion"]
    out = F.relu(F.linear(torch.cat([part.permute(0, 2, 1, 3).reshape(B, 21, -1), jf], -1), *fu))
    # oracle
    p = path_params
    pc, ix, cl, jt = pcl.cpu(), idx.cpu().long(), close.cpu(), joint.cpu()
    off = O.pcl_joint2offset(jt, pc, 0.8)
    pf, pr = O.gather_taps(inp["img_feat"], ix, cl), O.gather_taps(inp["img_feat_rgb"], ix, cl)
    pw = O.gather_taps(inp["img_offset"][:, 84:], ix, cl)
    ee = torch.relu(O.conv_bn(p, "block1.pcl_feat_emb.", pf) + O.conv_bn(p, "block1.pcl_xyz_emb.", pc) +
                    O.conv_bn(p, "block1.pcl_pose_emb.", torch.cat([pw, off], -1)))
    ee = torch.relu(ee + O.conv_bn(p, "block1.pcl_feat_emb_RGB.", pr))
    rjf = torch.relu(O.conv_bn(p, "block1.joint_feat_emb.", torch.softmax(pw.permute(0, 2, 1), -1) @ ee) + O.conv_bn(p, "block1.joint_xyz_emb.", jt))
    rout = O.desa(p, "block1.FA.", ee, rjf, pc, jt, radius=tuple(blk.FA.radius))
    print(f"[desa {which}] jf rms rel {rms_rel(jf, rjf):.2e}; desa output rms rel {rms_rel(out, rout):.2e} worst {worst_rel(out, rout):.2e}")
    assert rms_rel(jf, rjf) < _tol(), rms_rel(jf, rjf)
    assert rms_rel(out, rout) < _tol() and worst_rel(out, rout) < 10 * _tol(), rms_rel(out, rout)
    # the stand-alone drop-in module (model.py:166-204 signature) runs the same kernels with the joint features given
    mod = blk.FA(ee.to(DEV), rjf.to(DEV), pcl, joint)
    assert rms_rel(mod, rout) < _tol(), rms_rel(mod, rout)


@pytest.mark.parametrize("maps", ["bf16", "fp32"])
@pytest.mark.parametrize("B", [2, 5, 64])
def test_point_embed_staged_tiles(path_params, B, maps):
    """Block 2 of KPFusion gathers the same taps of the same maps as block 1 (model.py:297-306 runs per block).  A launch that
    stores its gathered operand tiles (stage_out) followed by one that loads them (stage_in: other joints, the other block's
    weights, no gather) must be BIT-identical to gathering again -- with and without the spatial processing order."""
    from keypointfusion_b200 import ops
    inp, c, pcl, close, idx, blk = _desa_setup(path_params, B, 90 + B)
    from keypointfusion_b200.model.model import KPFusion
    net = KPFusion(joint_num=21)
    net.load_state_dict(path_params)
    net = net.to(DEV).eval()
    k1, k2 = net.block1.kc(), net.block2.kc()
    cast = (lambda t: t.bfloat16()) if maps == "bf16" else (lambda t: t.float())
    featT = ops.repack_features(cast(c["img_feat"]), cast(c["img_feat_rgb"]), cast(c["img_offset"][:, 84:]))
    j1, j2 = _joint_sets(pcl, "dense"), _joint_sets(pcl, "sparse")
    for order in (None, ops.spatial_order(pcl, c["center"], c["M"], c["cube"], c["cam"], 128, 32)):
        stage = ops.point_embed_stage(B, pcl.shape[1], pcl.device)
        stage.fill_(0x5a)
        a = ops.point_embed(featT, idx, close, pcl, j1, k1["pe_wmat"], k1["pe_wvec"], 0.8, order=order, stage_out=stage)
        ref1 = ops.point_embed(featT, idx, close, pcl, j1, k1["pe_wmat"], k1["pe_wvec"], 0.8, order=order)
        for x, y in zip(a, ref1):
            assert torch.equal(x, y)                      # storing the tiles does not change the launch's own results
        got = ops.point_embed(featT, idx, close, pcl, j2, k2["pe_wmat"], k2["pe_wvec"], 0.8, order=order, stage_in=stage)
        ref2 = ops.point_embed(featT, idx, close, pcl, j2, k2["pe_wmat"], k2["pe_wvec"], 0.8, order=order)
        for x, y in zip(got, ref2):
            assert torch.equal(x, y)
