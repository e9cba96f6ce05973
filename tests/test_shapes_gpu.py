"""GPU: the fusion-path kernels across the shapes they accept, not only the benchmark's (21 joints, 1024 points, nsample 64, three
DESA scales): joint counts 1 .. 32 (padded tokens, the point stage's column layout, half-empty joint tiles), point counts 64 .. 2048,
every DESA group width and scale count, every K5 split and both K4a variants, each vs the fp32 oracle.

Bars as in the other GPU tests: split-precision outputs RMS relative < _tol() and worst entry < 10 x that of max|ref|; K4a and
CUDA-core fp32 results elementwise; indices bit-exact.  On top, every comparison bounds the worst entry of each (sample, joint) row
by the same worst-entry bar, relative to that SAMPLE's max|ref|: a defect confined to the last joint or the last sample cannot hide
in a figure taken over the whole batch."""
import functools
import itertools

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from keypointfusion_b200.utils import synth
from oracle import kpf_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _tol():
    from keypointfusion_b200 import ops
    return 2e-5 if ops.SPLIT_FMT == ops.FMT_F16 else 3e-4   # fp16 planes: 22 bits ; bf16 planes: 16 bits


def check(a, ref, rms, worst, what):
    """a, ref [B, rows, ...]: RMS relative error < rms; worst entry < worst of max|ref|; worst entry of every (sample, row) < worst
    of that sample's max|ref|."""
    a, ref = a.detach().double().cpu(), ref.detach().double().cpu()
    assert a.shape == ref.shape, (what, a.shape, ref.shape)
    B, R = ref.shape[:2]
    d = (a - ref).abs()
    r = float((a - ref).norm() / ref.norm())
    w = float(d.max() / ref.abs().max())
    scale = ref.reshape(B, -1).abs().amax(-1).clamp_min(1e-30)
    per_row = d.reshape(B, R, -1).amax(-1) / scale[:, None]
    b, j = divmod(int(per_row.argmax()), R)
    print(f"[{what}] rms rel {r:.2e}, worst {w:.2e}, worst row {float(per_row.max()):.2e} at (sample {b}, row {j})")
    assert r < rms and w < worst and float(per_row.max()) < worst, (what, r, w, float(per_row.max()), (b, j))


def close(a, ref, rtol, atol, row_bar, what):
    """elementwise |a - ref| <= atol + rtol |ref|, and every (sample, row)'s worst entry < row_bar of the sample's max|ref|."""
    a, ref = a.detach().double().cpu(), ref.detach().double().cpu()
    assert a.shape == ref.shape, (what, a.shape, ref.shape)
    d = (a - ref).abs()
    assert bool((d <= atol + rtol * ref.abs()).all()), (what, float(d.max()))
    B, R = ref.shape[:2]
    per_row = d.reshape(B, R, -1).amax(-1) / ref.reshape(B, -1).abs().amax(-1, keepdim=True).clamp_min(1e-30)
    assert float(per_row.max()) < row_bar, (what, float(per_row.max()), divmod(int(per_row.argmax()), R))


def cu(x):
    return (x if torch.is_tensor(x) else torch.from_numpy(np.asarray(x))).to(DEV)


def geo(inp):
    return [inp[k].numpy() for k in ("center", "M", "cube", "cam")]


@functools.lru_cache(maxsize=None)
def block(J):
    """Block_KPFusion(joint_num=J) with seeded parameters on the GPU, and a CPU copy of its state_dict for the oracle."""
    from keypointfusion_b200.model.model import Block_KPFusion
    blk = Block_KPFusion(joint_num=J)
    synth.fill_state_dict(blk, seed=J)
    sd = {k: v.clone() for k, v in blk.state_dict().items()}
    return blk.to(DEV).eval(), sd


def joint_set(pcl, J, which):
    """J centres on the cloud, spread over its point order (dense: well-populated balls), or pushed off the rim with the last one far
    away (sparse: balls of fewer than nsample hits, one holding nothing but its own centre)."""
    N = pcl.shape[1]
    j = pcl[:, (torch.arange(J) * N) // J].clone()
    if which == "dense":
        return j + 0.01
    j[:, ::3, 2] += 0.35
    j[:, 1::3, :2] += 0.3
    j[:, J - 1] = 3.0
    return j.contiguous()


# ------------------------------------------------------------------------------------------------ token stack
@functools.lru_cache(maxsize=None)
def token_program(J, program):
    from keypointfusion_b200 import ops
    blk, sd = block(J)
    if program == "cross":
        return ops.pack_token_program(J, cross=(sd, "crossTR.decoder.3.")).to(DEV)
    if program == "fusion_enc":
        return ops.pack_token_program(J, enc=(sd, "init_TR."), fusion=tuple(t.cpu() for t in blk.FA.kc()["fusion"])).to(DEV)
    return ops.pack_token_program(J, enc=(sd, program + ".")).to(DEV)


@pytest.mark.parametrize("B", [1, 5, 64])
@pytest.mark.parametrize("J", [1, 2, 8, 14, 21, 32])
@pytest.mark.parametrize("program", ["init_TR", "final_TR", "cross", "fusion_enc"])
def test_token_stack_joint_counts(program, J, B):
    """Padded tokens (J < 32) must not enter any softmax, LayerNorm or output: init_TR (D = 128) and final_TR (D = 131) encoders, the
    decoder cross layer of updatedDecoder(joint_num=J), and the DESA fusion conv + init_TR program."""
    from keypointfusion_b200 import ops
    blk, sd = block(J)
    pk = token_program(J, program)
    tol = _tol()
    rs = np.random.RandomState(1000 * J + B)
    randn = lambda *shape: torch.from_numpy(rs.standard_normal(shape).astype(np.float32))
    if program == "cross":
        a, k = randn(B, J, 128), randn(B, J, 128)
        jc = torch.zeros(B, J, 131, device=DEV)
        out = ops.token_stack(pk, x=a.to(DEV), y=k.to(DEV), out_jc=jc, out_jc_c0=3, want_cj=True)[2]
        check(out.permute(0, 2, 1), O.updated_decoder(sd, "crossTR.", a, k).permute(0, 2, 1), tol, 10 * tol, f"cross J={J} B={B}")
        assert torch.equal(jc[:, :, 3:], out.permute(0, 2, 1)) and not jc[:, :, :3].any()
        return
    if program == "fusion_enc":
        part, jf = randn(B, 3, J, 128).abs(), randn(B, J, 128).abs()
        tok, pred, _ = ops.token_stack(pk, desa=part.to(DEV), jf=jf.to(DEV))
        Wfu, bfu = (t.cpu() for t in blk.FA.kc()["fusion"])
        x = torch.relu(F.linear(torch.cat([part.permute(0, 2, 1, 3).reshape(B, J, -1), jf], -1), Wfu, bfu))
        prefix = "init_TR."
    else:
        x = randn(B, J, pk.D)
        if pk.D == 131:
            x[:, :, :3] *= 0.3
        tok, pred, _ = ops.token_stack(pk, x=x.to(DEV))
        prefix = program + "."
    rtok, rpred = O.kp_interaction_tr(sd, prefix, x)
    check(tok, rtok, tol, 10 * tol, f"{program} tokens J={J} B={B}")
    check(pred, rpred, tol, 10 * tol, f"{program} pred J={J} B={B}")


@pytest.mark.parametrize("J", [1, 32])
def test_cuda_core_cross_layer_joint_counts(J):
    from keypointfusion_b200 import ops
    _, sd = block(J)
    B = 5
    rs = np.random.RandomState(J)
    a = torch.from_numpy(rs.standard_normal((B, J, 128)).astype(np.float32))
    k = torch.from_numpy(rs.standard_normal((B, J, 128)).astype(np.float32))
    out = ops.cross_decoder_layer(cu(a), cu(k), cu(ops.pack_decoder_layer(sd, "crossTR.decoder.3.", J, 128)), heads=4, ffn=128)
    ref = O.updated_decoder(sd, "crossTR.", a, k)
    close(out.permute(0, 2, 1), ref.permute(0, 2, 1), 1e-3, 2e-5, 2e-5, f"CUDA-core cross J={J}")


# ------------------------------------------------------------------------------------------------ point stage
@functools.lru_cache(maxsize=None)
def point_inputs(J, N, B=3):
    """inputs, point cloud of N points, its nearest-cell taps and J joints (all on the GPU)"""
    from keypointfusion_b200 import ops
    inp = synth.make_inputs(B, 128, J, 128, seed=200 + J + N)
    c = {k: v.to(DEV) for k, v in inp.items()}
    pcl, _ = ops.getpcl(c["img"], c["center"], c["cube"], c["M"], c["cam"], sample_num=N, seed=2)
    close_, _, idx = ops.img2pcl_index(pcl, c["img"], c["center"], c["M"], c["cube"], c["cam"], 128, 4, fs=32, want_i64=False, want_i32=True)
    joint = cu(np.random.RandomState(J + N).uniform(-0.6, 0.6, (B, J, 3)).astype(np.float32))
    return inp, c, pcl, close_, idx, joint


def repack(c, J, maps):
    from keypointfusion_b200 import ops
    dt = torch.bfloat16 if maps == "bf16" else torch.float32
    return ops.repack_features(c["img_feat"].to(dt), c["img_feat_rgb"].to(dt), c["img_offset"][:, 4 * J:].to(dt))


@pytest.mark.parametrize("maps", ["bf16", "fp32"])
@pytest.mark.parametrize("N", [64, 1024, 2048])
@pytest.mark.parametrize("J", [1, 14, 21])
def test_point_stage_shapes(J, N, maps):
    """Point features and the per-joint softmax aggregation for J < 21 (A1 columns: offsets at 160 + 4j, xyz at 160 + 4J) and for
    one tile (N = 64) up to 32 tiles per sample."""
    from keypointfusion_b200 import ops
    inp, c, pcl, close_, idx, joint = point_inputs(J, N)
    blk, p = block(J)
    k = blk.kc()
    e16, acc, ms = ops.point_embed(repack(c, J, maps), idx, close_, pcl, joint, k["pe_wmat"], k["pe_wvec"], 0.8)
    e, agg = ops.e_to_float(e16), ops.combine_point_partials(acc, ms, J)
    # the oracle on the same maps: bf16 maps are exact in one plane; fp32 maps enter as two bf16 planes
    rnd = (lambda t: t.bfloat16().float()) if maps == "bf16" else (lambda t: t)
    pc, ix, cl = pcl.cpu(), idx.cpu().long(), close_.cpu()
    pf, pr = O.gather_taps(rnd(inp["img_feat"]), ix, cl), O.gather_taps(rnd(inp["img_feat_rgb"]), ix, cl)
    pw = O.gather_taps(rnd(inp["img_offset"])[:, 4 * J:], ix, cl)
    ee = torch.relu(O.conv_bn(p, "pcl_feat_emb.", pf) + O.conv_bn(p, "pcl_xyz_emb.", pc) +
                    O.conv_bn(p, "pcl_pose_emb.", torch.cat([pw, O.pcl_joint2offset(joint.cpu(), pc, 0.8)], -1)))
    ee = torch.relu(ee + O.conv_bn(p, "pcl_feat_emb_RGB.", pr))
    ragg = torch.softmax(pw.permute(0, 2, 1), -1) @ ee
    tol = _tol() if maps == "bf16" else 3e-5
    check(e, ee, tol, 10 * tol, f"point features J={J} N={N} {maps}")
    check(agg, ragg, tol, 10 * tol, f"joint aggregation J={J} N={N} {maps}")


@pytest.mark.parametrize("maps", ["bf16", "fp32"])
def test_point_stage_staged_tiles_14_joints_2048_points(maps):
    """stage_out (block 1) -> stage_in (block 2) of KPFusion(joint_num=14) at 32 tiles per sample: bit-identical to gathering again."""
    from keypointfusion_b200 import ops
    from keypointfusion_b200.model.model import KPFusion
    J, N = 14, 2048
    inp, c, pcl, close_, idx, _ = point_inputs(J, N)
    net = KPFusion(joint_num=J)
    synth.fill_state_dict(net, seed=5)
    net = net.to(DEV).eval()
    k1, k2 = net.block1.kc(), net.block2.kc()
    featT = repack(c, J, maps)
    j1, j2 = joint_set(pcl, J, "dense"), joint_set(pcl, J, "sparse")
    B = pcl.shape[0]
    for order in (None, ops.spatial_order(pcl, c["center"], c["M"], c["cube"], c["cam"], 128, 32)):
        stage = ops.point_embed_stage(B, N, pcl.device)
        stage.fill_(0x5a)
        a = ops.point_embed(featT, idx, close_, pcl, j1, k1["pe_wmat"], k1["pe_wvec"], 0.8, order=order, stage_out=stage)
        ref1 = ops.point_embed(featT, idx, close_, pcl, j1, k1["pe_wmat"], k1["pe_wvec"], 0.8, order=order)
        for x, y in zip(a, ref1):
            assert torch.equal(x, y)
        got = ops.point_embed(featT, idx, close_, pcl, j2, k2["pe_wmat"], k2["pe_wvec"], 0.8, order=order, stage_in=stage)
        ref2 = ops.point_embed(featT, idx, close_, pcl, j2, k2["pe_wmat"], k2["pe_wvec"], 0.8, order=order)
        for x, y in zip(got, ref2):
            assert torch.equal(x, y)


# ------------------------------------------------------------------------------------------------ DESA
RADII = (0.1, 0.2, 0.4)
DESA_J, DESA_N, NSAMPLE = (1, 13, 21, 32), (64, 2048), (32, 64, 128)


def _desa_module(ns, radius):
    from keypointfusion_b200.model.model import DESA
    m = DESA(128, [128, 128], [ns] * len(radius), list(radius))
    synth.fill_state_dict(m, seed=ns)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    return m.to(DEV).eval(), sd


desa_module = functools.lru_cache(maxsize=None)(_desa_module)


@functools.lru_cache(maxsize=None)
def desa_inputs(J, N, B=2):
    """point cloud of N points [B,N,3], point features [B,N,128] and joint features [B,J,128] (GPU)"""
    from keypointfusion_b200 import ops
    inp = synth.make_inputs(B, 128, J, 128, seed=100 + J + N)
    c = {k: inp[k].to(DEV) for k in ("img", "center", "M", "cube", "cam")}
    pcl, _ = ops.getpcl(c["img"], c["center"], c["cube"], c["M"], c["cam"], sample_num=N, seed=2)
    g = torch.Generator().manual_seed(J * N)
    return pcl, torch.randn(B, N, 128, generator=g).abs().to(DEV), torch.randn(B, J, 128, generator=g).abs().to(DEV)


def group_width(widest, ns):
    """rows per joint desa_tile_kernel groups for a scale whose widest ball (over the launch) holds `widest` points"""
    w = 16
    while w < widest:
        w *= 2
    return min(w, ns)


def ball_queries(pcl, joint, radii, ns):
    """oracle ball query over [points | joints] for every radius -> [(indices [B,J,ns], counts [B,J]), ...]"""
    xyz = torch.cat([pcl, joint], 1).cpu().numpy()
    return [O.ball_query(xyz, joint.cpu().numpy(), r, ns, return_counts=True) for r in radii]


def check_desa_scratch(buf, pcl, joint, radii, ns, what):
    """The prep kernel's ball-query indices (u16 [B,S,J,ns]) are bit-exact, and its widest ball per (sample, scale) (i32 [B,S], which
    sets the tile kernel's group width) is the oracle's.  Returns the group width of each scale."""
    B, N, _ = pcl.shape
    J, S = joint.shape[1], len(radii)
    off = B * S * J * 128 * 4 + B * (N + 32) * 16
    idx = buf[off:off + B * S * J * ns * 2].view(torch.int16).cpu().numpy().astype(np.uint16).reshape(B, S, J, ns)
    off += B * S * J * ns * 2
    gw = buf[off:off + B * S * 4].view(torch.int32).cpu().numpy().reshape(B, S)
    bq = ball_queries(pcl, joint, radii, ns)
    for s, (ri, _) in enumerate(bq):
        assert np.array_equal(idx[:, s].astype(np.int64), ri.astype(np.int64)), (what, radii[s])
    assert np.array_equal(gw, np.stack([np.minimum(cnt, ns).max(-1) for _, cnt in bq], 1)), (what, gw)
    return [group_width(int(gw[:, s].max()), ns) for s in range(S)]


def keep_desa_scratch(monkeypatch):
    """make the module's ops.desa_fused call keep its hand-over workspace for inspection"""
    from keypointfusion_b200 import ops
    scratch, real = {}, ops.desa_fused
    monkeypatch.setattr(ops, "desa_fused", lambda *a, **kw: real(*a, keep_scratch=scratch, **kw))
    return scratch


@pytest.mark.parametrize("which", ["dense", "sparse"])
@pytest.mark.parametrize("ns", NSAMPLE)
@pytest.mark.parametrize("N", DESA_N)
@pytest.mark.parametrize("J", DESA_J)
def test_desa_module_shapes(monkeypatch, J, N, ns, which):
    """The drop-in DESA module over joint counts (odd J: half-empty joint tiles), one point tile (N = 64) to 32, and nsample 32 / 64 /
    128 (group widths 16 .. 128 rows per joint)."""
    mod, sd = desa_module(ns, RADII)
    pcl, feat, nf = desa_inputs(J, N)
    joint = joint_set(pcl, J, which)
    scratch = keep_desa_scratch(monkeypatch)
    with torch.no_grad():
        out = mod(feat, nf, pcl, joint)
    torch.cuda.synchronize()
    ref = O.desa(sd, "", feat.cpu(), nf.cpu(), pcl.cpu(), joint.cpu(), radius=RADII, nsample=(ns,) * 3)
    what = f"DESA J={J} N={N} nsample={ns} {which}"
    check(out, ref, _tol(), 10 * _tol(), what)
    widths = check_desa_scratch(scratch["buf"], pcl, joint, RADII, ns, what)
    print(f"[{what}] group widths {widths}")


def test_desa_matrix_reaches_every_group_width():
    """The inputs of test_desa_module_shapes make the tile kernel group every width it has under every nsample (the kernel's widths
    are checked against these in each case), so a change of those inputs cannot drop a width unnoticed."""
    seen = set()
    for J, N, which in itertools.product(DESA_J, DESA_N, ("dense", "sparse")):
        pcl = desa_inputs(J, N)[0]
        joint = joint_set(pcl, J, which)
        for ns in NSAMPLE:
            seen.update((ns, group_width(int(np.minimum(cnt, ns).max()), ns)) for _, cnt in ball_queries(pcl, joint, RADII, ns))
    assert seen == {(32, 16), (32, 32), (64, 16), (64, 32), (64, 64), (128, 16), (128, 32), (128, 64), (128, 128)}, sorted(seen)


@pytest.mark.parametrize("which", ["dense", "sparse"])
@pytest.mark.parametrize("J", [13, 32])
@pytest.mark.parametrize("radii", [(0.2,), (0.1, 0.4), (0.1, 0.2, 0.3, 0.4)])
def test_desa_kernels_scale_count(radii, J, which):
    """kpf_desa_fused with 1, 2 and 4 scales vs the oracle's per-scale max-pooled outputs (the module itself takes three)."""
    from keypointfusion_b200 import ops
    ns, N, S = 64, 2048, len(radii)
    mod, sd = desa_module(ns, radii)
    eye, z = torch.eye(128, device=DEV), torch.zeros(128, device=DEV)
    wmat, wvec = ops.pack_desa(eye, z, torch.zeros(128, 3, device=DEV), z, mod.kc()["scales"])
    pcl, feat, nf = desa_inputs(J, N)
    joint = joint_set(pcl, J, which)
    scratch = {}
    part, _ = ops.desa_fused(ops.e_from_float(feat), None, None, pcl, joint, wmat, wvec, radii, ns, jf_in=nf, keep_scratch=scratch)
    torch.cuda.synchronize()
    ref = torch.stack(O.desa_scales(sd, "", feat.cpu(), nf.cpu(), pcl.cpu(), joint.cpu(), radius=radii, nsample=(ns,) * S), 1)
    what = f"DESA S={S} J={J} {which}"
    check(part.permute(0, 2, 1, 3), ref.permute(0, 2, 1, 3), _tol(), 10 * _tol(), what)
    check_desa_scratch(scratch["buf"], pcl, joint, radii, ns, what)


def test_desa_module_follows_joint_count():
    """One DESA module called with 21, then 14, then 21 joints: each call runs the fusion program packed for its own J."""
    mod, sd = _desa_module(64, RADII)
    for J in (21, 14, 21):
        pcl, feat, nf = desa_inputs(J, 2048)
        joint = joint_set(pcl, J, "dense")
        with torch.no_grad():
            out = mod(feat, nf, pcl, joint)
        ref = O.desa(sd, "", feat.cpu(), nf.cpu(), pcl.cpu(), joint.cpu(), radius=RADII, nsample=(64,) * 3)
        check(out, ref, _tol(), 10 * _tol(), f"DESA module, J={J} after another J")


# ------------------------------------------------------------------------------------------------ K5
def k5_oracle(p, f, hm, gam, prev, chunk=8):
    """O.spatial_aggregate in batch chunks (it materialises [B,J,C,HW])"""
    outs = [O.spatial_aggregate(p, "", f[i:i + chunk], hm[i:i + chunk], gam[i:i + chunk], None if prev is None else prev[i:i + chunk])
            for i in range(0, f.shape[0], chunk)]
    return torch.cat([o[0] for o in outs]), torch.cat([o[1] for o in outs])


@pytest.mark.parametrize("maps", ["bf16", "fp32"])
@pytest.mark.parametrize("J", [1, 14, 21, 32])
@pytest.mark.parametrize("B", [3, 64])
def test_spatial_aggregate_every_split(B, J, maps):
    """K5 with a sample's 8 cell tiles on 1 (one CTA per sample: what bench.py times), 2, 4 and 8 CTAs.  A launch twice gives the same
    bits, and leaves the last-CTA counters at zero for the next launch."""
    from keypointfusion_b200 import ops
    _, p = block(J)
    inp = synth.make_inputs(B, 128, J, 128, seed=300 + B + J)
    g = geo(inp)
    j3 = torch.from_numpy(np.random.RandomState(B + J).uniform(-0.7, 0.7, (B, J, 3)).astype(np.float32))
    prev = torch.from_numpy(np.random.RandomState(B * J).standard_normal((B, J, 128)).astype(np.float32))
    f = inp["img_feat_rgb"].bfloat16().float() if maps == "bf16" else inp["img_feat_rgb"]
    hm = O.joint2heatmap(j3[:, :, :2], 0.8, 32, sigma=1)
    gam = O.img2anchor_dis(j3, O.nearest_down(inp["img"], 32), *g, 128)
    refs = {pv is None: k5_oracle(p, f, hm, gam, pv) for pv in (None, prev)}
    planes = cu(f).bfloat16() if maps == "bf16" else ops.split_map(cu(f))
    jd = cu(j3)
    args = (jd, cu(inp["img"]), *[cu(x) for x in g], cu(ops.pack_spatial_wa(p["atten_spatial.weight"], J)), cu(p["atten_spatial.bias"]),
            cu(p["weight_dis"]), cu(p["fc_spatial2joint_feature.weight"]), cu(p["fc_spatial2joint_feature.bias"]))
    saved = ops.K5_SPLIT
    try:
        for split in (1, 2, 4, 8):
            ops.K5_SPLIT = split
            for pv in (None, cu(prev)):
                runs = []
                for _ in range(2):
                    runs.append(ops.spatial_aggregate_tc(planes, *args, prev=pv))
                    torch.cuda.synchronize()
                    assert not ops._zero_counters(B, jd.device).any(), split
                (sw, fj), (sw2, fj2) = runs
                assert torch.equal(sw, sw2) and torch.equal(fj, fj2), split
                rsw, rfj = refs[pv is None]
                what = f"K5 split={split} B={B} J={J} {maps} prev={pv is not None}"
                check(sw, rsw, 3e-5, 3e-4, what + " sw")
                check(fj, rfj, 3e-5, 3e-4, what + " fj")
    finally:
        ops.K5_SPLIT = saved


# ------------------------------------------------------------------------------------------------ K4a
@pytest.mark.parametrize("J", [1, 14, 20, 21])
def test_offset2joint_weight_variants(J):
    """bf16 maps: 3 joints per CTA at B = 2, 7 joints per CTA from the smallest batch that selects them (B * ceil(J/7) >= 592).  A joint's
    sums and their order do not depend on the CTA's joint count, so the B = 2 rows equal the same samples of the large batch."""
    from keypointfusion_b200 import ops
    big = -(-592 // -(-J // 7))
    assert big * -(-J // 7) >= 592 > (big - 1) * -(-J // 7)
    inp = synth.make_inputs(big, 128, J, 8, seed=400 + J)
    off, img = inp["img_offset"].bfloat16(), inp["img"]
    for ks in (0.8, torch.linspace(0.6, 1.0, J)):
        out = ops.offset2joint_weight(cu(off), cu(img), ks)
        small = ops.offset2joint_weight(cu(off[:2]), cu(img[:2]), ks)
        what = f"K4a J={J} kernel={'per joint' if torch.is_tensor(ks) else ks}"
        close(out, O.offset2joint_weight(off.float(), img, ks), 1e-3, 2e-6, 2e-5, what)
        assert torch.equal(small, out[:2]), what


# ------------------------------------------------------------------------------------------------ end to end at 14 joints
def mm_err(a, b):
    return float(np.linalg.norm((a.detach().float().cpu().numpy() - np.asarray(b)) * 125.0, axis=-1).mean())  # cube/2 = 125 mm


@functools.lru_cache(maxsize=None)
def kpfusion(J):
    from keypointfusion_b200.model.model import KPFusion
    net = KPFusion(joint_num=J)
    synth.fill_state_dict(net, seed=J)
    p = {k: v.clone() for k, v in net.state_dict().items()}
    return net.to(DEV).eval(), p


def path_inputs(B, J, seed, maps):
    inp = synth.make_inputs(B, 128, J, 128, seed=seed, bf16_round=maps == "bf16")
    c = {k: v.to(DEV) for k, v in inp.items()}
    if maps == "bf16":
        for k in ("img_feat", "img_feat_rgb", "img_offset"):
            c[k] = c[k].bfloat16()
    return inp, c


def check_joints(a, ref, what):
    e = mm_err(a, ref.numpy())
    print(f"[{what}] mean error {e:.5f} mm")
    assert e <= 0.05, (what, e)
    check(a, ref, 1e-3, 1e-2, what)


@pytest.mark.parametrize("maps", ["bf16", "fp32"])
@pytest.mark.parametrize("N", [512, 2048])
def test_fusion_path_14_joints(N, maps):
    """KPFusion(joint_num=14).forward_path on N-point clouds vs the oracle: the bars of test_fusion_path_tensor_core_meets_joint_bar.
    Stage 2 starts with DESA's ball query around stage 1's joints, where one membership flip under stage 1's float error moves the
    output by ~0.15 mm (DESIGN.md section 2), so it is checked against the oracle continued from OUR stage-1 joints."""
    from keypointfusion_b200 import ops
    from keypointfusion_b200.dataloader.loader import loader
    J, B = 14, 3
    net, p = kpfusion(J)
    inp, c = path_inputs(B, J, 500 + N, maps)
    g = geo(inp)
    L = loader(img_size=128)
    with torch.no_grad():
        pcl, _ = ops.getpcl(c["img"], c["center"], c["cube"], c["M"], c["cam"], sample_num=N, seed=4)
        res, sws, _ = net.forward_path(c["img_offset"], c["img_feat"], None, c["img_feat_rgb"], c["img"], pcl, L, c["center"], c["M"],
                                       c["cube"], c["cam"], 0.8)
    ores, osw, ex = O.fusion_path(p, inp["img"], pcl.cpu(), inp["img_offset"], inp["img_feat"], inp["img_feat_rgb"], *g, J=J)
    check_joints(res[2], ores[0], f"r3d_1 N={N} {maps}")
    check_joints(res[3], ores[1], f"r2d_1 N={N} {maps}")
    check(sws[0], osw[0], 1e-3, 1e-2, f"spatial weight 1 N={N} {maps}")
    with torch.no_grad():   # block 1's updated 2-D feature, the other input stage 2 takes from stage 1
        _, _, fj1, _, _ = net.block1(c["img_feat"], c["img_feat_rgb"], pcl, ex["joint_xyz0"].to(DEV), ex["closeness"].to(DEV),
                                     ex["index"].to(DEV).int(), c["img_offset"], None, L, c["img"][:, :, ::4, ::4], c["center"], c["M"],
                                     c["cube"], c["cam"])
    (q3, q2, _, qsw, _), _ = O.block_kpfusion(p, "block2.", inp["img_feat"], inp["img_feat_rgb"], pcl.cpu(), res[3].cpu(), ex["closeness"],
                                              ex["index"], inp["img_offset"], fj1.cpu(), O.nearest_down(inp["img"], 32), *g, 128, J=J)
    check_joints(res[4], q3, f"r3d_2 N={N} {maps}")
    check_joints(res[5], q2, f"r2d_2 N={N} {maps}")
    check(sws[1], qsw, 1e-3, 1e-2, f"spatial weight 2 N={N} {maps}")


def test_graphed_fusion_path_14_joints_512_points():
    from keypointfusion_b200 import ops
    from keypointfusion_b200.dataloader.loader import loader
    from keypointfusion_b200.runtime import GraphedFusionPath
    net, _ = kpfusion(14)
    _, c = path_inputs(3, 14, 600, "bf16")
    c.pop("img_rgb")
    L = loader(img_size=128)
    with torch.no_grad():
        pcl, _ = ops.getpcl(c["img"], c["center"], c["cube"], c["M"], c["cam"], sample_num=512, seed=0)
        res, _, _ = net.forward_path(c["img_offset"], c["img_feat"], None, c["img_feat_rgb"], c["img"], pcl, L, c["center"], c["M"],
                                     c["cube"], c["cam"], 0.8)
    graphed = GraphedFusionPath(net, L, c, sample_num=512, kernel=0.8, seed=0)
    assert torch.equal(graphed(c)["joints"], res[-1])
