"""Generate the golden fixtures in this directory by running the UNMODIFIED reference (/root/reference) on CPU
through ref_shims.py.  Runs only in the build container (the reference does not travel to the GPU box);
the .npz / .json files it writes are committed.

    python tests/golden/make_golden.py
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
import ref_shims  # noqa: E402

ref_shims.install()
from keypointfusion_b200.utils import synth  # noqa: E402

import torch.nn as nn  # noqa: E402
import torch.nn.functional as F  # noqa: E402
from model import model as ref_model  # noqa: E402
from model.model import Block_KPFusion  # noqa: E402
from model.transfusion_head import updatedDecoder  # noqa: E402
from model.fusion_layer import RGBDFusion, ACFusion, FSP  # noqa: E402
from util.generateFeature import GFM  # noqa: E402

torch.set_grad_enabled(False)
SEED = 7
B, S, J, C = 2, 128, 21, 128
H = S // 4


def npy(t):
    return t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t)


def shapes(sd):
    return {k: list(v.shape) for k, v in sd.items()}


def main():
    out = {}
    meta = {"seed": SEED, "B": B, "S": S, "J": J}
    loader = ref_shims.ref_loader(S)
    inp = synth.make_inputs(B, S, J, C, seed=SEED)
    img, center, M, cube, cam = inp["img"], inp["center"], inp["M"], inp["cube"], inp["cam"]
    # input checksums guard against generator drift
    meta["input_sums"] = {k: float(v.double().sum()) for k, v in inp.items()}

    # ---- a1/a2/a3: loader.getpcl per sample (numpy), explicit ranks --------------------------------
    pcl_s = np.zeros((B, 1024, 3), np.float32)
    counts = []
    for b in range(B):
        pcl = loader.getpcl(img[b, 0].numpy().copy(), center[b].numpy(), cube[b].numpy(), M[b].numpy().astype(np.float64),
                            tuple(float(x) for x in cam[b]))
        counts.append(pcl.shape[0])
        ranks = synth.explicit_ranks(pcl.shape[0], 1024, SEED + b)
        pcl_s[b] = pcl[ranks].astype(np.float32)
        if b == 0:
            out["getpcl_full0"] = pcl.astype(np.float64)
    out["getpcl_counts"] = np.array(counts, np.int32)
    out["pcl_sample"] = pcl_s
    # small-crop + sparse cases (P < 1024, P == 0)
    img64 = synth.make_depth_crops(2, 32, SEED + 1)
    img64[1] = 1.0
    c64, M64, cube64, cam64 = synth.make_camera(2, 32, SEED + 1)
    for b in range(2):
        pcl = loader.getpcl(img64[b, 0].copy(), c64[b], cube64[b], M64[b].astype(np.float64), tuple(float(x) for x in cam64[b]))
        out[f"getpcl_small{b}"] = pcl.astype(np.float64).reshape(-1, 3)
    pcl_t = torch.from_numpy(pcl_s)

    # ---- a5 -----------------------------------------------------------------------------------------
    rs = np.random.RandomState(SEED)
    uvd = torch.from_numpy(rs.uniform(-0.9, 0.9, (B, J, 3)).astype(np.float32))
    out["a5_uvd"] = npy(uvd)
    xyz = loader.uvd_nl2xyznl_tensor(uvd, center, M, cube, cam)
    out["a5_xyz"] = npy(xyz)
    out["a5_uvd_back"] = npy(loader.xyz_nl2uvdnl_tensor(xyz, center, M, cube, cam))

    # ---- a4 -----------------------------------------------------------------------------------------
    joint_uvd = ref_model.offset2joint_weight(inp["img_offset"], img, 0.8)
    out["a4_joint_uvd"] = npy(joint_uvd)
    out["a4_joint_uvd_gfm"] = npy(GFM().offset2joint_weight(inp["img_offset"], img, 0.8))
    ks = torch.linspace(0.6, 1.0, J)
    out["a4_joint_uvd_ktensor"] = npy(ref_model.offset2joint_weight(inp["img_offset"], img, ks))

    # ---- a6 -----------------------------------------------------------------------------------------
    img_down = F.interpolate(img, [H, H])
    out["img_down"] = npy(img_down)
    joint_xyz = loader.uvd_nl2xyznl_tensor(joint_uvd, center, M, cube, cam)
    out["joint_xyz0"] = npy(joint_xyz)
    close, index = loader.img2pcl_index(pcl_t, img_down, center, M, cube, cam, select_num=4)
    out["a6_closeness"] = npy(close)
    out["a6_index"] = npy(index).astype(np.int32)
    c9, i9 = loader.img2pcl_index(pcl_t[:, :64], img_down, center, M, cube, cam)  # default select_num=9
    out["a6_closeness9"], out["a6_index9"] = npy(c9), npy(i9).astype(np.int32)

    # ---- a7 -----------------------------------------------------------------------------------------
    out["a7_pcl_offset"] = npy(ref_model.pcl_joint2offset(joint_xyz, pcl_t, 0.8))[:, :128]
    out["a7_pcl_offset_gfm"] = npy(GFM().pcl_joint2offset(joint_xyz, pcl_t, 0.8))[:, :128]

    # ---- a8 (model.py:297-306, literal, using the reference's own ops) ------------------------------
    def ref_gather(feat):
        Cc = feat.shape[1]
        fi = index.view(B, 1, -1).repeat(1, Cc, 1)
        g = torch.gather(feat.reshape(B, Cc, -1), -1, fi).view(B, Cc, 1024, -1)
        return torch.sum(g * close.unsqueeze(1), dim=-1).permute(0, 2, 1)
    out["a8_pcl_feat"] = npy(ref_gather(inp["img_feat"]))[:, :64]
    out["a8_pcl_feat_rgb"] = npy(ref_gather(inp["img_feat_rgb"]))[:, :64]
    out["a8_pcl_weight"] = npy(ref_gather(inp["img_offset"][:, 4 * J:]))[:, :64]

    # ---- a10 / a11 ----------------------------------------------------------------------------------
    j3 = torch.from_numpy(rs.uniform(-0.7, 0.7, (B, J, 3)).astype(np.float32))
    out["a10_joint"] = npy(j3)
    out["a10_hm_s1"] = npy(GFM().joint2heatmap(j3[:, :, :2], 0.8, H, sigma=1))[:1]
    out["a10_hm_default"] = npy(GFM().joint2heatmap(j3, 0.8, H))[:1]
    out["a11_gam"] = npy(loader.img2anchor_dis(j3, img_down, center, M, cube, cam))[:1]

    # ---- a16 ----------------------------------------------------------------------------------------
    g = GFM()
    out["a16_joint2offset_gfm"] = npy(g.joint2offset(j3, img, 0.8, H))[:1]
    out["a16_joint2offset_model"] = npy(ref_model.joint2offset(j3, img, 0.8, H))[:1]
    feat = g.joint2feature(j3, img, [0.8], H, ['weight_offset'])
    out["a16_joint2feature"] = npy(feat)[:1]
    pix = torch.cat([feat, torch.from_numpy(rs.standard_normal((B, J, H, H)).astype(np.float32))], 1)
    out["a16_feature2joint"] = npy(g.feature2joint(img, pix, ['weight_offset'], [0.8]))
    out["a16_feature2joint_in_w"] = npy(pix[:, 4 * J:])

    # ---- a13 updatedDecoder -------------------------------------------------------------------------
    dec = updatedDecoder(joint_num=J, hidden_channel=128, num_heads=4, ffn_channel=128, dropout=0.1,
                         num_decoder_layers=4, activation='relu').eval()
    synth.fill_state_dict(dec, SEED)
    a = torch.from_numpy(rs.standard_normal((B, J, 128)).astype(np.float32))
    k = torch.from_numpy(rs.standard_normal((B, J, 128)).astype(np.float32))
    out["a13_anchor"], out["a13_key"] = npy(a), npy(k)
    out["a13_out"] = npy(dec(a, k))
    meta["updatedDecoder_keys"] = shapes(dec.state_dict())
    mha = dec.decoder[3].multihead_attn
    q = torch.from_numpy(rs.standard_normal((J, B, 128)).astype(np.float32))
    kk = torch.from_numpy(rs.standard_normal((9, B, 128)).astype(np.float32))
    o, w = mha(q, kk, kk)
    out["a13_mha_q"], out["a13_mha_k"], out["a13_mha_out"], out["a13_mha_w"] = npy(q), npy(kk), npy(o), npy(w)

    # ---- a14 / a15 ----------------------------------------------------------------------------------
    for name, cls in (("rgbd", RGBDFusion), ("ac", ACFusion)):
        m = cls(64, 64).eval()
        synth.fill_state_dict(m, SEED)
        r = torch.from_numpy(rs.standard_normal((B, 64, 8, 8)).astype(np.float32))
        d = torch.from_numpy(rs.standard_normal((B, 64, 8, 8)).astype(np.float32))
        (ro, do), mg = m([r, d])
        out[f"a14_{name}_rgb"], out[f"a14_{name}_depth"] = npy(r), npy(d)
        out[f"a14_{name}_rgb_out"], out[f"a14_{name}_depth_out"], out[f"a14_{name}_merge"] = npy(ro), npy(do), npy(mg)
        meta[f"{cls.__name__}_keys"] = shapes(m.state_dict())
    fsp = FSP(64, 64).eval()
    synth.fill_state_dict(fsp, SEED)
    out["a15_fsp_out"] = npy(fsp(torch.from_numpy(out["a14_rgbd_rgb"]), torch.from_numpy(out["a14_rgbd_depth"])))
    meta["FSP_keys"] = shapes(fsp.state_dict())

    # ---- a9/a12/a17 + "next" rows: the whole path after the backbones (model.py:399-426) -----------
    class Path(nn.Module):
        def __init__(self):
            super().__init__()
            self.block1 = Block_KPFusion(joint_num=J)
            self.block2 = Block_KPFusion(joint_num=J)
    net = Path().eval()
    synth.fill_state_dict(net, SEED)
    meta["Block_KPFusion_keys"] = shapes(net.block1.state_dict())
    caps = {}

    def hook(name):
        def f(mod, args, o):
            caps[name] = o
        return f
    for i, blk in ((1, net.block1), (2, net.block2)):
        blk.FA.register_forward_hook(hook(f"b{i}_desa"))
        blk.init_TR.register_forward_hook(hook(f"b{i}_init_TR"))
        blk.crossTR.register_forward_hook(hook(f"b{i}_cross"))
    jx = joint_xyz
    prev = None
    for i, blk in ((1, net.block1), (2, net.block2)):
        r3d, r2d, prev, sw, _ = blk(inp["img_feat"], inp["img_feat_rgb"], pcl_t, jx, close, index, inp["img_offset"],
                                    prev, loader, img_down, center, M, cube, cam)
        out[f"b{i}_r3d"], out[f"b{i}_r2d"], out[f"b{i}_img_feat_j"] = npy(r3d), npy(r2d), npy(prev)
        out[f"b{i}_sw0"] = npy(sw)[:1]
        out[f"b{i}_desa"] = npy(caps[f"b{i}_desa"])
        out[f"b{i}_tok_init"] = npy(caps[f"b{i}_init_TR"][0])
        out[f"b{i}_cross"] = npy(caps[f"b{i}_cross"])
        jx = r2d

    # stored compactly, no fixture file above 1 MB: the inputs drawn from `rs` above are regenerated by tests/conftest.py, the
    # outputs the reference computes identically twice are stored once, and the per-cell joint maps go to a file of their own
    sys.path.insert(0, os.path.dirname(HERE))
    from conftest import fingerprint, seeded_draws
    meta["seeded_sha256"] = {}
    for k, v in seeded_draws(SEED, B, J, H).items():
        assert np.array_equal(out[k], v) and out[k].dtype == v.dtype, k
        meta["seeded_sha256"][k] = fingerprint(out.pop(k))
    meta["copies_sha256"] = {}
    for k, src in (("a4_joint_uvd_gfm", "a4_joint_uvd"), ("a7_pcl_offset_gfm", "a7_pcl_offset"), ("a16_joint2feature", "a16_joint2offset_gfm")):
        meta["copies_sha256"][k] = [src, fingerprint(out.pop(k))]
    np.savez_compressed(os.path.join(HERE, "golden_maps.npz"), **{k: out.pop(k) for k in ("a10_hm_s1", "a10_hm_default", "a11_gam")})
    np.savez_compressed(os.path.join(HERE, "golden_path.npz"), **out)
    with open(os.path.join(HERE, "golden_meta.json"), "w") as f:
        json.dump(meta, f, indent=0, sort_keys=True)
    sz = os.path.getsize(os.path.join(HERE, "golden_path.npz"))
    print("wrote golden_path.npz", sz / 1e6, "MB;", len(out), "arrays; counts", counts)


if __name__ == "__main__":
    main()


def add_eval_tail_golden():
    """SURVEY 8f-4: GFM.rigid_align of the reference on seeded joint sets incl. a reflection (det(R) < 0 branch); appended to
    golden_path.npz as f4_A / f4_B / f4_aligned."""
    g = GFM()
    rs = np.random.RandomState(11)
    A = rs.uniform(-0.8, 0.8, (6, 21, 3)).astype(np.float32)
    Rm = np.linalg.qr(rs.standard_normal((3, 3)))[0]
    B2 = (1.3 * (A @ Rm.T) + 0.1 + 0.02 * rs.standard_normal(A.shape)).astype(np.float32)
    B2[1] = (A[1] * np.array([1, 1, -1], np.float32)) + 0.01 * rs.standard_normal((21, 3)).astype(np.float32)
    B2[2] = A[2] + 0.05 * rs.standard_normal((21, 3)).astype(np.float32)
    out = np.stack([g.rigid_align(A[i], B2[i]) for i in range(6)])
    path = os.path.join(HERE, "golden_path.npz")
    d = dict(np.load(path))
    d.update(f4_A=A, f4_B=B2, f4_aligned=out.astype(np.float64))
    np.savez_compressed(path, **d)


if __name__ == "__main__":
    add_eval_tail_golden()
