import hashlib
import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def fingerprint(a):
    """sha256 of an array's dtype, shape and bytes (tests/golden/make_golden.py records these for the arrays it does not store)."""
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def seeded_draws(seed, B, J, H):
    """The inputs tests/golden/make_golden.py draws from RandomState(seed) for the reference, in the order it draws them."""
    rs = np.random.RandomState(seed)
    d = {}
    d["a5_uvd"] = rs.uniform(-0.9, 0.9, (B, J, 3))
    d["a10_joint"] = rs.uniform(-0.7, 0.7, (B, J, 3))
    d["a16_feature2joint_in_w"] = rs.standard_normal((B, J, H, H))
    d["a13_anchor"] = rs.standard_normal((B, J, 128))
    d["a13_key"] = rs.standard_normal((B, J, 128))
    d["a13_mha_q"] = rs.standard_normal((J, B, 128))
    d["a13_mha_k"] = rs.standard_normal((9, B, 128))
    for name in ("rgbd", "ac"):
        d[f"a14_{name}_rgb"] = rs.standard_normal((B, 64, 8, 8))
        d[f"a14_{name}_depth"] = rs.standard_normal((B, 64, 8, 8))
    return {k: v.astype(np.float32) for k, v in d.items()}


@pytest.fixture(scope="session")
def golden(golden_meta):
    """The reference's outputs (golden_path.npz, golden_maps.npz) plus the seeded inputs it was fed, regenerated here, and the
    copies it produced bit-identically twice, stored once; both are checked against the fingerprints of what the reference saw."""
    m = golden_meta
    d = {}
    for name in ("golden_path.npz", "golden_maps.npz"):
        d.update(np.load(os.path.join(GOLDEN, name)))
    for k, v in seeded_draws(m["seed"], m["B"], m["J"], m["S"] // 4).items():
        assert fingerprint(v) == m["seeded_sha256"][k], f"seeded draw {k} differs from the one the reference was fed"
        d[k] = v
    for k, (src, sha) in m["copies_sha256"].items():
        assert fingerprint(d[src]) == sha, f"{k} is not a bit-identical copy of {src}"
        d[k] = d[src]
    return d


@pytest.fixture(scope="session")
def golden_meta():
    with open(os.path.join(GOLDEN, "golden_meta.json")) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def golden_inputs(golden_meta):
    from keypointfusion_b200.utils import synth
    m = golden_meta
    inp = synth.make_inputs(m["B"], m["S"], m["J"], 128, seed=m["seed"])
    for k, v in m["input_sums"].items():  # generator drift guard
        assert abs(float(inp[k].double().sum()) - v) <= 1e-6 * max(1.0, abs(v)), k
    return inp


@pytest.fixture(scope="session")
def path_params(golden_meta):
    """state_dict {block1.*, block2.*} with the SAME deterministic fill the golden run used."""
    from keypointfusion_b200.utils import synth
    sd = {}
    for blk in ("block1.", "block2."):
        for k, shp in golden_meta["Block_KPFusion_keys"].items():
            dt = torch.int64 if k.endswith("num_batches_tracked") or k.endswith("position_ids") else torch.float32
            sd[blk + k] = torch.zeros(shp, dtype=dt)
    synth.fill_state_dict(sd, golden_meta["seed"])
    return sd
