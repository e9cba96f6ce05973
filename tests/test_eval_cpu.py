"""CPU: the device evaluation layer without a device.  kpf::eval_accumulate is a registered custom op that declares its one in-place
effect; stage_joints + Evaluator.update shape-propagate after forward_path under FakeTensorMode; summary()'s statistics follow from a
hand-built accumulator; malformed arguments raise ValueError before any launch."""
import numpy as np
import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

from keypointfusion_b200 import custom_ops, ops
from keypointfusion_b200.dataloader.loader import loader
from keypointfusion_b200.evaluation import DEFAULT_STAGES, Evaluator, stage_joints
from keypointfusion_b200.model.model import KPFusion
from keypointfusion_b200.utils import synth


def test_eval_accumulate_is_registered_and_mutates_acc():
    assert "eval_accumulate" in custom_ops.REGISTERED
    schema = str(torch.ops.kpf.eval_accumulate.default._schema)
    assert "Tensor(a0!) acc" in schema and "-> ()" in schema


def test_stage_joints_and_update_shape_propagate_under_fake_tensors():
    net = KPFusion(joint_num=21).eval()
    synth.fill_state_dict(net, 0)
    with torch.no_grad():
        net.block1.kc(), net.block2.kc()
        with FakeTensorMode(allow_non_fake_inputs=True):
            B, dev = 3, "cuda"
            img = torch.empty(B, 1, 128, 128, device=dev)
            maps = [torch.empty(B, c, 32, 32, device=dev, dtype=torch.bfloat16) for c in (128, 128, 105)]
            center, cube, M, cam = (torch.empty(B, 3, device=dev), torch.empty(B, 3, device=dev), torch.empty(B, 3, 3, device=dev),
                                    torch.empty(B, 4, device=dev))
            L = loader(img_size=128)
            pcl, _ = torch.ops.kpf.getpcl(img, center, cube, M, cam, 1024, 0, False, 1.0, None)
            res, _, _ = net.forward_path(maps[2], maps[0], None, maps[1], img, pcl, L, center, M, cube, cam, 0.8)
            sets = stage_joints(res, img, center, M, cube, cam, L)
            assert [tuple(s.shape) for s in sets] == [(B, 21, 3)] * len(DEFAULT_STAGES)
            assert all(s.dtype == torch.float32 and s.device.type == "cuda" for s in sets)
            ev = Evaluator(21, device=dev)
            ev.update(sets, torch.empty(B, 21, 3, device=dev), cube, torch.empty(B, device=dev, dtype=torch.uint8))
            assert tuple(ev.acc.shape) == (5, ops.eval_row_length(21, 51)) and ev.acc.dtype == torch.int64
            with pytest.raises(ValueError, match="offset_rgb"):
                stage_joints(res, img, center, M, cube, cam, L, names=("offset_rgb",))
            with pytest.raises(ValueError, match="r2d_3"):
                stage_joints(res, img, center, M, cube, cam, L, names=("r2d_3",))


def _put(acc, s, J, T, samples, err_sum_mm, pa_sum_mm, err_nf, pa_nf, err_hist, pa_hist):
    row = acc[s]
    row[0] = samples
    row[1:1 + J] = torch.as_tensor(np.rint(np.asarray(err_sum_mm) * ops.EVAL_SCALE).astype(np.int64))
    row[1 + J:1 + 2 * J] = torch.as_tensor(np.rint(np.asarray(pa_sum_mm) * ops.EVAL_SCALE).astype(np.int64))
    row[1 + 2 * J:1 + 3 * J] = torch.as_tensor(err_nf)
    row[1 + 3 * J:1 + 4 * J] = torch.as_tensor(pa_nf)
    row[1 + 4 * J:1 + 4 * J + T + 1] = torch.as_tensor(err_hist)
    row[1 + 4 * J + T + 1:] = torch.as_tensor(pa_hist)


def test_summary_math_on_a_hand_built_accumulator():
    J, thr = 3, (0.0, 10.0, 20.0, 40.0)
    T = len(thr)
    ev = Evaluator(J, stage_names=("a", "b"), thresholds_mm=torch.tensor(thr), device="cpu")
    # stage a: 4 samples, all 12 joint errors finite, spread over the bins 1, 2, 3 and beyond the last threshold
    _put(ev.acc, 0, J, T, 4, [10.0, 20.0, 30.0], [4.0, 8.0, 12.0], [0, 0, 0], [0, 0, 0], [0, 3, 5, 2, 2], [0, 12, 0, 0, 0])
    # stage b: 2 samples, joint 1 non-finite in one sample (plain error) and in both (aligned error)
    _put(ev.acc, 1, J, T, 2, [2.0, 3.0, 4.0], [1.0, 0.0, 1.0], [0, 1, 0], [0, 2, 0], [1, 4, 0, 0, 1], [0, 4, 0, 0, 2])
    st = ev.summary()
    a, b = st["a"], st["b"]
    assert a["samples"] == 4 and b["samples"] == 2
    assert a["mean_error_mm"] == pytest.approx(60.0 / 12) and a["pa_mean_error_mm"] == pytest.approx(24.0 / 12)
    np.testing.assert_allclose(a["per_joint_error_mm"], [2.5, 5.0, 7.5])
    np.testing.assert_allclose(a["pck"], np.cumsum([0, 3, 5, 2]) / 12)
    np.testing.assert_allclose(a["pa_pck"], [0, 1, 1, 1])
    pck = np.cumsum([0, 3, 5, 2]) / 12
    auc = ((pck[0] + pck[1]) / 2 * 10 + (pck[1] + pck[2]) / 2 * 10 + (pck[2] + pck[3]) / 2 * 20) / 40
    assert a["auc"] == pytest.approx(auc)
    assert a["pa_auc"] == pytest.approx((0.5 * 10 + 10 + 20) / 40)
    # means over finite joints only; a non-finite joint is a PCK miss (it sits in bin T)
    assert b["mean_error_mm"] == pytest.approx(9.0 / 5) and b["pa_mean_error_mm"] == pytest.approx(2.0 / 4)
    np.testing.assert_allclose(b["per_joint_error_mm"], [1.0, 3.0, 2.0])
    pj = b["pa_per_joint_error_mm"]
    assert pj[0] == pytest.approx(0.5) and np.isnan(pj[1]) and pj[2] == pytest.approx(0.5)
    np.testing.assert_allclose(b["pck"], np.array([1, 5, 5, 5]) / 6)
    np.testing.assert_allclose(b["pa_pck"], np.array([0, 4, 4, 4]) / 6)
    assert b["nonfinite"] == 1 and b["pa_nonfinite"] == 2 and a["nonfinite"] == 0
    # nothing accumulated: NaN statistics, no division error
    ev.reset()
    st = ev.summary()
    assert st["a"]["samples"] == 0 and np.isnan(st["a"]["mean_error_mm"]) and np.all(np.isnan(st["a"]["pck"]))


def test_summary_sums_are_exact_beyond_float64():
    """Per-joint sums are integers: totals across joints are summed as Python integers, not in int64 or float64."""
    J = 3
    ev = Evaluator(J, stage_names=("a",), thresholds_mm=[1.0, 2.0], device="cpu")
    big = 2 ** 62
    ev.acc[0, 0] = 2 ** 23
    ev.acc[0, 1:1 + J] = big
    assert ev.summary()["a"]["mean_error_mm"] == pytest.approx(3 * big / ops.EVAL_SCALE / (3 * 2 ** 23), rel=1e-15)


def _args(S=2, B=4, J=21, T=51):
    pred = [torch.zeros(B, J, 3) for _ in range(S)]
    return dict(acc=torch.zeros(S, ops.eval_row_length(J, T), dtype=torch.int64), pred_sets=pred, gt=torch.zeros(B, J, 3),
                cube=torch.ones(B, 3), valid=torch.ones(B, dtype=torch.uint8), thresholds=torch.arange(0, float(T)))


@pytest.mark.parametrize("case, match", [
    (dict(thresholds=[0.0, 2.0, 1.0]), "increasing"),
    (dict(thresholds=[0.0, 1.0, 1.0]), "increasing"),
    (dict(thresholds=[0.0, float("nan")]), "finite"),
    (dict(thresholds=list(range(257))), "257 thresholds"),
    (dict(thresholds=[]), "0 thresholds"),
    (dict(pred_sets=[torch.zeros(4, 21, 3)] * 9, acc=torch.zeros(9, ops.eval_row_length(21, 51), dtype=torch.int64)), "9 joint sets"),
    (dict(gt=torch.zeros(4, 20, 3)), "gt"),
    (dict(pred_sets=[torch.zeros(4, 33, 3)] * 2, gt=torch.zeros(4, 33, 3)), "33 joints"),
    (dict(valid=torch.ones(4, dtype=torch.bool)), "uint8"),
    (dict(valid=torch.ones(5, dtype=torch.uint8)), "uint8"),
    (dict(acc=torch.zeros(2, ops.eval_row_length(21, 51), dtype=torch.int32)), "int64"),
    (dict(acc=torch.zeros(2, ops.eval_row_length(21, 50), dtype=torch.int64)), "int64"),
    (dict(cube=torch.ones(4, 4)), "cube"),
])
def test_eval_accumulate_rejects_bad_arguments_before_launch(case, match):
    a = _args()
    a.update(case)
    with pytest.raises(ValueError, match=match):
        ops.eval_accumulate(**a)
    # the same checks under the custom op's fake kernel (what torch.compile / FakeTensorMode tracing sees)
    pred, thr = torch.stack(a["pred_sets"]), [float(x) for x in a["thresholds"]]
    with FakeTensorMode(allow_non_fake_inputs=True), pytest.raises(ValueError, match=match):
        torch.ops.kpf.eval_accumulate(a["acc"], pred, a["gt"], a["cube"], a["valid"], thr)


def test_thresholds_are_host_values_and_evaluator_checks_its_shape():
    with pytest.raises(ValueError, match="host"):
        ops.eval_thresholds(torch.zeros(3, device="meta"))
    with pytest.raises(ValueError, match="9 stages"):
        Evaluator(21, stage_names=[str(i) for i in range(9)], device="cpu")
    with pytest.raises(ValueError, match="increasing"):
        Evaluator(21, thresholds_mm=[5.0, 1.0], device="cpu")
    ev = Evaluator(21, stage_names=("a", "b"), device="cpu")
    with pytest.raises(ValueError, match="expected"):
        ev.update([torch.zeros(4, 21, 3)] * 3, torch.zeros(4, 21, 3), torch.ones(4, 3))
    with pytest.raises(RuntimeError, match="CUDA"):   # valid arguments on the host: no CPU fallback exists
        ev.update([torch.zeros(4, 21, 3)] * 2, torch.zeros(4, 21, 3), torch.ones(4, 3))
