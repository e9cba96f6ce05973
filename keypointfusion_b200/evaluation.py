"""Evaluation on the device (SURVEY.md 8f-4): what the reference's Trainer.test prints (train.py:330-396: mean_Error and PA_mean_Error,
from xyz2error :470-488 and GFM.rigid_align, util/generateFeature.py:681-703), plus PCK / AUC, accumulated per joint set inside the
step by one kernel (kpf_eval_accumulate) and read back once at the end, summed across ranks.

    ev = Evaluator(joint_num=21)                  # stages "offset", "r3d_1", "r2d_1", "r3d_2", "r2d_2"; thresholds 0..50 mm
    ev.update(stage_joints(result, img, center, M, cube, cam, loader), gt, cube, valid)    # per step, graph-safe, no sync
    stats = ev.summary(group)                     # every rank calls it
    stats["r2d_2"]["mean_error_mm"], stats["r2d_2"]["pa_mean_error_mm"]

runtime.GraphedEvalPath runs the update inside the captured step."""
import re

import numpy as np
import torch

from . import ops
from .model.model import offset2joint_weight

DEFAULT_STAGES = ("offset", "r3d_1", "r2d_1", "r3d_2", "r2d_2")


def stage_joints(result, img, center, M, cube, cam, loader, kernel=0.8, names=DEFAULT_STAGES):
    """KPFusion.forward_path's `result` = [img_offset, img_offset_rgb, r3d_1, r2d_1, r3d_2, r2d_2, ...] -> one normalised-xyz joint set
    [B,J,3] per entry of `names`, in that order.  "r3d_k" / "r2d_k" are block k's outputs as they are; "offset" and "offset_rgb" are
    the depth and rgb backbones' offset maps turned into joints the way the network turns them (model.py:399-410, GFM.feature2joint):
    offset2joint_weight against the depth crop `img`, then uvd2xyz with the step's center, M, cube and cam."""
    sets = []
    for name in names:
        if name in ("offset", "offset_rgb"):
            off = result[0 if name == "offset" else 1]
            if off is None:
                raise ValueError(f"stage {name!r}: forward_path returned no {name} map")
            uvd = offset2joint_weight(off, img, kernel)
            sets.append(torch.ops.kpf.uvd2xyz(uvd, center, M, cube, cam, float(loader.img_size), float(loader.flip)))
            continue
        m = re.fullmatch(r"(r3d|r2d)_([1-9][0-9]*)", name)
        i = 2 + 2 * (int(m.group(2)) - 1) + (m.group(1) == "r2d") if m else -1
        if not 2 <= i < len(result):
            raise ValueError(f"unknown stage {name!r}: expected offset, offset_rgb or r3d_k / r2d_k with k <= {(len(result) - 2) // 2}")
        sets.append(result[i])
    return sets


def summarize(acc, joint_num, thresholds, stage_names):
    """Accumulator rows (int64 [S, ops.eval_row_length(J, T)], host or device) -> {stage name: statistics}.  For the plain error and,
    under the prefix "pa_", the Procrustes-aligned error:
      mean_error_mm       sum of the finite joint errors / their number (every joint of every valid sample, finite ones only);
      per_joint_error_mm  [J] the same per joint;
      pck                 [T] fraction of all samples * J joints with error <= threshold k: cumulative histogram / (samples * J),
                          so a non-finite joint counts as a miss;
      auc                 trapz(pck, thresholds) / (thresholds[-1] - thresholds[0]) (NaN with one threshold);
      nonfinite           number of NaN / inf joint errors;
    and `samples`, the valid samples seen.  Empty counts give NaN."""
    a = acc.cpu().numpy() if torch.is_tensor(acc) else np.asarray(acc)
    J, T = int(joint_num), len(thresholds)
    thr = np.asarray(thresholds, np.float64)
    out = {}
    for s, name in enumerate(stage_names):
        row = a[s]
        n = int(row[0])
        st = {"samples": n}
        for k, pre in enumerate(("", "pa_")):
            sums = [int(x) for x in row[1 + k * J:1 + (k + 1) * J]]      # Python ints: no overflow across joints
            nonfinite = [int(x) for x in row[1 + (2 + k) * J:1 + (3 + k) * J]]
            hist = row[1 + 4 * J + k * (T + 1):1 + 4 * J + (k + 1) * (T + 1)].astype(np.int64)
            finite = [n - c for c in nonfinite]
            st[pre + "mean_error_mm"] = sum(sums) / ops.EVAL_SCALE / sum(finite) if sum(finite) else float("nan")
            st[pre + "per_joint_error_mm"] = np.array([x / ops.EVAL_SCALE / f if f else np.nan for x, f in zip(sums, finite)])
            pck = np.cumsum(hist[:T]) / (n * J) if n else np.full(T, np.nan)
            st[pre + "pck"] = pck
            st[pre + "auc"] = float(np.sum((pck[1:] + pck[:-1]) / 2 * np.diff(thr)) / (thr[-1] - thr[0])) if T > 1 else float("nan")
            st[pre + "nonfinite"] = sum(nonfinite)
        out[name] = st
    return out


class Evaluator:
    """Device-resident evaluation of several joint sets ("stages") at once: `acc` [S, ops.eval_row_length(J, T)] int64 holds, per
    stage, the valid samples, per-joint fixed-point sums (2^20 units per mm) and non-finite counts of the error and the aligned error,
    and their histograms over `thresholds_mm` (include/kpf_b200.h: kpf_eval_accumulate).  The totals are integer sums: exact, and the
    same whatever the batch order, batch split, steps in flight or number of ranks.

    Statistics (`summary`, definitions in `summarize`): means over finite joints; PCK = cumulative histogram / (samples * J), a
    non-finite joint counting as a miss; AUC = trapz(pck, thr) / (thr[-1] - thr[0]).  The means are the reference's mean_Error and
    PA_mean_Error (train.py:330-396; kpf_eval_errors is pinned to its rigid_align).  The reference's util/eval_utils.py is not
    available, so PCK and AUC follow the definitions above and make no claim of parity with its eval_auc."""

    def __init__(self, joint_num, stage_names=DEFAULT_STAGES, thresholds_mm=np.arange(0, 51.0), device="cuda"):
        self.joint_num = int(joint_num)
        self.stage_names = tuple(stage_names)
        self.thresholds = ops.eval_thresholds(thresholds_mm)
        if not 1 <= len(self.stage_names) <= ops.EVAL_MAX_SETS:
            raise ValueError(f"{len(self.stage_names)} stages: 1..{ops.EVAL_MAX_SETS} are supported")
        if not 3 <= self.joint_num <= ops.EVAL_MAX_JOINTS:
            raise ValueError(f"{self.joint_num} joints: 3..{ops.EVAL_MAX_JOINTS} are supported")
        self.acc = torch.zeros(len(self.stage_names), ops.eval_row_length(self.joint_num, len(self.thresholds)), dtype=torch.int64,
                               device=device)

    def update(self, sets, gt, cube, valid=None):
        """Add one batch: sets = one [B,J,3] normalised-xyz joint set per stage (a sequence, e.g. stage_joints(...), or a stacked
        [S,B,J,3] tensor), gt [B,J,3] normalised xyz, cube [B,3] mm, valid [B] uint8 (0: a padding row, ignored) or None.
        Enqueues one kernel on the current stream: no host synchronisation, so it can run inside a captured CUDA graph."""
        pred = sets if torch.is_tensor(sets) else torch.stack(list(sets))
        if pred.dim() != 4 or pred.shape[0] != len(self.stage_names) or pred.shape[2] != self.joint_num:
            raise ValueError(f"joint sets {tuple(pred.shape)}: expected [{len(self.stage_names)}, B, {self.joint_num}, 3] "
                             f"(stages {self.stage_names})")
        torch.ops.kpf.eval_accumulate(self.acc, pred, gt, cube, valid, list(self.thresholds))

    def reset(self):
        self.acc.zero_()

    def summary(self, group=None):
        """-> {stage name: statistics} (see `summarize`).  Synchronises the device once (every stream: updates enqueued on other
        streams are included); with a process group, sums a copy of the accumulator over its ranks first (one all_reduce), so
        every rank of the group must call it and every rank gets the same result."""
        acc = self.acc
        if acc.is_cuda:
            torch.cuda.synchronize(acc.device)
        if group is not None:
            import torch.distributed as dist
            acc = acc.clone()
            dist.all_reduce(acc, op=dist.ReduceOp.SUM, group=group)
        return summarize(acc, self.joint_num, self.thresholds, self.stage_names)
