"""CPU: argument checks of the graphed runtime that must fire before any CUDA work."""
import pytest
import torch

from keypointfusion_b200.utils import synth


def test_graphed_fusion_path_rejects_chains(monkeypatch):
    """A step is one kernel chain on one stream: any chains other than 1 is refused, pointing to OverlappedSteps, before a stream
    or a graph is created."""
    from keypointfusion_b200.model.model import KPFusion
    from keypointfusion_b200.runtime import GraphedFusionPath

    def no_cuda(*a, **k):
        raise AssertionError("CUDA was touched")
    for name in ("Stream", "CUDAGraph", "synchronize"):
        monkeypatch.setattr(torch.cuda, name, no_cuda)
    net = KPFusion(joint_num=21)
    example = synth.make_inputs(2, 128, 21, 128, seed=0)
    for chains in (2, 0):
        with pytest.raises(ValueError, match="OverlappedSteps"):
            GraphedFusionPath(net, None, example, chains=chains)
