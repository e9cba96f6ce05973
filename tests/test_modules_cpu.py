"""CPU: argument checks of the drop-in modules that must fire before any CUDA work."""
import pytest
import torch


@pytest.mark.parametrize("radius", [[0.1, 0.2, 0, 4], [0.2], [0.1, 0.4]])
def test_desa_refuses_other_than_three_scales(radius):
    """The fusion conv runs in the token-stack prologue, which reads exactly three scales: DESA with the reference's default radii
    (four entries) or with one or two is refused, not computed.  CPU tensors: a check that came too late would fail on them with a
    RuntimeError from the launch wrappers instead."""
    from keypointfusion_b200.model.model import DESA
    m = DESA(128, [128, 128], [64] * len(radius), radius) if len(radius) != 4 else DESA(128, [128, 128])
    m.eval()
    B, N, J = 2, 64, 21
    with torch.no_grad(), pytest.raises(NotImplementedError, match="three scales"):
        m(torch.rand(B, N, 128), torch.rand(B, J, 128), torch.rand(B, N, 3), torch.rand(B, J, 3))
