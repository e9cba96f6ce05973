"""GPU: tcgen05 building blocks (shared-memory descriptors, K-major / MN-major operands, TMEM read-back)."""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("N,K", [(128, 128), (256, 64), (32, 128), (128, 32), (48, 16)])
@pytest.mark.parametrize("a_mn,b_mn", [(0, 0), (0, 1), (1, 0), (1, 1)])
def test_umma_gemm(N, K, a_mn, b_mn):
    from keypointfusion_b200 import _lib, ops
    torch.manual_seed(N * 7 + K + a_mn * 2 + b_mn)
    A = torch.randn(128, K, device="cuda").bfloat16()
    B = torch.randn(N, K, device="cuda").bfloat16()
    D = torch.zeros(128, N, device="cuda")
    Ain = A.t().contiguous() if a_mn else A
    Bin = B.t().contiguous() if b_mn else B
    ops._call("kpf_umma_selftest", ops._p(Ain), ops._p(Bin), ops._p(D), N, K, a_mn, b_mn)
    torch.cuda.synchronize()
    ref = A.float() @ B.float().t()
    assert torch.allclose(D, ref, rtol=1e-4, atol=1e-3), (D - ref).abs().max()


@pytest.mark.parametrize("fmt", [0, 1])
@pytest.mark.parametrize("a_tmem", [0, 1])
@pytest.mark.parametrize("N,K", [(32, 128), (64, 128), (128, 128), (64, 256), (16, 32)])
def test_umma_split_gemm(N, K, fmt, a_tmem, capsys):
    """fp32 operands as (hi, lo) 16-bit planes, three MMAs: ~2^-16 (bf16 planes) / ~2^-21 (fp16 planes) instead of 2^-9;
    A from shared memory and from tensor memory.  Prints the cycle counts used in DESIGN.md."""
    from keypointfusion_b200 import ops
    torch.manual_seed(N + K + fmt)
    A = torch.randn(128, K, device="cuda")
    B = torch.randn(N, K, device="cuda")
    D = torch.zeros(128, N, device="cuda")
    cyc = torch.zeros(2, dtype=torch.int64, device="cuda")
    ops._call("kpf_umma_split_selftest", ops._p(A), ops._p(B), ops._p(D), N, K, fmt, a_tmem, 0, ops._p(cyc))
    torch.cuda.synchronize()
    ref = (A.double() @ B.double().t())
    rel = float((D.double() - ref).norm() / ref.norm())
    with capsys.disabled():
        print(f"\n[split gemm] N={N} K={K} fmt={'bf16' if fmt else 'fp16'} A={'tmem' if a_tmem else 'smem'}: rel err {rel:.2e}, "
              f"cycles 1 gemm {int(cyc[0])}, 8 gemms {int(cyc[1])}")
    assert rel < (3e-5 if fmt else 2e-6), rel
    # exact-A form: A already representable in 16 bits, two MMAs
    A16 = A.bfloat16().float() if fmt else A.half().float()
    ops._call("kpf_umma_split_selftest", ops._p(A16), ops._p(B), ops._p(D), N, K, fmt, a_tmem, 1, None)
    torch.cuda.synchronize()
    ref = (A16.double() @ B.double().t())
    assert float((D.double() - ref).norm() / ref.norm()) < (3e-5 if fmt else 2e-6)

