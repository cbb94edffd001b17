"""The tcgen05 MMA plumbing the tensor-core kernels share (jt_tc_selftest: shared-memory operand layouts, UMMA
descriptors, fp16 operands) against torch matrix products."""
import pytest
import torch

from joint_tensorf_b200 import ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _bf(x):
    return x.to(torch.bfloat16).float()


@pytest.mark.parametrize("k,n", [(16, 16), (144, 32), (160, 64), (80, 64), (64, 160)])
def test_umma_kmajor(k, n):
    g = torch.Generator().manual_seed(0)
    a = torch.randn(128, k, generator=g).to(DEV)
    b = torch.randn(n, k, generator=g).to(DEV)
    d = ops.tc_selftest(0, a, b, k, n)
    ref = _bf(a) @ _bf(b).T
    assert (d - ref).abs().max() <= 1e-3 * ref.abs().max(), float((d - ref).abs().max())


@pytest.mark.parametrize("ma,n", [(64, 80), (32, 144), (8, 80), (64, 160)])
def test_umma_mnmajor(ma, n):
    g = torch.Generator().manual_seed(1)
    x = torch.randn(128, ma, generator=g).to(DEV)
    y = torch.randn(128, n, generator=g).to(DEV)
    d = ops.tc_selftest(1, x, y, 128, n, ma)
    ref = _bf(x).T @ _bf(y)
    assert (d[:ma] - ref).abs().max() <= 1e-3 * ref.abs().max(), float((d[:ma] - ref).abs().max())
    assert float(d[ma:].abs().max()) == 0.0


@pytest.mark.parametrize("k,n", [(144, 32), (32, 16)])
def test_umma_kmajor_fp16_operands(k, n):
    g = torch.Generator().manual_seed(2)
    a = torch.randn(128, k, generator=g).to(DEV)
    b = torch.randn(n, k, generator=g).to(DEV)
    d = ops.tc_selftest(2, a, b, k, n)
    ref = a.half().float() @ b.half().float().T
    assert (d - ref).abs().max() <= 1e-5 * ref.abs().max() + 1e-5, float((d - ref).abs().max())
    full = a @ b.T
    assert (d - full).abs().max() <= 2e-3 * full.abs().max()

