"""Tensor-core (tcgen05) shading-head kernels against plain fp32 torch."""
import pytest
import torch

import joint_tensorf_b200 as jt
from joint_tensorf_b200 import ops
from oracle import vm_oracle as vo

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


def _head_inputs(a_count, seed=0):
    g = torch.Generator().manual_seed(seed)
    p = vo.init_params([8, 8, 8], [16] * 3, [48] * 3, 27, "MLP_Fea", 64, 2, 2, 0.1, 0.0, seed=seed)
    comps = (torch.rand(a_count, 144, generator=g) * 0.05)
    n_rays, S = 37, 64
    rays_d = torch.randn(n_rays, 3, generator=g)
    sidx = (torch.randint(0, n_rays, (a_count,), generator=g) * S + torch.randint(0, S, (a_count,), generator=g)).int()
    aidx = torch.randperm(a_count, generator=g).int()
    return p, comps, rays_d, sidx, aidx, S


def _head_reference(p, comps, rays_d, sidx, aidx, S, fprog=1.0, vprog=1.0):
    field = vo.Field(aabb=torch.zeros(2, 3), grid=[8, 8, 8], params=p)
    feat = comps @ p["basis_mat.weight"].T
    dirs = rays_d[(sidx[aidx.long()] // S).long()]
    return vo.shade_mlp_fea(field, dirs, feat, vprog, fprog), feat


@pytest.mark.parametrize("split,tol", [(2, 3e-5), (1, 2e-2)])
@pytest.mark.parametrize("a_count", [1, 128, 1000, 20000])
def test_head_fwd_tc_matches_fp32(split, tol, a_count):
    p, comps, rays_d, sidx, aidx, S = _head_inputs(a_count)
    ref, feat_ref = _head_reference(p, comps, rays_d, sidx, aidx, S, 0.8, 0.6)
    d = {k: v.to(DEV).contiguous() for k, v in p.items()}
    rgb = torch.zeros((a_count, 4), device=DEV)
    feat = torch.zeros((a_count, 28), device=DEV)
    cnt = torch.tensor([a_count], device=DEV, dtype=torch.int32)
    ops.head_fwd_tc(split, comps.to(DEV), aidx.to(DEV), sidx.to(DEV), rays_d.to(DEV), S, False,
                    d["basis_mat.weight"], d["renderModule.mlp.0.weight"], d["renderModule.mlp.0.bias"],
                    d["renderModule.mlp.2.weight"], d["renderModule.mlp.2.bias"], d["renderModule.mlp.4.weight"],
                    d["renderModule.mlp.4.bias"], cnt, a_count + 500, 0.8, 0.6, rgb, feat)
    assert (feat[:, :27].cpu() - feat_ref).abs().max() <= tol * max(1.0, float(feat_ref.abs().max()))
    assert (rgb[:, :3].cpu() - ref).abs().max() <= tol
