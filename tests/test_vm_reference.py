"""The float64 VM reference (tests/vm_reference.py) against float64 autograd of the oracle's F.grid_sample
evaluation (vo.density_feature / vo.app_components) on the golden grids: forward, the six factor gradients and the
per-sample coordinate gradient agree to 1e-12 of the sum of absolute terms. Runs on the CPU.

The samples include exact lattice points, u = +-1 and points just outside [-1, 1] (a point on the aabb face can
normalise to 1 +- 1 ulp), where the one-sided derivative the kernels take must be the one ATen takes."""
import math
from types import SimpleNamespace

import pytest
import torch

from common import load_golden, vo
from vm_reference import MAT, VEC, vm_adjoint

CASES = ["cubic_blur", "noncubic_blur", "cubic_mlp", "ndc_weakview"]    # 8/12, 8/12 non-cubic, 16/48, 16/20
TOL = 1e-12


def _samples(grid, n_rand, gen):
    u = torch.rand((n_rand, 3), dtype=torch.float64, generator=gen) * 2 - 1
    pts = [u]
    for a in range(3):                       # lattice points, the faces and just outside them on every axis
        n = grid[a]
        lat = -1.0 + 2.0 * torch.arange(n, dtype=torch.float64) / (n - 1)
        edge = torch.tensor([-1.0, 1.0, math.nextafter(1.0, 2.0), math.nextafter(-1.0, -2.0),
                             math.nextafter(1.0, 0.0), math.nextafter(-1.0, 0.0), 1.0 + 1e-7, -1.0 - 1e-7, 1.05, -1.05,
                             1.0 + 2.0 / (n - 1), -1.0 - 2.0 / (n - 1), 3.0, -3.0], dtype=torch.float64)
        for vals in (lat, edge):
            v = torch.rand((vals.shape[0], 3), dtype=torch.float64, generator=gen) * 2 - 1
            v[:, a] = vals
            pts.append(v)
    lat3 = torch.stack([(-1.0 + 2.0 * torch.randint(0, grid[a], (64,), generator=gen).double() / (grid[a] - 1))
                        for a in range(3)], 1)               # lattice points on all three axes at once
    pts.append(lat3)
    return torch.cat(pts)


@pytest.mark.parametrize("prefix", ["density", "app"])
@pytest.mark.parametrize("name", CASES)
def test_reference_matches_float64_autograd(name, prefix):
    g = load_golden(name)
    grid = list(g["case"]["grid"])
    gen = torch.Generator().manual_seed(7)
    sd = g["state_dict"]
    params = {k: v.detach().double().clone().requires_grad_(True) for k, v in sd.items()}
    field = SimpleNamespace(params=params)
    u = _samples(grid, 500, gen).requires_grad_(True)
    n = u.shape[0]
    fn = vo.density_feature if prefix == "density" else vo.app_components
    out = fn(field, None, u)
    gin = torch.randn(out.shape, dtype=torch.float64, generator=gen)
    (out * gin).sum().backward()

    planes = [params[f"{prefix}_plane.{i}"].detach()[0].permute(1, 2, 0) for i in range(3)]    # [H,W,C]
    lines = [params[f"{prefix}_line.{i}"].detach()[0, :, :, 0].t() for i in range(3)]         # [L,C]
    for i in range(3):   # the layout the reference assumes: plane i is [g[MAT[i][1]], g[MAT[i][0]]], line i g[VEC[i]]
        assert planes[i].shape[:2] == (grid[MAT[i][1]], grid[MAT[i][0]]) and lines[i].shape[0] == grid[VEC[i]]
    S, n_rays = 16, (n + 15) // 16
    samp = torch.zeros((n, 4), dtype=torch.float64)
    samp[:, :3] = u.detach()
    samp[:, 3] = torch.rand(n, dtype=torch.float64, generator=gen) * 4
    sidx = torch.arange(n, dtype=torch.int32)                # ray e // 16
    inv = (0.5, 0.75, 2.0)
    r = vm_adjoint(planes, lines, samp, gin=gin, sidx=sidx, S=S, n_rays=n_rays, inv=inv, tap_dtype="float64")

    def check(what, got, ref, mag):
        err = (got - ref).abs()
        bad = err > TOL * mag
        assert not bad.any(), (what, float((err / mag.clamp_min(1e-300)).max()), int(bad.sum()))

    check("value", r.value, out.detach(), r.value_mag)
    for i in range(3):
        check(f"plane {i}", r.gp[i], params[f"{prefix}_plane.{i}"].grad[0].permute(1, 2, 0), r.gp_mag[i])
        check(f"line {i}", r.gl[i], params[f"{prefix}_line.{i}"].grad[0, :, :, 0].t(), r.gl_mag[i])
    check("du", r.du, u.grad, r.du_mag)
    invt = torch.tensor(inv, dtype=torch.float64)
    ray = torch.arange(n) // S
    d_o = torch.zeros((n_rays, 3), dtype=torch.float64).index_add_(0, ray, u.grad * invt)
    d_d = torch.zeros((n_rays, 3), dtype=torch.float64).index_add_(0, ray, u.grad * samp[:, 3:] * invt)
    check("d_o", r.d_o, d_o, r.d_o_mag)
    check("d_d", r.d_d, d_d, r.d_d_mag)
    # the reference is not trivially satisfied: every output has terms, and the edge samples reach the zero padding
    assert all(float(x.abs().max()) > 0 for x in (r.value, r.du, *r.gp, *r.gl))
    assert float(r.du_mag.max()) > 0


def test_fp32_taps_match_float64_taps_on_dyadic_samples():
    """On samples whose positions are exact in fp32 both tap modes give the same reference."""
    gen = torch.Generator().manual_seed(3)
    planes = [torch.randn((17, 33, 8), generator=gen), torch.randn((65, 33, 8), generator=gen),
              torch.randn((65, 17, 8), generator=gen)]          # grid [33, 17, 65]
    lines = [torch.randn((65, 8), generator=gen), torch.randn((17, 8), generator=gen), torch.randn((33, 8), generator=gen)]
    n = 3000
    samp = torch.zeros((n, 4))
    samp[:, :3] = torch.randint(-70, 71, (n, 3), generator=gen).float() / 64      # includes the out-of-range band
    gin = torch.randn((n, 24), generator=gen)
    a = vm_adjoint(planes, lines, samp, gin=gin, tap_dtype="fp32")
    b = vm_adjoint(planes, lines, samp, gin=gin, tap_dtype="float64")
    for x, y in [(a.value, b.value), (a.du, b.du)] + list(zip(a.gp, b.gp)) + list(zip(a.gl, b.gl)):
        assert torch.equal(x, y)
