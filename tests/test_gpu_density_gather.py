"""Density feature gather with 16 channels per plane (vm_density16_fwd_kernel, vm_gather.cu) at the benchmark's field
sizes: sigma_feature against a float64 evaluation of the same bilinear x linear sums.

The reference takes the tap positions and weights in fp32 exactly as the kernel forms them (ATen grid_sampler,
align_corners=True: x = (u + 1) * (0.5 (n - 1)), floor, fraction, 1 - fraction; the plane weight is the fp32 product
of the two axis weights), so that what is left is the rounding of the channel sums."""
import pytest
import torch

import joint_tensorf_b200 as jt
from joint_tensorf_b200 import ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MAT = ((0, 1), (0, 2), (1, 2))
VEC = (2, 1, 0)


def _axis(g, n):
    """fp32 tap setup of make_tap (jt_common.cuh): clamped indices and weights (0 for out-of-range taps)"""
    scale = torch.tensor(0.5 * (n - 1), dtype=torch.float32, device=g.device)
    x = (g + 1.0) * scale
    xf = torch.floor(x)
    f = x - xf
    i0 = torch.clamp(xf, -2.0, float(n)).to(torch.int64)
    i1 = i0 + 1
    m0 = ((i0 >= 0) & (i0 < n)).float()
    m1 = ((i1 >= 0) & (i1 < n)).float()
    return i0.clamp(0, n - 1), i1.clamp(0, n - 1), (1.0 - f) * m0, f * m1


def _reference(fs, u):
    """float64 sum_i sum_c P_ic(u) L_ic(u) and sum_i sum_c |P_ic(u) L_ic(u)| with fp32 tap weights"""
    val = torch.zeros(u.shape[0], dtype=torch.float64, device=DEV)
    mag = torch.zeros_like(val)
    for i in range(3):
        P, L = fs.planes[i].double(), fs.lines[i].double()          # [H,W,C], [L,C]
        H, W, _ = fs.planes[i].shape
        x0, x1, wx0, wx1 = _axis(u[:, MAT[i][0]], W)
        y0, y1, wy0, wy1 = _axis(u[:, MAT[i][1]], H)
        l0, l1, wl0, wl1 = _axis(u[:, VEC[i]], L.shape[0])
        w = [(wx0 * wy0), (wx1 * wy0), (wx0 * wy1), (wx1 * wy1)]    # fp32 products, as the kernel forms them
        pv = (P[y0, x0] * w[0].double()[:, None] + P[y0, x1] * w[1].double()[:, None] +
              P[y1, x0] * w[2].double()[:, None] + P[y1, x1] * w[3].double()[:, None])
        lv = L[l0] * wl0.double()[:, None] + L[l1] * wl1.double()[:, None]
        val += (pv * lv).sum(1)
        mag += (pv * lv).abs().sum(1)
    return val, mag


def _batch(wl):
    kw, run = jt.synth.config(wl)
    kw = dict(kw)
    ndc = bool(run["ndc"])
    if ndc:
        kw["near_far"] = [-1.0, 1.0]
    torch.manual_seed(0)
    m = jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), DEV, **kw)
    S = run["n_samples"]
    o, d, _ = jt.synth.llff_ndc_rays(4096, 1) if ndc else jt.synth.blender_rays(4096, 1)
    o, d = o.to(DEV).contiguous(), d.to(DEV).contiguous()
    if ndc:
        aux = m._ndc_table(S, False).contiguous()
    else:
        aux = torch.rand((o.shape[0],), generator=torch.Generator().manual_seed(1)).to(DEV).contiguous()
    comp = ops.march_compact(o, d, aux, ndc, S, m._h_geom(), None)
    gen = torch.Generator(device=DEV).manual_seed(2)
    planes = [torch.randn(p.shape, device=DEV, generator=gen) * 0.3 for p in m.density_plane]
    lines = [torch.randn(p.shape, device=DEV, generator=gen) * 0.3 for p in m.density_line]
    return comp, ops.FactorSet(planes, lines)


@pytest.mark.parametrize("bf16_factors", [False, True])
@pytest.mark.parametrize("wl", ["cfg2_sh", "cfg4"])
def test_density_feature_matches_float64_evaluation(wl, bf16_factors):
    comp, fs = _batch(wl)
    assert all(c == 16 for c in fs.C)
    n = int(comp.count.item())
    assert n > 100000, n
    if bf16_factors:
        fs = fs.with_bf16_store()
    out = torch.full((comp.cap,), float("nan"), device=DEV)
    ops.vm_gather_fwd(0, fs, comp.samp, None, comp.count, comp.cap, out)
    torch.cuda.synchronize()
    ref_fs = fs
    if bf16_factors:   # the kernel reads the bf16 copy: evaluate the reference on those values
        ref_fs = ops.FactorSet([s.float().permute(2, 0, 1)[None] for s in fs.store[:3]],
                               [s.float().t()[None, :, :, None] for s in fs.store[3:]])
    u = comp.samp[:n, :3]
    val, mag = _reference(ref_fs, u)
    got = out[:n].double()
    assert torch.isfinite(got).all()
    rel = float(((got - val).abs() / mag.clamp_min(1e-30)).max())
    assert rel <= 1e-6, rel
    assert torch.isnan(out[n:]).all()          # nothing written past the device-side count
