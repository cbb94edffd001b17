"""Density feature gather with 16 channels per plane (vm_density16_fwd_kernel, vm_gather.cu) at the benchmark's field
sizes: sigma_feature against a float64 evaluation of the same bilinear x linear sums.

The reference takes the tap positions and weights in fp32 exactly as the kernel forms them (ATen grid_sampler,
align_corners=True: x = (u + 1) * (0.5 (n - 1)), floor, fraction, 1 - fraction; the plane weight is the fp32 product
of the two axis weights), so that what is left is the rounding of the channel sums."""
import pytest
import torch

import joint_tensorf_b200 as jt
from joint_tensorf_b200 import ops
from vm_reference import density_feature

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


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
    val, mag = density_feature(ref_fs.planes, ref_fs.lines, u)
    got = out[:n].double()
    assert torch.isfinite(got).all()
    rel = float(((got - val).abs() / mag.clamp_min(1e-30)).max())
    assert rel <= 1e-6, rel
    assert torch.isnan(out[n:]).all()          # nothing written past the device-side count
