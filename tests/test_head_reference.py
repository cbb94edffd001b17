"""The float64 head reference (tests/head_reference.py) against float64 autograd of the oracle's shaders
(shade_sh / shade_mlp_fea / shade_weakview), with basis_mat as a Linear: values and every gradient to 1e-12, at PE
progress 1, 0.65 and 0 (masks [1, 1], [1, 0.3], [0, 0]), with and without normalised view directions of non-unit
rays. Also: every magnitude bounds its value, so that a bound stated on the magnitude is never tighter than the value
itself."""
from types import SimpleNamespace

import pytest
import torch
import torch.nn.functional as Fn

from head_reference import head_backward, head_forward, view_dirs
from oracle import vm_oracle as vo

F64 = torch.float64
# shading -> (components, app_dim, hidden, parameter names of (w1, b1, w2, b2, w3, b3))
HEADS = {
    "SH": (144, 27, 0, ()),
    "MLP_Fea": (144, 27, 64, tuple(f"renderModule.mlp.{i}.{k}" for i in (0, 2, 4) for k in ("weight", "bias"))),
    "MLP_Fea_WeakView": (60, 20, 32, tuple(f"renderModule.layer{i}.{k}" for i in (1, 2, 3)
                                           for k in ("weight", "bias"))),
}
PROGRESS = [(1.0, 1.0), (0.65, 0.65), (0.0, 0.0), (1.0, 0.65), (0.65, 0.0), (0.0, 1.0)]


def _inputs(shading, n, normalize_dir, seed=0):
    K, F, H, names = HEADS[shading]
    g = torch.Generator().manual_seed(seed)
    p = vo.init_params([8, 8, 8], [16] * 3, [K // 3] * 3, F, shading, max(H, 1), 2, 2, 0.1, 0.0, seed=seed)
    params = tuple(p[k].to(F64) for k in names)
    wb = p["basis_mat.weight"].to(F64)
    comps = torch.randn(n, K, generator=g, dtype=F64) * 0.3
    S, n_rays = 64, 29
    rays_d = torch.randn(n_rays, 3, generator=g, dtype=F64) * 1.7          # non-unit directions
    sidx = (torch.randint(0, n_rays, (n,), generator=g) * S + torch.randint(0, S, (n,), generator=g)).int()
    aidx = torch.randperm(n, generator=g).int()
    dirs = view_dirs(rays_d, sidx, aidx, n, S, normalize_dir)
    ray = (sidx[aidx.long()].long() // S)
    want = rays_d[ray] / rays_d[ray].norm(dim=1, keepdim=True) if normalize_dir else rays_d[ray]
    assert torch.equal(dirs, want)
    dout = torch.randn(n, 4, generator=g, dtype=F64)
    return params, names, wb, comps, dirs, dout


def _oracle(shading, names, params, wb, comps, dirs, fprog, vprog):
    """Oracle forward with basis_mat as a Linear; returns (feat, rgb, leaves)."""
    leaves = [t.clone().requires_grad_(True) for t in (comps, wb, *params)]
    c, w = leaves[0], leaves[1]
    field = SimpleNamespace(params=dict(zip(names, leaves[2:])), fea_pe=2, view_pe=2)
    feat = Fn.linear(c, w)
    shader = {"SH": vo.shade_sh, "MLP_Fea": vo.shade_mlp_fea, "MLP_Fea_WeakView": vo.shade_weakview}[shading]
    return feat, shader(field, dirs, feat, vprog, fprog), leaves


def _close(a, b, what):
    err = float((a - b).abs().max()) if a.numel() else 0.0
    assert err <= 1e-12 * max(1.0, float(b.abs().max()) if b.numel() else 0.0), (what, err)


@pytest.mark.parametrize("normalize_dir", [False, True])
@pytest.mark.parametrize("fprog,vprog", PROGRESS)
@pytest.mark.parametrize("shading", list(HEADS))
def test_reference_matches_oracle_autograd(shading, fprog, vprog, normalize_dir):
    params, names, wb, comps, dirs, dout = _inputs(shading, 300, normalize_dir)
    f = head_forward(shading, comps, dirs, wb, params, fprog, vprog)
    feat, rgb, leaves = _oracle(shading, names, params, wb, comps, dirs, fprog, vprog)
    _close(f.feat, feat.detach(), "feat")
    _close(f.rgb, rgb.detach(), "rgb")
    if shading == "SH":
        # rgb = relu(pre): dL/d rgb = dout where pre > 0; rows at pre <= 0 get dout = 0 (jt_render_bwd folds relu')
        dout[:, :3] = dout[:, :3] * (f.pre > 0)
        grad_rgb = dout[:, :3]
        _close(f.pre.clamp_min(0), rgb.detach(), "pre")
    else:
        # rgb = sigmoid(pre): dL/d rgb = dout / sigmoid'(pre)
        s = torch.sigmoid(f.pre)
        grad_rgb = dout[:, :3] / (s * (1 - s))
        _close(torch.sigmoid(f.pre), rgb.detach(), "pre")
    rgb.backward(grad_rgb)
    b = head_backward(f, dout)
    _close(b.dcomps, leaves[0].grad, "dcomps")
    _close(b.grads["wb"], leaves[1].grad, "wb")
    for key, leaf in zip(("w1", "b1", "w2", "b2", "w3", "b3"), leaves[2:]):
        _close(b.grads[key], leaf.grad, key)
    if shading != "SH":
        assert set(b.grads) == {"wb", "w1", "b1", "w2", "b2", "w3", "b3"}


@pytest.mark.parametrize("shading", list(HEADS))
def test_magnitudes_bound_values(shading):
    """|value| <= magnitude for every forward and backward output, and the ambiguous rows are the ones with a relu
    unit near 0 relative to its magnitude."""
    params, names, wb, comps, dirs, dout = _inputs(shading, 500, True, seed=1)
    amb = 2.0 ** -16
    f = head_forward(shading, comps, dirs, wb, params, 0.65, 0.65, amb=amb)
    b = head_backward(f, dout)
    pairs = [(f.feat, f.feat_mag), (f.pre, f.pre_mag), (b.dcomps, b.dcomps_mag), (b.dfeat, b.dfeat_mag)]
    pairs += [(b.grads[k], b.grads_mag[k]) for k in b.grads]
    for v, m in pairs:
        assert bool((v.abs() <= m * (1 + 1e-12)).all())
    if shading != "SH":
        near = (f.p1.abs() <= amb * f.p1_mag).any(1) | (f.p2.abs() <= amb * f.p2_mag).any(1)
        assert torch.equal(f.ambiguous, near)
        assert 0 < int(f.ambiguous.sum()) < 500          # this amb is coarse enough to flag some rows
    else:
        assert not bool(f.ambiguous.any())
