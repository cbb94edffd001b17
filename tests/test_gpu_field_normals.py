"""Field geometry queries on the GPU: the density gradient at points (jt_field_density_grad through
B200_VMSplit.compute_density_grad) against a float64 autograd reference, its agreement with jt_field_alpha and
jt_vm_gather_bwd, unit normals (compute_normals), normal maps (render_normals) against the no-grad forward and a
float64 composite, and extract_mesh(colors=True, normal_source="field")."""
import pytest
import torch

import joint_tensorf_b200 as jt
from common import field_from_golden, golden_names, load_golden
from density_grad_reference import density_and_grad, lattice_coords, outward_normals, safe_points
from gpu_common import default_opt, forward_kwargs, module_from_golden, record_err
from joint_tensorf_b200 import ops
from oracle import vm_oracle as vo

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SIGMA_RTOL = 1e-5        # sigma, relative to the largest sigma and to itself (where it exceeds 1e-3 of the largest)
GRAD_TOL = 1e-4          # grad, relative to the largest |grad| entry
NMAP_TOL = 1e-4          # normal map against the float64 composite, absolute


def _synthetic(grid, comps, aabb, act, seed=0, shift=None):
    torch.manual_seed(seed)
    kw = dict(density_n_comp=comps, appearance_n_comp=[8] * 3, app_dim=27, shadingMode="SH", fea2denseAct=act,
              density_shift=(-10 if act == "softplus" else 0.0) if shift is None else shift, volume_init_scale=0.1,
              volume_init_bias=0.1 if act == "softplus" else 0.2, step_ratio=0.5)
    return jt.B200_VMSplit(torch.tensor(aabb, dtype=torch.float32), list(grid), DEV, **kw)


def _reference(m, xyz, planes=None, lines=None, keep=None):
    planes = [p for p in m.density_plane] if planes is None else planes
    lines = [l for l in m.density_line] if lines is None else lines
    return density_and_grad(planes, lines, m.aabb.cpu(), xyz.cpu(), float(m.density_shift), m.fea2denseAct,
                            inv=m._h_inv, keep=keep, grid=m._grid)


def _compare(tag, sigma, grad, ref_s, ref_g):
    sigma, grad = sigma.double().cpu(), grad.double().cpu()
    s_scale = float(ref_s.abs().max())
    s_err = float((sigma - ref_s).abs().max()) / max(s_scale, 1e-30)
    s_elem = float(((sigma - ref_s).abs() / ref_s.abs().clamp_min(1e-30))[ref_s.abs() > 1e-3 * s_scale].max())
    g_scale = float(ref_g.abs().max())
    g_err = float((grad - ref_g).abs().max()) / max(g_scale, 1e-30)
    record_err(f"density_grad[{tag}]", sigma_rel_to_max=s_err, sigma_rel_elementwise=s_elem, grad_rel_to_max=g_err,
               grad_max=g_scale)
    assert s_err <= SIGMA_RTOL and s_elem <= SIGMA_RTOL, (tag, s_err, s_elem)
    assert g_err <= GRAD_TOL, (tag, g_err)
    return s_err, g_err


def _outside(m, n, seed):
    g = torch.Generator().manual_seed(seed)
    lo, hi = m.aabb[0].cpu(), m.aabb[1].cpu()
    p = lo + (hi - lo) * torch.rand(n, 3, generator=g)
    p[:, 1] = torch.where(torch.rand(n, generator=g) < 0.5, lo[1] - 0.3 * (hi[1] - lo[1]), hi[1] + 0.3 * (hi[1] - lo[1]))
    return p


SYNTH = [  # (tag, grid, comps, aabb, act)
    ("cubic16_softplus", (32, 32, 32), [16] * 3, [[-1.5] * 3, [1.5] * 3], "softplus"),
    ("noncubic16_relu", (40, 24, 56), [16] * 3, [[-1.5, -1.67, -2.0], [1.5, 1.67, 1.0]], "relu"),
    ("noncubic8_softplus", (24, 32, 20), [8] * 3, [[-1.0, -0.5, -2.0], [1.5, 0.5, 1.0]], "softplus"),
    ("cubic48_relu", (20, 20, 20), [48] * 3, [[-1.5] * 3, [1.5] * 3], "relu"),
    ("mixed_16_8_12_softplus", (18, 22, 26), [16, 8, 12], [[-1.0] * 3, [1.0, 1.2, 0.8]], "softplus"),
]


@pytest.mark.parametrize("tag,grid,comps,aabb,act", SYNTH, ids=[s[0] for s in SYNTH])
def test_density_grad_against_float64(tag, grid, comps, aabb, act):
    m = _synthetic(grid, comps, aabb, act, seed=1)
    gen = torch.Generator().manual_seed(2)
    xyz = torch.cat([safe_points(m.aabb.cpu(), grid, 6000, gen), _outside(m, 200, 3)]).to(DEV)
    sigma, grad = m.compute_density_grad(xyz)
    assert sigma.shape == (xyz.shape[0],) and grad.shape == (xyz.shape[0], 3)
    ref_s, ref_g = _reference(m, xyz)
    _compare(tag, sigma, grad, ref_s, ref_g)
    out = slice(6000, None)              # outside the aabb on y: no tap in range
    assert float(grad[out].abs().max()) == 0.0


def test_density_grad_300_cubed():
    kw, _ = jt.synth.config("cfg2_sh")
    kw = dict(kw)
    torch.manual_seed(0)
    m = jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), DEV, **kw)
    xyz = safe_points(m.aabb.cpu(), m._grid, 4000, torch.Generator().manual_seed(5)).to(DEV)
    sigma, grad = m.compute_density_grad(xyz)
    _compare("cfg2_sh_300^3", sigma, grad, *_reference(m, xyz))


def test_density_grad_with_alpha_mask():
    m = _synthetic((30, 26, 34), [16] * 3, [[-1.2, -1.0, -1.5], [1.2, 1.4, 1.0]], "softplus", seed=4)
    g = torch.Generator().manual_seed(6)
    vol = (torch.rand((9, 8, 7), generator=g) < 0.4).float()
    m.alphaMask = jt.AlphaGridMask(DEV, m.aabb.clone(), vol.to(DEV))
    xyz = safe_points(m.aabb.cpu(), m._grid, 6000, torch.Generator().manual_seed(7)).to(DEV)
    keep = vo.alpha_mask_lookup(vol, m.aabb.cpu(), xyz.cpu()) > 0
    assert 0 < int(keep.sum()) < keep.numel()
    sigma, grad = m.compute_density_grad(xyz)
    k = keep.to(DEV)
    assert float(sigma[~k].abs().max()) == 0.0 and float(grad[~k].abs().max()) == 0.0
    _compare("alpha_mask", sigma, grad, *_reference(m, xyz, keep=keep))
    assert float(m.compute_normals(xyz)[~k].abs().max()) == 0.0


def _golden_reference(m, g, xyz):
    """The float64 reference on the golden field as compute_density_grad sees it (cached blur, mask)."""
    field = field_from_golden(g, requires_grad=False)
    field.params = {k: v.double() for k, v in field.params.items()}
    fc = vo.grid_constants(field.aabb, field.grid, field.step_ratio)
    taps = None
    if g["case"]["blur"] is not None:
        taps = vo.blur_taps(fc, "uniform-gaussian", g["case"]["blur"][0], 64)
    pl = vo._factors(field, fc, "density", taps)
    keep = None
    if g["mask_volume"] is not None:
        keep = vo.alpha_mask_lookup(g["mask_volume"], g["aabb"], xyz.cpu()) > 0
    return _reference(m, xyz, [p for p, _ in pl], [l for _, l in pl], keep)


def _forward_nograd(m, g, o, d):
    kw = forward_kwargs(g, DEV)
    kw.update(is_train=False)
    kw.pop("jitter", None)
    with torch.no_grad():
        return m.forward(default_opt(g["case"]["shading"], g["case"].get("ndc", False)), o, d, **kw)


@pytest.mark.parametrize("name", golden_names())
def test_density_grad_golden_fields(name):
    g = load_golden(name)
    m = module_from_golden(g, DEV)
    if g["case"]["blur"] is not None:        # a forward with c2f_mode caches the density kernel
        _forward_nograd(m, g, g["rays_o"].to(DEV), g["rays_d"].to(DEV))
    xyz = safe_points(m.aabb.cpu(), m._grid, 5000, torch.Generator().manual_seed(11)).to(DEV)
    sigma, grad = m.compute_density_grad(xyz)
    _compare(f"golden_{name}", sigma, grad, *_golden_reference(m, g, xyz))
    # against jt_field_alpha: 1 - exp(-sigma * len), same taps and summation order
    length = float(m._h_step)
    a_ref = m.compute_alpha(xyz, length)
    a_new = 1.0 - torch.exp(-sigma * length)
    err = float((a_new - a_ref).abs().max())
    record_err(f"density_grad_vs_alpha[{name}]", err=err, bitwise_sigma_path=int(err == 0.0))
    assert err <= 2e-7, err


@pytest.mark.parametrize("name", ["cubic_mlp", "noncubic_blur", "sh"])
def test_density_grad_matches_the_gather_backward(name):
    """grad / (act' * inv) against jt_vm_gather_bwd's dsamp with gin = 1 (the coordinate gradient of the feature),
    and the compacted-sample form through a slot list against the explicit-point form."""
    g = load_golden(name)
    m = module_from_golden(g, DEV)
    xyz = safe_points(m.aabb.cpu(), m._grid, 3000, torch.Generator().manual_seed(12)).to(DEV)
    n = xyz.shape[0]
    fs = m._density_factorset()
    u = m.normalize_coord(xyz)
    samp = ops._samp_from_xyz(u)
    feat = torch.empty((n,), device=DEV)
    ops.vm_gather_fwd(0, fs, samp, None, None, n, feat)
    gp, gl = fs.zero_grads()
    dsamp = torch.zeros_like(samp)
    ops.vm_gather_bwd(0, fs, gp, gl, samp, None, None, n, torch.ones((n,), device=DEV), dsamp, 0)
    _, grad = m.compute_density_grad(xyz)
    x = (feat + m.density_shift).double()
    dact = torch.sigmoid(x) if m.fea2denseAct == "softplus" else (x > 0).double()
    inv = m._h_inv.to(DEV).double()
    ok = dact > 0
    du = grad.double()[ok] / (dact[ok, None] * inv)
    ref = dsamp[:n, :3].double()[ok]
    err = float((du - ref).abs().max() / ref.abs().max())
    record_err(f"density_grad_vs_gather_bwd[{name}]", err=err)
    assert err <= 1e-6, err
    # compacted samples through a slot list: the same values as explicit points
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(3)).to(DEV).int()
    cnt = torch.tensor([n], device=DEV, dtype=torch.int32)
    s2, g2 = ops.field_density_grad(fs, m._h_geom(), m.density_shift, 0 if m.fea2denseAct == "softplus" else 1,
                                    samp=samp, slot=perm, n_dev=cnt, n_max=n)
    s1, g1 = ops.field_density_grad(fs, m._h_geom(), m.density_shift, 0 if m.fea2denseAct == "softplus" else 1,
                                    samp=samp, n_max=n)
    assert torch.equal(s2, s1[perm.long()]) and torch.equal(g2, g1[perm.long()])


def test_density_grad_is_deterministic_and_order_independent():
    m = _synthetic((32, 32, 32), [16] * 3, [[-1.5] * 3, [1.5] * 3], "softplus", seed=8)
    xyz = safe_points(m.aabb.cpu(), m._grid, 10000, torch.Generator().manual_seed(9)).to(DEV)
    s, gr = m.compute_density_grad(xyz)
    s2, gr2 = m.compute_density_grad(xyz)
    assert torch.equal(s, s2) and torch.equal(gr, gr2)
    perm = torch.randperm(xyz.shape[0], generator=torch.Generator().manual_seed(1)).to(DEV)
    s3, gr3 = m.compute_density_grad(xyz[perm])
    assert torch.equal(s3, s[perm]) and torch.equal(gr3, gr[perm])
    s4, gr4 = m.compute_density_grad(xyz[:37].view(37, 1, 3))
    assert s4.shape == (37, 1) and gr4.shape == (37, 1, 3)
    assert torch.equal(s4.view(-1), s[:37]) and torch.equal(gr4.view(-1, 3), gr[:37])
    s0, g0 = m.compute_density_grad(torch.zeros((0, 3), device=DEV))
    assert s0.shape == (0,) and g0.shape == (0, 3)


def test_normals_are_unit_and_zero_where_the_gradient_vanishes():
    m = _synthetic((24, 30, 20), [8] * 3, [[-1.0, -0.5, -2.0], [1.5, 0.5, 1.0]], "relu", seed=10)
    xyz = torch.cat([safe_points(m.aabb.cpu(), m._grid, 8000, torch.Generator().manual_seed(13)),
                     _outside(m, 100, 4)]).to(DEV)
    _, grad = m.compute_density_grad(xyz)
    nrm = m.compute_normals(xyz)
    nz = (grad != 0).any(dim=1)
    assert 0 < int(nz.sum()) < nz.numel()         # relu: zero gradient where the pre-activation is negative
    assert float(nrm[~nz].abs().max()) == 0.0
    err = float((nrm[nz].double().norm(dim=1) - 1).abs().max())
    record_err("normals_unit_length", err=err)
    assert err <= 1e-6
    ref = outward_normals(grad[nz].double().cpu())
    assert float((nrm[nz].double().cpu() - ref).abs().max()) <= 1e-6


def test_normals_point_away_from_a_blob():
    """One channel per plane set to a separable bump: feat = 3 b(x) b(y) b(z), a blob at c; on shells around c the
    normals point away from c."""
    grid = (40, 40, 40)
    m = _synthetic(grid, [4] * 3, [[-1.0] * 3, [1.0] * 3], "softplus", seed=0, shift=-2.0)
    c = torch.tensor([0.1, -0.15, 0.2])
    t = torch.linspace(-1, 1, 40)
    with torch.no_grad():
        for i in range(3):
            m0, m1 = ops.MAT_MODE[i]
            a = ops.VEC_MODE[i]
            bx, by, bl = (torch.exp(-((t - c[k]) / 0.4) ** 2) for k in (m0, m1, a))
            m.density_plane[i].zero_()
            m.density_line[i].zero_()
            m.density_plane[i][0, 0] = (by[:, None] * bx[None, :]).to(DEV)
            m.density_line[i][0, 0, :, 0] = bl.to(DEV)
    g = torch.Generator().manual_seed(14)
    d = torch.randn(3000, 3, generator=g)
    d = d / d.norm(dim=1, keepdim=True)
    r = 0.15 + 0.35 * torch.rand(3000, 1, generator=g)
    xyz = (c + r * d).to(DEV)
    nrm = m.compute_normals(xyz)
    cos = (nrm.cpu().double() * d.double()).sum(dim=1)
    record_err("normals_blob", min_cos=float(cos.min()), median_cos=float(cos.median()))
    # the bumps are piecewise linear between texels: in the cell holding a bump's peak its slope can point either way
    assert float(cos.min()) > 0.9 and float(cos.median()) > 0.99


def _nmap_reference(m, g, o, d):
    """float64 composite: oracle weights of vo.render(exact=True) x reference normals at the samples."""
    field = field_from_golden(g, requires_grad=False)
    field.params = {k: v.double() for k, v in field.params.items()}
    if field.mask_volume is not None:            # exact mode looks the mask up at float64 points
        field.mask_volume, field.mask_aabb = field.mask_volume.double(), field.mask_aabb.double()
    case = g["case"]
    ndc = case.get("ndc", False)
    kw = dict(n_samples=g["n_samples"], white_bg=not ndc, ndc=ndc)
    if case["blur"] is not None:
        kw.update(blur_mode="uniform-gaussian", blur_density=case["blur"][0], blur_color=case["blur"][1], kernel_size=64)
    with torch.no_grad():
        _, _, _, det = vo.render(field, o.cpu(), d.cpu(), exact=True, detail=True, **kw)
    w, pts, valid = det["weight"], det["pts"], det["valid"]
    fc = vo.grid_constants(field.aabb, field.grid, field.step_ratio)
    pl = vo._factors(field, fc, "density", det["taps_d"])
    _, grad = _reference(m, pts[valid], [p for p, _ in pl], [l for _, l in pl])
    n_s = torch.zeros(pts.shape, dtype=torch.float64)
    n_s[valid] = outward_normals(grad)
    return (w[..., None] * n_s).sum(dim=1), pts[valid], w[valid]


@pytest.mark.parametrize("name", golden_names())
def test_render_normals_matches_forward_and_float64(name):
    g = load_golden(name)
    m = module_from_golden(g, DEV)
    o, d = g["rays_o"].to(DEV), g["rays_d"].to(DEV)
    ndc = g["case"].get("ndc", False)
    _, depth_f, acc_f = _forward_nograd(m, g, o, d)
    nmap, depth, acc = m.render_normals(o, d, ndc_ray=ndc, N_samples=g["n_samples"])
    assert torch.equal(depth, depth_f) and torch.equal(acc, acc_f)
    ref, pts, w = _nmap_reference(m, g, o, d)
    err = float((nmap.double().cpu() - ref).abs().max())
    c = lattice_coords(m.aabb.cpu(), m._grid, pts, inv=m._h_inv.double())
    frac = c - torch.floor(c)
    near_edge = torch.minimum(frac, 1 - frac).min(dim=1).values < 1e-4
    record_err(f"render_normals[{name}]", err=err, max_abs_ref=float(ref.abs().max()),
               weight_near_cell_edges=float(w[near_edge].sum()))
    assert err <= NMAP_TOL, err
    assert bool((nmap.norm(dim=1) <= acc * (1 + 1e-5) + 1e-6).all())
    # determinism and batch independence
    n2, d2, a2 = m.render_normals(o, d, ndc_ray=ndc, N_samples=g["n_samples"])
    assert torch.equal(n2, nmap) and torch.equal(d2, depth) and torch.equal(a2, acc)
    h = o.shape[0] // 2
    na, da, aa = m.render_normals(o[:h], d[:h], ndc_ray=ndc, N_samples=g["n_samples"])
    nb, db, ab = m.render_normals(o[h:], d[h:], ndc_ray=ndc, N_samples=g["n_samples"])
    assert torch.equal(torch.cat([na, nb]), nmap) and torch.equal(torch.cat([da, db]), depth)
    assert torch.equal(torch.cat([aa, ab]), acc)


@pytest.mark.parametrize("storage", ["fp32", "bf16"])
def test_render_normals_full_size_slices(storage):
    """cfg2_sh at 300^3: depth / opacity equal the no-grad forward's on a frame slice, in both factor storages."""
    kw, run = jt.synth.config("cfg2_sh")
    kw = dict(kw)
    torch.manual_seed(0)
    m = jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), DEV, **kw)
    m.factor_storage = storage
    o, d = jt.synth.frame_rays()
    o, d = o[320000:324096].to(DEV), d[320000:324096].to(DEV)
    with torch.no_grad():
        _, depth_f, acc_f = m.forward(default_opt("SH", False), o, d, white_bg=True, is_train=False,
                                      N_samples=run["n_samples"])
    nmap, depth, acc = m.render_normals(o, d, N_samples=run["n_samples"])
    assert torch.equal(depth, depth_f) and torch.equal(acc, acc_f)
    assert float(acc.max()) > 0 and bool(torch.isfinite(nmap).all())
    assert bool((nmap.norm(dim=1) <= acc * (1 + 1e-5) + 1e-6).all())


def test_render_normals_misses_and_empty_input():
    g = load_golden("cubic_mlp")
    m = module_from_golden(g, DEV)
    o = torch.tensor([[0.0, 0.0, 4.0], [5.0, 5.0, 5.0]], device=DEV)
    d = torch.tensor([[0.0, 0.0, 1.0], [1.0, 0.0, 0.0]], device=DEV)       # both pointing away from the box
    nmap, depth, acc = m.render_normals(o, d, N_samples=g["n_samples"])
    assert float(nmap.abs().max()) == 0.0 and float(acc.abs().max()) == 0.0
    _, depth_f, _ = _forward_nograd(m, g, o, d)
    assert torch.equal(depth, depth_f)
    e = torch.zeros((0, 3), device=DEV)
    n0, d0, a0 = m.render_normals(e, e, N_samples=g["n_samples"])
    assert n0.shape == (0, 3) and d0.shape == (0,) and a0.shape == (0,)


@pytest.mark.parametrize("name", ["alpha_mask", "noncubic_blur", "ndc_weakview"])
def test_extract_mesh_field_normals(name):
    g = load_golden(name)
    m = module_from_golden(g, DEV)
    m.head_precision = "fp32"
    if g["case"]["blur"] is not None:
        _forward_nograd(m, g, g["rays_o"].to(DEV), g["rays_d"].to(DEV))
    alpha = m._dense_alpha_zyx(m._grid)
    level = float(alpha.flatten().median())
    v0, f0, n0, c0 = m.extract_mesh(level, colors=True)
    v1, f1, n1, c1 = m.extract_mesh(level, colors=True, normal_source="lattice")
    assert torch.equal(v0, v1) and torch.equal(f0, f1) and torch.equal(n0, n1) and torch.equal(c0, c1)
    v, f, n, c = m.extract_mesh(level, colors=True, normal_source="field")
    assert v.shape[0] > 0
    assert torch.equal(v, v0) and torch.equal(f, f0)
    assert torch.equal(n, m.compute_normals(v))
    assert torch.equal(c, m.compute_rgb(v, -n))
    both = (n.norm(dim=1) > 0) & (n0.norm(dim=1) > 0)
    agree = float(((n * n0).sum(dim=1)[both] > 0).float().mean()) if bool(both.any()) else 1.0
    record_err(f"mesh_field_normals[{name}]", agree_with_lattice=agree)
    vg, fg = m.extract_mesh(level, normal_source="field")
    assert torch.equal(vg, v0) and torch.equal(fg, f0)
    with pytest.raises(jt._lib.JtError):
        m.extract_mesh(level, colors=True, normal_source="alpha")
