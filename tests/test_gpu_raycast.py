"""Ray casting against the field's surface on the GPU (jt_raycast through B200_VMSplit.raycast / ops.raycast): the hit
predicate bit for bit against compute_alpha at the marcher's own sample points, the refinement replayed in fp32 with
compute_alpha as the predicate, agreement with a float64 ray caster, a blob of known geometry, the normal and colour
outputs, determinism, edge cases and full-size fields."""
import pytest
import torch

import joint_tensorf_b200 as jt
from common import golden_names, load_golden
from gpu_common import default_opt, forward_kwargs, module_from_golden, record_err
from joint_tensorf_b200 import ops
from oracle import vm_oracle as vo
from raycast_reference import cast64, field_alpha64, in_box64, refine

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
AERR_REL = 1e-5          # fp32 alpha against float64, relative to the level (sigma measured <= 6e-6 relative)
AERR_ABS = 2.0 ** -24    # plus the rounding of 1 - fl(exp(-sigma len)): half an ulp of values just below 1 is 2^-25


def _synthetic(grid, comps, aabb, act, seed=0, shift=None):
    torch.manual_seed(seed)
    kw = dict(density_n_comp=comps, appearance_n_comp=[8] * 3, app_dim=27, shadingMode="SH", fea2denseAct=act,
              density_shift=(-10 if act == "softplus" else 0.0) if shift is None else shift, volume_init_scale=0.1,
              volume_init_bias=0.1 if act == "softplus" else 0.2, step_ratio=0.5, near_far=[0.0, 10.0])
    return jt.B200_VMSplit(torch.tensor(aabb, dtype=torch.float32), list(grid), DEV, **kw)


SYNTH = [  # (tag, grid, comps, aabb, act): the fields of test_gpu_field_normals.py
    ("cubic16_softplus", (32, 32, 32), [16] * 3, [[-1.5] * 3, [1.5] * 3], "softplus"),
    ("noncubic16_relu", (40, 24, 56), [16] * 3, [[-1.5, -1.67, -2.0], [1.5, 1.67, 1.0]], "relu"),
    ("noncubic8_softplus", (24, 32, 20), [8] * 3, [[-1.0, -0.5, -2.0], [1.5, 0.5, 1.0]], "softplus"),
    ("cubic48_relu", (20, 20, 20), [48] * 3, [[-1.5] * 3, [1.5] * 3], "relu"),
    ("mixed_16_8_12_softplus", (18, 22, 26), [16, 8, 12], [[-1.0] * 3, [1.0, 1.2, 0.8]], "softplus"),
]


def _rays(aabb, n, seed):
    """Rays from outside the box through random points inside it, and a quarter starting inside the box."""
    g = torch.Generator().manual_seed(seed)
    lo, hi = torch.tensor(aabb[0]), torch.tensor(aabb[1])
    target = lo + (hi - lo) * torch.rand(n, 3, generator=g)
    d = torch.randn(n, 3, generator=g)
    d = d / d.norm(dim=1, keepdim=True) * (0.5 + torch.rand(n, 1, generator=g))    # not unit length
    back = torch.where(torch.arange(n)[:, None] % 4 == 0, torch.zeros(n, 1), (hi - lo).norm() * torch.ones(n, 1))
    o = target - back * d / d.norm(dim=1, keepdim=True)
    return o.to(DEV), d.to(DEV)


def _levels(m):
    a = m._dense_alpha_zyx(m._grid).reshape(-1).sort().values
    n = a.numel()
    return {q: min(max(float(a[int(q * (n - 1))]), 1e-30), 1.0 - 1e-6) for q in (0.5, 0.9)}


def _lanes(m):
    """Interior points per refinement round: 15 with 16 channels on every plane, else 7."""
    return 15 if all(int(c) == 16 for c in m.density_n_comp) else 7


def _cast(m, o, d, level, ndc, S, **kw):
    ztab = m._ndc_table(S, False).contiguous() if ndc else None
    return ops.raycast(m._density_factorset(), m._h_geom(), m.density_shift, 0 if m.fea2denseAct == "softplus" else 1,
                       float(m._h_step), level, o, d, S, ztab=ztab, mask=m.alphaMask, **kw)


def _samples(m, o, d, ndc, S):
    if ndc:
        pts, z, valid = m.sample_ray_ndc(o, d, is_train=False, N_samples=S)
        z = z.expand(o.shape[0], S)
    else:
        pts, z, valid = m.sample_ray(o, d, is_train=False, N_samples=S)
    return pts, z, valid.bool()


def _inside32(m, o, d, level, rows, t):
    """The kernel's predicate at o + d t (fp32, separately rounded): point_in_box and compute_alpha >= level."""
    p = o[rows, None, :] + d[rows, None, :] * t.to(DEV)[..., None]
    a0, a1 = m.aabb[0], m.aabb[1]
    inb = ~((a0 > p) | (p > a1)).any(dim=-1)
    a = torch.zeros(t.shape, device=DEV)
    if bool(inb.any()):
        a[inb] = m.compute_alpha(p[inb], float(m._h_step))
    return (inb & (a >= level)).cpu()


def check_bit_exact(m, o, d, level, ndc, S, tag):
    """Every hit point is o + d t and inside; every in-box sample before the hit (all of them on a miss) is outside; the
    refinement replayed in fp32 with compute_alpha gives the same t bit for bit. Returns (t, xyz, k, lo32)."""
    t, xyz, k, rounds = _cast(m, o, d, level, ndc, S, rounds=True)
    hit = k >= 0
    assert torch.equal(torch.isfinite(t), hit) and bool((t[~hit] == float("inf")).all())
    assert not bool(xyz[~hit].any())
    assert torch.equal(xyz[hit], o[hit] + d[hit] * t[hit][:, None])
    length = float(m._h_step)
    if bool(hit.any()):
        assert bool((m.compute_alpha(xyz[hit], length) >= level).all())
    pts, z, valid = _samples(m, o, d, ndc, S)
    alpha = torch.zeros(valid.shape, device=DEV)
    alpha[valid] = m.compute_alpha(pts[valid], length)
    inside = valid & (alpha >= level)
    idx = torch.arange(S, device=DEV)[None, :]
    before = idx < torch.where(hit, k, torch.full_like(k, S)).long()[:, None]
    assert not bool((inside & before).any()), tag
    kk = k.long().clamp_min(0)
    assert bool(inside[hit, kk[hit]].all()), tag
    # the refinement, replayed in fp32 with compute_alpha as the predicate
    ref = (k > 0).nonzero().squeeze(1)
    lo32 = t.clone()
    if ref.numel():
        lo_r, hi_r, rnd = refine(z[ref, kk[ref] - 1].cpu(), z[ref, kk[ref]].cpu(),
                                 lambda a, tt: _inside32(m, o, d, level, ref[a.to(DEV)], tt), _lanes(m))
        assert torch.equal(hi_r.to(DEV), t[ref]), tag
        assert torch.equal(rnd.to(DEV).int(), rounds[ref]), tag
        lo32[ref] = lo_r.to(DEV)
    assert bool((rounds[k <= 0] == 0).all())
    record_err(f"raycast_bit_exact[{tag}]", rays=int(k.numel()), hits=int(hit.sum()), starts_inside=int((k == 0).sum()),
               max_rounds=int(rounds.max()) if rounds.numel() else 0)
    return t, xyz, k, lo32


@pytest.mark.parametrize("tag,grid,comps,aabb,act", SYNTH, ids=[s[0] for s in SYNTH])
def test_bit_exact_synthetic(tag, grid, comps, aabb, act):
    m = _synthetic(grid, comps, aabb, act, seed=1)
    o, d = _rays(aabb, 1500, seed=2)
    for q, level in _levels(m).items():
        check_bit_exact(m, o, d, level, False, m.nSamples, f"{tag}_q{q}")


def _forward_nograd(m, g, o, d):
    kw = forward_kwargs(g, DEV)
    kw.update(is_train=False)
    kw.pop("jitter", None)
    with torch.no_grad():
        return m.forward(default_opt(g["case"]["shading"], g["case"].get("ndc", False)), o, d, **kw)


def _golden(name):
    g = load_golden(name)
    m = module_from_golden(g, DEV)
    if g["case"]["blur"] is not None:        # a forward with c2f_mode caches the density kernel
        _forward_nograd(m, g, g["rays_o"].to(DEV), g["rays_d"].to(DEV))
    return g, m


@pytest.mark.parametrize("name", golden_names())
def test_bit_exact_golden_fields(name):
    g, m = _golden(name)
    o, d = g["rays_o"].to(DEV), g["rays_d"].to(DEV)
    ndc = g["case"].get("ndc", False)
    for q, level in _levels(m).items():
        check_bit_exact(m, o, d, level, ndc, g["n_samples"], f"golden_{name}_q{q}")


def _against_float64(m, o, d, level, ndc, S, tag, keep_fn=None):
    t, xyz, k, lo32 = check_bit_exact(m, o, d, level, ndc, S, tag)
    planes, lines = m._blurred(m.density_plane, m.density_line, m.kernel_density if m.c2f_mode is not None else None)
    length = float(m._h_step)
    alpha_fn, grad_fn = field_alpha64(planes, lines, m.aabb.cpu(), float(m.density_shift), m.fea2denseAct, length,
                                      inv=m._h_inv, keep_fn=keep_fn)
    pts, z, valid = _samples(m, o, d, ndc, S)
    res = cast64(o.cpu(), d.cpu(), z.cpu(), pts.cpu(), valid.cpu(), alpha_fn, m.aabb.cpu(), level, _lanes(m))
    k32, k64 = k.long().cpu(), res["k"]
    aerr = AERR_REL * level + AERR_ABS
    # rays whose predicate fp32 and float64 may disagree on: a sample up to the later hit within aerr of the level
    upto = torch.maximum(torch.where(k32 < 0, S - 1, k32), torch.where(k64 < 0, S - 1, k64))
    near = ((res["alpha_samp"] - level).abs() <= aerr) & valid.cpu()
    near &= torch.arange(S)[None, :] <= upto[:, None]
    amb = near.any(dim=1)
    assert torch.equal(k32[~amb], k64[~amb]), (tag, int((k32[~amb] != k64[~amb]).sum()))
    # crossing depth: both hits in the same sample, refined
    both = (~amb & (k32 > 0)).nonzero().squeeze(1)
    t32 = t.cpu().double()[both]
    t_star = res["t_star"][both]
    width = (t.cpu().double() - lo32.cpu().double())[both]
    p_star = o.cpu().double()[both] + d.cpu().double()[both] * t_star[:, None]
    dadt = (grad_fn(p_star) * d.cpu().double()[both]).sum(dim=1).abs() if both.numel() else torch.zeros(0)
    zc = z.cpu()
    spacing = (zc[both, k32[both]] - zc[both, k32[both] - 1]).double()
    slack = 8.0 * aerr / dadt.clamp_min(1e-300)
    # the crossing is the aabb face where the ray enters (the field is above the level there): no alpha slope applies
    lo64 = o.cpu().double()[both] + d.cpu().double()[both] * res["lo"][both][:, None]
    box_face = ~in_box64(m.aabb.cpu(), lo64)
    grazing = ~box_face & (slack > spacing)
    tol = width + slack + 1e-6 * (1.0 + t32.abs())
    ok = ~grazing & ~box_face
    err = (t32 - t_star).abs()
    assert bool((err[ok] <= tol[ok]).all()), (tag, float((err - tol)[ok].max()))
    rel = float((err[ok] / spacing[ok]).max()) if bool(ok.any()) else 0.0
    record_err(f"raycast_vs_float64[{tag}]", rays=int(k32.numel()), k_checked=int((~amb).sum()),
               k_excluded_near_level=int(amb.sum()), t_checked=int(ok.sum()), t_excluded_grazing=int(grazing.sum()),
               t_excluded_box_face=int(box_face.sum()),
               max_abs_t_err=float(err[ok].max()) if bool(ok.any()) else 0.0, max_t_err_over_spacing=rel,
               max_bracket_over_spacing=float((width / spacing).max()) if both.numel() else 0.0)
    # fields whose alpha is a few fp32 ulps (random-init softplus at shift -10) leave many rays within 2^-24 of the level
    assert int((~amb).sum()) > 0, tag


@pytest.mark.parametrize("tag,grid,comps,aabb,act", SYNTH, ids=[s[0] for s in SYNTH])
def test_against_float64_synthetic(tag, grid, comps, aabb, act):
    m = _synthetic(grid, comps, aabb, act, seed=1)
    o, d = _rays(aabb, 400, seed=3)
    for q, level in _levels(m).items():
        _against_float64(m, o, d, level, False, m.nSamples, f"{tag}_q{q}")


@pytest.mark.parametrize("name", golden_names())
def test_against_float64_golden_fields(name):
    g, m = _golden(name)
    o, d = g["rays_o"].to(DEV), g["rays_d"].to(DEV)
    keep_fn = None
    if g["mask_volume"] is not None:
        vol, box = g["mask_volume"].double(), g["aabb"].double()
        keep_fn = lambda x: vo.alpha_mask_lookup(vol, box, x) > 0      # noqa: E731
    level = _levels(m)[0.5]
    _against_float64(m, o, d, level, g["case"].get("ndc", False), g["n_samples"], f"golden_{name}", keep_fn)


def _blob():
    """feat = 3 b(x) b(y) b(z), b(s) = exp(-((s - c) / 0.4)^2): level sets of feat are spheres of radius
    0.4 sqrt(ln(3 / feat)) around c (test_gpu_field_normals.test_normals_point_away_from_a_blob's field)."""
    grid = (40, 40, 40)
    m = _synthetic(grid, [4] * 3, [[-1.0] * 3, [1.0] * 3], "softplus", seed=0, shift=-2.0)
    c = torch.tensor([0.1, -0.15, 0.2])
    s = torch.linspace(-1, 1, 40)
    with torch.no_grad():
        for i in range(3):
            m0, m1 = ops.MAT_MODE[i]
            a = ops.VEC_MODE[i]
            bx, by, bl = (torch.exp(-((s - c[j]) / 0.4) ** 2) for j in (m0, m1, a))
            m.density_plane[i].zero_()
            m.density_line[i].zero_()
            m.density_plane[i][0, 0] = (by[:, None] * bx[None, :]).to(DEV)
            m.density_line[i][0, 0, :, 0] = bl.to(DEV)
    return m, c


def test_blob_known_geometry():
    m, c = _blob()
    r0 = 0.3
    feat = 3.0 * torch.exp(torch.tensor(-(r0 / 0.4) ** 2, dtype=torch.float64))
    sigma = torch.nn.functional.softplus(feat - 2.0)
    level = float(1.0 - torch.exp(-sigma * float(m._h_step)))
    g = torch.Generator().manual_seed(21)
    u = torch.randn(2000, 3, generator=g)
    u = u / u.norm(dim=1, keepdim=True)
    o = (c + 3.0 * u).to(DEV)
    d = (-u).to(DEV)
    hit, t, xyz, normal = m.raycast(o, d, level=level)
    assert bool(hit.all())
    h = 2.0 / 39                                   # texel spacing
    # the field interpolates each bump linearly between texels: |b - lerp(b)| <= h^2 / 8 |b''| <= 0.0041 b per
    # factor, about 0.02 of feat on the sphere, whose radial slope is 6.4: a radius error of ~0.003 = h / 16
    err = (t.double() - (3.0 - r0)).abs()
    record_err("raycast_blob", max_radius_err=float(err.max()), texel=h)
    assert float(err.max()) <= h / 8
    rad = (xyz.cpu() - c).double()
    cos = (normal.cpu().double() * rad / rad.norm(dim=1, keepdim=True)).sum(dim=1)
    record_err("raycast_blob_normals", min_cos=float(cos.min()))
    assert float(cos.min()) > 0.9
    verts, _ = m.extract_mesh(level)
    dist = torch.cdist(xyz, verts).min(dim=1).values
    record_err("raycast_blob_vs_mesh", max_dist=float(dist.max()), cell_diagonal=h * 3 ** 0.5)
    assert float(dist.max()) <= h * 3 ** 0.5


HEADS = [("sh_vm48", "tc"), ("cubic_mlp", "tc"), ("ndc_weakview", "tc"), ("cubic_blur", "fp32"), ("sh", "fp32")]


@pytest.mark.parametrize("name,head", HEADS)
def test_normal_and_colour_outputs(name, head):
    g, m = _golden(name)
    m.head_precision = head
    o, d = g["rays_o"].to(DEV), g["rays_d"].to(DEV)
    ndc = g["case"].get("ndc", False)
    level = _levels(m)[0.5]
    hit, t, xyz, normal, rgb = m.raycast(o, d, level=level, ndc_ray=ndc, N_samples=g["n_samples"], colors=True)
    assert bool(hit.any())
    assert torch.equal(normal[hit], m.compute_normals(xyz[hit])) and not bool(normal[~hit].any())
    viewdir = d / torch.linalg.vector_norm(d, dim=-1, keepdim=True) if ndc else d
    assert torch.equal(rgb[hit], m.compute_rgb(xyz[hit], viewdir[hit]))
    assert not bool(rgb[~hit].any())
    hit2, t2, xyz2, normal2 = m.raycast(o, d, level=level, ndc_ray=ndc, N_samples=g["n_samples"])
    assert torch.equal(hit2, hit) and torch.equal(t2, t) and torch.equal(xyz2, xyz) and torch.equal(normal2, normal)
    m.factor_storage = "bf16"              # geometry reads the fp32 factors whatever the storage
    out = m.raycast(o, d, level=level, ndc_ray=ndc, N_samples=g["n_samples"])
    assert all(torch.equal(a, b) for a, b in zip(out, (hit, t, xyz, normal)))


def test_deterministic_and_batch_independent():
    m = _synthetic((32, 32, 32), [16] * 3, [[-1.5] * 3, [1.5] * 3], "softplus", seed=8)
    o, d = _rays([[-1.5] * 3, [1.5] * 3], 3000, seed=9)
    level = _levels(m)[0.5]
    ref = _cast(m, o, d, level, False, m.nSamples)
    assert all(torch.equal(a, b) for a, b in zip(_cast(m, o, d, level, False, m.nSamples), ref))
    assert all(torch.equal(a, b) for a, b in zip(_cast(m, o, d, level, False, m.nSamples, counter=False), ref))
    h = 1234
    for a, b, r in zip(_cast(m, o[:h], d[:h], level, False, m.nSamples),
                       _cast(m, o[h:], d[h:], level, False, m.nSamples), ref):
        assert torch.equal(torch.cat([a, b]), r)
    perm = torch.randperm(o.shape[0], generator=torch.Generator().manual_seed(1)).to(DEV)
    for a, r in zip(_cast(m, o[perm], d[perm], level, False, m.nSamples), ref):
        assert torch.equal(a, r[perm])
    m8 = _synthetic((24, 32, 20), [8] * 3, [[-1.0, -0.5, -2.0], [1.5, 0.5, 1.0]], "softplus", seed=8)
    o8, d8 = _rays([[-1.0, -0.5, -2.0], [1.5, 0.5, 1.0]], 2000, seed=10)
    l8 = _levels(m8)[0.5]
    r8 = _cast(m8, o8, d8, l8, False, m8.nSamples)
    p8 = torch.randperm(o8.shape[0], generator=torch.Generator().manual_seed(2)).to(DEV)
    for a, r in zip(_cast(m8, o8[p8], d8[p8], l8, False, m8.nSamples, counter=False), r8):      # 4-lane layout
        assert torch.equal(a, r[p8])


def test_edge_cases():
    m = _synthetic((32, 32, 32), [16] * 3, [[-1.5] * 3, [1.5] * 3], "softplus", seed=8)
    level = _levels(m)[0.5]
    e = torch.zeros((0, 3), device=DEV)
    hit, t, xyz, n, rgb = m.raycast(e, e, level=level, colors=True)
    assert hit.shape == (0,) and t.shape == (0,) and xyz.shape == (0, 3) and n.shape == (0, 3) and rgb.shape == (0, 3)
    # pointing away from the box, and starting beyond it
    o = torch.tensor([[0.0, 0.0, 4.0], [5.0, 5.0, 5.0], [0.0, 3.0, 0.0]], device=DEV)
    d = torch.tensor([[0.0, 0.0, 1.0], [1.0, 0.0, 0.0], [0.0, 1.0, 0.0]], device=DEV)
    hit, t, xyz, n = m.raycast(o, d, level=level)
    assert not bool(hit.any()) and bool((t == float("inf")).all()) and float(xyz.abs().max()) == 0.0
    assert float(n.abs().max()) == 0.0
    # a ray starting inside: a dense field is inside at the first sample, which is where the ray enters the box
    dense = _synthetic((32, 32, 32), [16] * 3, [[-1.5] * 3, [1.5] * 3], "softplus", seed=8, shift=10.0)
    o2, d2 = torch.tensor([[0.0, 0.0, -4.0], [0.2, 0.1, 0.0]], device=DEV), torch.tensor([[0.0, 0.0, 1.0]] * 2, device=DEV)
    t2, xyz2, k2 = _cast(dense, o2, d2, 0.2, False, dense.nSamples)
    assert k2.tolist() == [0, 0]
    assert float(t2[0]) == 2.5 and float(xyz2[0, 2]) == -1.5
    # an all-empty field: every ray misses
    empty = _synthetic((32, 32, 32), [16] * 3, [[-1.5] * 3, [1.5] * 3], "softplus", seed=8, shift=-100.0)
    o3, d3 = _rays([[-1.5] * 3, [1.5] * 3], 500, seed=11)
    hit3, t3, _, _ = empty.raycast(o3, d3, level=1e-3)
    assert not bool(hit3.any()) and bool((t3 == float("inf")).all())
    for bad in (0.0, 1.0, -0.5, 1.5, float("nan")):
        with pytest.raises(jt._lib.JtError):
            m.raycast(o, d, level=bad)
    # the ABI takes fp32 factors only
    with pytest.raises(jt._lib.JtError):
        ops.raycast(m._density_factorset().with_bf16_store(None), m._h_geom(), m.density_shift, 0, float(m._h_step),
                    level, o, d, m.nSamples)


@pytest.mark.parametrize("workload", ["cfg2_sh", "cfg4"])
def test_full_size_slice(workload):
    kw, run = jt.synth.config(workload)
    kw = dict(kw)
    torch.manual_seed(0)
    m = jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), DEV, **kw)
    if run["ndc"]:
        o, d, _ = jt.synth.llff_ndc_rays(n_rays=4096)
    else:
        o, d = jt.synth.frame_rays()
        o, d = o[320000:324096], d[320000:324096]
    o, d = o.to(DEV), d.to(DEV)
    for q, level in _levels(m).items():
        check_bit_exact(m, o, d, level, run["ndc"], run["n_samples"], f"{workload}_q{q}")
