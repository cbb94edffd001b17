"""The VM factor-gradient scatter (jt_vm_scatter_rays), the gathers (jt_vm_gather_fwd) and the standalone gather
backward (jt_vm_gather_bwd) against the float64 reference of tests/vm_reference.py.

Bit-exact cases. The fields and sample lists are built so that every product and every partial sum the kernels form
is exactly representable in fp32: axes of n = 2^p + 1 texels, aabb [-1, 1]^3 (inv = 1), coordinates on the lattice
u = -1 + h / (n - 1) (tap fractions 0 or 1/2), small-integer factors, upstream gradients in multiples of 1/8 and
depths in multiples of 1/16 -- all bf16-exact too. `_premise` checks this on the reference's outputs and magnitudes.
Then any summation order gives the same bits, and the kernels must reproduce the reference with torch.equal: a lost,
duplicated or misplaced contribution cannot hide inside a tolerance. The hand-built sample lists hold long runs in
one plane cell, runs that continue from one ray into the next, rays that leave a cell and come back, thousands of
samples of many rays in one cell, one-sample rays, empty rays, in-ray gaps, the first and last texel of every axis
and the out-of-range band, and they run under every launch form of the render op's backward.

Full-size cases. The cfg2_sh and cfg4 batches with random factors and upstream gradients, in every launch form the
render op's backward uses: every factor-gradient element and every d_o / d_d entry within FULL_TOL of the sum of
absolute terms.

Data-parallel backward sequences. The render op's backward with an active gradient synchroniser (per-plane launches,
the 2+1 appearance split, the 2-rank form with and without reserved SMs), on one GPU through a synchroniser stub
whose collectives do nothing: every gradient of a full-size step matches the step without a synchroniser."""
import random

import pytest
import torch

import joint_tensorf_b200 as jt
from gpu_common import default_opt, record_err
from joint_tensorf_b200 import ops
from joint_tensorf_b200._lib import floats
from vm_reference import vm_adjoint

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# ------------------------------------------------------------------ bit-exact cases
GRID = (65, 129, 257)            # texels per axis: n - 1 a power of two, a different one per axis
S = 1024                         # samples per ray (sidx = ray * S + k)
PAD = 77                         # list capacity past the device-side count, filled with NaN / in-range garbage
CONFIGS = {                      # channels per plane / line pair
    "c16": (16, 16, 16),         # every shipped density field
    "c48": (48, 48, 48),         # cfg2 appearance: 4 lanes x 3 quads per walker
    "c32": (32, 32, 32),         # 4 lanes x 2 quads
    "c20": (20, 20, 20),         # cfg4 appearance: runtime lane count, one quad per lane
    "c12": (12, 12, 12),
    "mixed": (16, 20, 48),       # runtime lane count with lanes idle on the narrower planes
}
# (max_ctas, plane_mask) of every launch form: the default persistent grid, fixed segments of 1 .. 80 samples and one
# segment that covers the whole list on a non-persistent grid, persistent grids of 1 and 2 x 148 CTAs, every plane
# subset (the data-parallel backward walks planes 0+1, then plane 2, or one plane per launch)
ONE_WALKER = -(1 << 20)
FORMS = ([(0, 7), (-1, 7), (-2, 7), (-3, 7), (-7, 7), (-80, 7), (ONE_WALKER, 7), (1, 7), (296, 7)] +
         [(0, m) for m in range(1, 7)] + [(-80, 1), (-80, 2), (-80, 4)])


def _hmax(a):
    return 2 * (GRID[a] - 1)     # half-cell positions 0 .. hmax are in range (u = -1 .. 1)


def _sample_list(seed=0):
    """Ray-major list of (ray, k, h0, h1, h2): h is the position on axis a in half texels (x = h / 2)."""
    rng = random.Random(seed)
    recs = []
    ray = [-1]

    def add(samples, skip=0):    # one ray; `skip` empty rays before it
        ray[0] += 1 + skip
        ks = [k for k, _ in samples]
        assert ks == sorted(set(ks)) and ks[-1] < S
        recs.extend((ray[0], k, *h) for k, h in samples)

    def cell_pts(c, m):          # m random positions inside cell c (h in {2c, 2c + 1} per axis)
        return [tuple(2 * c[a] + rng.randrange(2) for a in range(3)) for _ in range(m)]

    def rand_cell():
        return [rng.randrange(GRID[a] - 1) for a in range(3)]

    def ks(m, start=0, gaps=False):
        k, out = start, []
        for _ in range(m):
            out.append(k)
            k += rng.randrange(1, 5) if gaps else 1
        return out

    # a long run in one plane cell while crossing line cells: ray along axis a, the other two fixed
    for a in range(3):
        h = [rng.randrange(_hmax(b) + 1) for b in range(3)]
        h[a] = rng.randrange(-6, 4)
        p_step = min(0.8, _hmax(a) / 210)
        pts = []
        for _ in range(200):
            pts.append(tuple(h))
            h[a] += 1 if rng.random() < p_step else 0
        add(list(zip(ks(200, 3), pts)))
    # consecutive rays in the same cell (a plane / line run continuing from one ray into the next)
    c = rand_cell()
    for r in range(6):
        m = rng.randrange(2, 12)
        add(list(zip(ks(m, rng.randrange(10), gaps=r % 2 == 1), cell_pts(c, m))))
    # sid = ray * S + S - 1 followed by (ray + 1) * S, in the same cell
    c = rand_cell()
    add(list(zip([S - 3, S - 2, S - 1], cell_pts(c, 3))))
    add(list(zip([0, 1, 2], cell_pts(c, 3))))
    # a ray that leaves a cell and comes back, on each axis
    for a in range(3):
        h = [2 * x for x in rand_cell()]
        pts = []
        for d in [0, 1, 2, 3, 2, 1, 0, 1, 2, 3, 4, 3, 2, 1, 0, -1, 0, 1]:
            p = list(h)
            p[a] = h[a] + d
            pts.append(tuple(p))
        add(list(zip(ks(len(pts), 5), pts)))
    # thousands of samples of many rays in one cell: REDs of many walkers collide
    c = rand_cell()
    for _ in range(48):
        add(list(zip(ks(40, rng.randrange(50)), cell_pts(c, 40))))
    # one-sample rays, some after empty rays
    for r in range(24):
        h = tuple(rng.randrange(-4, _hmax(a) + 5) for a in range(3))
        add([(rng.randrange(S), h)], skip=r % 3)
    # the first and last texel of every axis, and the out-of-range band (|u| up to ~1.1) and far outside (|u| = 3)
    for a in range(3):
        for lo, hi in [(0, 1), (_hmax(a) - 1, _hmax(a)), (-12, -1), (_hmax(a) + 1, _hmax(a) + 12)]:
            pts = []
            for _ in range(30):
                h = [rng.randrange(-2, _hmax(b) + 3) for b in range(3)]
                h[a] = rng.randrange(lo, hi + 1)
                pts.append(tuple(h))
            add(list(zip(ks(30, rng.randrange(20), gaps=True), pts)), skip=rng.randrange(2))
        h = [rng.randrange(_hmax(b) + 1) for b in range(3)]
        far = []
        for v in (-2 * (GRID[a] - 1), 4 * (GRID[a] - 1), 0, _hmax(a)):       # u = -3, 3, -1, 1
            p = list(h)
            p[a] = v
            far.append(tuple(p))
        add(list(zip(ks(4), far)))
    # random walks: cell changes on one, two or three axes, in-ray gaps, empty rays
    for r in range(150):
        h = [rng.randrange(-3, _hmax(a) + 4) for a in range(3)]
        m = rng.randrange(1, 100)
        pr = [rng.random() * 0.9 for _ in range(3)]
        pts = []
        for _ in range(m):
            pts.append(tuple(h))
            for a in range(3):
                if rng.random() < pr[a]:
                    h[a] += rng.choice((-1, 1, 1))
        add(list(zip(ks(m, rng.randrange(40), gaps=r % 4 == 0), pts)), skip=int(rng.random() < 0.1))
    return recs, ray[0] + 3


def _slot_subset(recs, seed):
    """Increasing subset of the list that drops whole rays and runs inside rays."""
    rng = random.Random(seed)
    dropped = {r for r in {x[0] for x in recs} if rng.random() < 0.15}
    keep, run = [], 0
    for e, x in enumerate(recs):
        if run == 0 and rng.random() < 0.04:
            run = rng.randrange(1, 15)
        if run > 0:
            run -= 1
            continue
        if x[0] not in dropped:
            keep.append(e)
    return keep


class _Case:
    """Factors, sample buffers and upstream gradients of one bit-exact case (device buffers padded past the count)."""

    def __init__(self, chans, use_slot, seed=0):
        recs, self.n_rays = _sample_list(seed)
        gen = torch.Generator().manual_seed(seed + 1)
        self.C = chans
        MAT, VEC = ((0, 1), (0, 2), (1, 2)), (2, 1, 0)
        self.planes = [torch.randint(-2, 3, (GRID[MAT[i][1]], GRID[MAT[i][0]], chans[i]), generator=gen).float().to(DEV)
                       for i in range(3)]
        self.lines = [torch.randint(-2, 3, (GRID[VEC[i]], chans[i]), generator=gen).float().to(DEV) for i in range(3)]
        V = len(recs)
        r = torch.tensor(recs, dtype=torch.float64)
        samp = torch.full((V + PAD, 4), float("nan"), dtype=torch.float64)
        for a in range(3):
            samp[:V, a] = -1.0 + r[:, 2 + a] / (GRID[a] - 1)
        samp[:V, 3] = torch.remainder(r[:, 1] * 5, 4) / 16           # t in multiples of 1/16
        self.samp = samp.float().to(DEV)
        sidx = torch.randint(0, self.n_rays * S, (V + PAD,), generator=gen, dtype=torch.int32)   # garbage in range
        sidx[:V] = (r[:, 0] * S + r[:, 1]).int()
        self.sidx = sidx.to(DEV)
        if use_slot:
            keep = _slot_subset(recs, seed + 2)
            self.n = len(keep)
            slot = torch.randint(0, V + PAD, (self.n + PAD,), generator=gen, dtype=torch.int32)  # garbage in range
            slot[:self.n] = torch.tensor(keep, dtype=torch.int32)
            self.slot = slot.to(DEV)
        else:
            self.n, self.slot = V, None
        self.n_max = self.n + PAD
        self.count = torch.tensor([self.n], dtype=torch.int32, device=DEV)
        ctot = sum(chans)
        gin_d = torch.full((self.n_max,), float("nan"))
        gin_d[:self.n] = torch.randint(-16, 17, (self.n,), generator=gen).float() / 8
        gin_a = torch.full((self.n_max, ctot), float("nan"))
        gin_a[:self.n] = torch.randint(-16, 17, (self.n, ctot), generator=gen).float() / 8
        self.gin = {0: gin_d.to(DEV), 1: gin_a.to(DEV)}
        self.ref = {app: vm_adjoint(self.planes, self.lines, self.samp, n=self.n, slot=self.slot,
                                    gin=self.gin[app][:self.n], sidx=self.sidx, S=S, n_rays=self.n_rays)
                    for app in (0, 1)}

    def factor_set(self, bf16_taps):
        fs = ops.FactorSet([p.permute(2, 0, 1)[None] for p in self.planes], [l.t()[None, :, :, None] for l in self.lines])
        return fs.with_bf16_store() if bf16_taps else fs


def _premise(case):
    """Every reference output, scaled by the power of two of its finest term, is an integer, and its magnitude (a
    bound of every partial sum) stays below 2^24 in those units: every fp32 operation of the kernels is exact."""
    # finest term of each output: tap weights are multiples of 1/2 per axis, gin of 1/8, t of 1/16; factors are
    # integers; du on axis a carries the factor (n_a - 1) / 2 = 2^(p_a - 1)
    k_du = torch.tensor([5.0 - ((GRID[a] - 1).bit_length() - 2) for a in range(3)], dtype=torch.float64, device=DEV)
    checks = []
    for app, r in case.ref.items():
        checks += [(f"value{app}", r.value, r.value_bound, 3.0)]
        checks += [(f"plane{app}.{i}", r.gp[i], r.gp_mag[i], 6.0) for i in range(3)]
        checks += [(f"line{app}.{i}", r.gl[i], r.gl_mag[i], 6.0) for i in range(3)]
        checks += [(f"du{app}", r.du, r.du_mag, k_du), (f"d_o{app}", r.d_o, r.d_o_mag, k_du),
                   (f"d_d{app}", r.d_d, r.d_d_mag, k_du + 4)]
    r0, r1 = case.ref[0], case.ref[1]
    checks.append(("du0+du1", r0.du + r1.du, r0.du_mag + r1.du_mag, k_du))       # jt_vm_gather_bwd accumulate
    for name, val, mag, k in checks:
        scale = torch.pow(2.0, torch.as_tensor(k, dtype=torch.float64, device=DEV))
        v, m = val * scale, mag * scale
        assert torch.equal(v, torch.round(v)), name
        assert float(m.max()) < 2 ** 24, (name, float(m.max()))
        assert float(m.max()) > 0, name


def _mismatch(got, ref):
    ref = ref.float()
    if torch.equal(got, ref):
        return None
    bad = got != ref
    return f"{int(bad.sum())} of {got.numel()} differ, max |diff| {float((got - ref).abs().nan_to_num(float('inf')).max()):.3g}"


_CASES = {}


def _case(chans_key, use_slot):
    key = (chans_key, use_slot)
    if key not in _CASES:
        _CASES.clear()
        _CASES[key] = _Case(CONFIGS[chans_key], use_slot)
    return _CASES[key]


@pytest.mark.parametrize("use_slot", [False, True], ids=["list", "slot"])
@pytest.mark.parametrize("chans", list(CONFIGS))
def test_bit_exact_premise(chans, use_slot):
    case = _case(chans, use_slot)
    _premise(case)
    assert case.n > 5000 and case.n_rays > 250


@pytest.mark.parametrize("bf16_taps", [False, True], ids=["fp32taps", "bf16taps"])
@pytest.mark.parametrize("use_slot", [False, True], ids=["list", "slot"])
@pytest.mark.parametrize("chans", list(CONFIGS))
def test_scatter_bit_exact(chans, use_slot, bf16_taps):
    """jt_vm_scatter_rays in every launch form, with and without factor gradients, density and appearance, fp32 and
    bf16 upstream gradients: torch.equal with the reference."""
    case = _case(chans, use_slot)
    fs = case.factor_set(bf16_taps)
    h_inv = floats([1.0, 1.0, 1.0])
    gp = [torch.empty_like(p) for p in case.planes]
    gl = [torch.empty_like(l) for l in case.lines]
    d_o = torch.empty((case.n_rays, 3), device=DEV)
    d_d = torch.empty_like(d_o)
    fails = []
    for app in (0, 1):
        ref = case.ref[app]
        for gin in ([case.gin[1], case.gin[1].to(torch.bfloat16)] if app else [case.gin[0]]):
            for max_ctas, mask in FORMS:
                for fg in (True, False):
                    for t in gp + gl + [d_o, d_d]:
                        t.zero_()
                    ops.vm_scatter_rays(app, fs, gp if fg else None, gl if fg else None, case.samp, case.slot,
                                        case.sidx, case.count, case.n_max, gin, S, h_inv, d_o, d_d,
                                        max_ctas=max_ctas, plane_mask=mask)
                    tag = f"app={app} gin={str(gin.dtype)[6:]} max_ctas={max_ctas} mask={mask} fg={fg}"
                    on = [i for i in range(3) if mask >> i & 1]
                    want = [("d_o", d_o, sum(ref.d_o_plane[i] for i in on)),
                            ("d_d", d_d, sum(ref.d_d_plane[i] for i in on))]
                    if fg:
                        for i in range(3):
                            want += [(f"plane{i}", gp[i], ref.gp[i] if i in on else torch.zeros_like(ref.gp[i])),
                                     (f"line{i}", gl[i], ref.gl[i] if i in on else torch.zeros_like(ref.gl[i]))]
                    for name, got, r in want:
                        bad = _mismatch(got, r)
                        if bad:
                            fails.append(f"{tag} {name}: {bad}")
    assert not fails, f"{len(fails)} mismatches; first: " + "; ".join(fails[:6])


@pytest.mark.parametrize("bf16_taps", [False, True], ids=["fp32taps", "bf16taps"])
@pytest.mark.parametrize("use_slot", [False, True], ids=["list", "slot"])
@pytest.mark.parametrize("chans", list(CONFIGS))
def test_gathers_bit_exact(chans, use_slot, bf16_taps):
    """jt_vm_gather_fwd (vm_density16_fwd_kernel, vm_fwd_kernel<false / true>) and jt_vm_gather_bwd (vm_bwd_kernel,
    QI 0..3; fp32 factors only) on the same lists: torch.equal with the reference, nothing written past the count."""
    case = _case(chans, use_slot)
    fs = case.factor_set(bf16_taps)
    n, fails = case.n, []
    rows = case.slot[:n].long() if case.slot is not None else torch.arange(n, device=DEV)
    for app in (0, 1):
        out = torch.full((case.n_max, sum(case.C)) if app else (case.n_max,), float("nan"), device=DEV)
        ops.vm_gather_fwd(app, fs, case.samp, case.slot, case.count, case.n_max, out)
        bad = _mismatch(out[:n], case.ref[app].value)
        if bad:
            fails.append(f"gather_fwd app={app}: {bad}")
        if not torch.isnan(out[n:]).all():
            fails.append(f"gather_fwd app={app}: written past the count")
    if not bf16_taps:
        dsamp = torch.full(case.samp.shape, float("nan"), device=DEV)
        du = torch.zeros((n, 3), dtype=torch.float64, device=DEV)
        for app in (0, 1):              # density stores dL/du, appearance adds to it (accumulate = 1)
            gp = [torch.zeros_like(p) for p in case.planes]
            gl = [torch.zeros_like(l) for l in case.lines]
            ops.vm_gather_bwd(app, fs, gp, gl, case.samp, case.slot, case.count, case.n_max, case.gin[app], dsamp, app)
            ref = case.ref[app]
            du = du + ref.du
            for name, got, r in ([(f"plane{i}", gp[i], ref.gp[i]) for i in range(3)] +
                                 [(f"line{i}", gl[i], ref.gl[i]) for i in range(3)] +
                                 [("du", dsamp[rows, :3], du), ("dsamp.w", dsamp[rows, 3], torch.zeros(n, device=DEV))]):
                bad = _mismatch(got, r)
                if bad:
                    fails.append(f"gather_bwd app={app} {name}: {bad}")
        untouched = torch.ones(dsamp.shape[0], dtype=torch.bool, device=DEV)
        untouched[rows] = False
        if not torch.isnan(dsamp[untouched]).all():
            fails.append("gather_bwd: dsamp written outside the listed samples")
    assert not fails, f"{len(fails)} mismatches; first: " + "; ".join(fails[:6])


# ------------------------------------------------------------------ full size, against the float64 adjoint
# |got - ref| <= tol * (sum of |terms|), per element. Measured on one NVIDIA B200 (1000 W): at most 4.5e-7 for the
# factor gradients and d_o / d_d of both workloads in every launch form
FULL_TOL = 4e-6
FWD_TOL = 1e-6           # appearance components (one product each: the terms are w P x w L, value_bound)


def _full_batch(wl):
    kw, run = jt.synth.config(wl)
    kw = dict(kw)
    ndc = bool(run["ndc"])
    if ndc:
        kw["near_far"] = [-1.0, 1.0]
    torch.manual_seed(0)
    m = jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), DEV, **kw)
    Sr = run["n_samples"]
    o, d, _ = jt.synth.llff_ndc_rays(4096, 1) if ndc else jt.synth.blender_rays(4096, 1)
    o, d = o.to(DEV).contiguous(), d.to(DEV).contiguous()
    if ndc:
        aux = m._ndc_table(Sr, False).contiguous()
    else:
        aux = torch.rand((o.shape[0],), generator=torch.Generator().manual_seed(1)).to(DEV).contiguous()
    comp = ops.march_compact(o, d, aux, ndc, Sr, m._h_geom(), None)
    gen = torch.Generator(device=DEV).manual_seed(2)
    rnd = lambda ps: [torch.randn(p.shape, device=DEV, generator=gen) * 0.3 for p in ps]     # noqa: E731
    dfs = ops.FactorSet(rnd(m.density_plane), rnd(m.density_line))
    afs = ops.FactorSet(rnd(m.app_plane), rnd(m.app_line))
    n = int(comp.count.item())
    keep = torch.rand((n,), device=DEV, generator=gen) < 0.6      # the appearance list: an increasing subset
    aidx = torch.zeros((comp.cap,), dtype=torch.int32, device=DEV)
    sel = torch.nonzero(keep).flatten().int()
    aidx[:sel.numel()] = sel
    a_count = torch.tensor([sel.numel()], dtype=torch.int32, device=DEV)
    gin_d = torch.randn((comp.cap,), device=DEV, generator=gen)
    gin_a = torch.randn((comp.cap, afs.ctot), device=DEV, generator=gen) * 0.1
    return dict(comp=comp, dfs=dfs, afs=afs, aidx=aidx, a_count=a_count, n=n, na=sel.numel(), gin_d=gin_d,
                gin_a=gin_a, S=Sr, h_inv=m._h_inv.tolist())


def _ref_planes(fs):
    if fs.store is None:
        return fs.planes, fs.lines
    return [s.float() for s in fs.store[:3]], [s.float() for s in fs.store[3:]]


def _rel(got, ref, mag):
    return float(((got.double() - ref).abs() / mag.clamp_min(1e-300)).max())


@pytest.mark.parametrize("bf16_taps", [False, True], ids=["fp32taps", "bf16taps"])
@pytest.mark.parametrize("wl", ["cfg2_sh", "cfg4"])
def test_full_size_scatter_matches_float64_adjoint(wl, bf16_taps):
    B = _full_batch(wl)
    comp, N, Sr = B["comp"], B["comp"].n_rays, B["S"]
    h_inv = floats(B["h_inv"])
    errs, fails = {}, []
    # density: the default launch, fixed 80-sample segments, a persistent grid that leaves SMs to a collective
    # appearance: the default launch, planes 0+1 then plane 2 (80-sample segments), one launch per plane
    seqs = {0: {"default": [(0, 7)], "seg80": [(-80, 7)], "ctas560": [(560, 7)]},
            1: {"default": [(0, 7)], "split21": [(0, 3), (-80, 4)], "per_plane": [(-80, 1), (-80, 2), (-80, 4)]}}
    for app in (0, 1):
        fs = B["afs"] if app else B["dfs"]
        if bf16_taps:
            fs = fs.with_bf16_store()
        planes, lines = _ref_planes(fs)
        slot, n_dev, n = (B["aidx"], B["a_count"], B["na"]) if app else (None, comp.count, B["n"])
        gins = [B["gin_a"], B["gin_a"].to(torch.bfloat16)] if app else [B["gin_d"]]
        for gin in gins:
            ref = vm_adjoint(planes, lines, comp.samp, n=n, slot=slot, gin=gin[:n], sidx=comp.sidx, S=Sr, n_rays=N,
                             inv=B["h_inv"])
            gname = "bf16" if gin.dtype == torch.bfloat16 else "fp32"
            if app and gname == "fp32":        # the appearance gather (vm_fwd_kernel<true>) on the same list
                out = torch.full((comp.cap, fs.ctot), float("nan"), device=DEV)
                ops.vm_gather_fwd(1, fs, comp.samp, slot, n_dev, comp.cap, out)
                e = _rel(out[:n], ref.value, ref.value_bound)
                errs["app_fwd"] = e
                if not e <= FWD_TOL or not torch.isnan(out[n:]).all():
                    fails.append(f"app gather: {e:.3g}")
            for sname, seq in seqs[app].items():
                gp, gl = fs.zero_grads()
                d_o, d_d = torch.zeros((N, 3), device=DEV), torch.zeros((N, 3), device=DEV)
                for max_ctas, mask in seq:
                    ops.vm_scatter_rays(app, fs, gp, gl, comp.samp, slot, comp.sidx, n_dev, comp.cap, gin, Sr, h_inv,
                                        d_o, d_d, max_ctas=max_ctas, plane_mask=mask)
                torch.cuda.synchronize()
                for name, got, r, mag in ([(f"plane{i}", gp[i], ref.gp[i], ref.gp_mag[i]) for i in range(3)] +
                                          [(f"line{i}", gl[i], ref.gl[i], ref.gl_mag[i]) for i in range(3)] +
                                          [("d_o", d_o, ref.d_o, ref.d_o_mag), ("d_d", d_d, ref.d_d, ref.d_d_mag)]):
                    e = _rel(got, r, mag)
                    key = f"{'app' if app else 'dens'}/{gname}/{sname}/{name}"
                    errs[key] = e
                    if not e <= FULL_TOL:
                        fails.append(f"{key}: {e:.3g}")
            del ref
    record_err(f"vm_adjoint_full:{wl}:{'bf16' if bf16_taps else 'fp32'}taps", tol=FULL_TOL, **errs)
    assert not fails, fails


# ------------------------------------------------------------------ the render op's data-parallel backward sequences
class _StubSync:
    """A gradient synchroniser that reports itself active but issues no collective: the render op's backward takes
    its data-parallel launch sequence on one GPU (the stub's on_app_grads / on_rest are no-ops, so the gradients stay
    the rank-local ones). Nothing else in the module consults the synchroniser during a step: the loss scale and the
    pose-table reduce are the caller's (OverlappedGradSync.finish), and with every input trainable the synchroniser's
    "full backward" computes what the single-GPU backward computes."""

    def __init__(self, per_plane=False, split21=False, reserve_sms=0):
        self.per_plane, self.split21, self.reserve_sms = per_plane, split21, reserve_sms
        self.calls = 0

    def _active(self):
        return True

    def use_split21(self, n_app, n_total):
        return self.split21

    def on_app_grads(self, region):
        self.calls += 1

    def on_rest(self, region):
        self.calls += 1


SYNC_NOISE = 2e-5        # max |a - b| / max |b| per gradient tensor: fp32 atomic-order noise only (measured on one
                         # NVIDIA B200: at most 5.2e-6, on the density lines)

SYNC_VARIANTS = {"per_plane": dict(per_plane=True), "split21": dict(split21=True),
                 "two_rank": dict(), "two_rank_reserve": dict(reserve_sms=8)}


@pytest.mark.parametrize("wl", ["cfg2_sh", "cfg4"])
def test_data_parallel_backward_sequences_match_single_gpu(wl):
    kw, run = jt.synth.config(wl)
    kw = dict(kw)
    ndc = bool(run["ndc"])
    if ndc:
        kw["near_far"] = [-1.0, 1.0]
    torch.manual_seed(0)
    m = jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), DEV, **kw)
    Sr = run["n_samples"]
    o, d, _ = jt.synth.llff_ndc_rays(4096, 1) if ndc else jt.synth.blender_rays(4096, 1)
    o, d = o.to(DEV), d.to(DEV)
    tgt = torch.rand((4096, 3), generator=torch.Generator().manual_seed(5)).to(DEV)
    opt = default_opt(m.shadingMode, ndc)

    def step(sync):
        m.grad_sync = sync
        for p in m.parameters():
            p.grad = None
        og, dg = o.clone().requires_grad_(True), d.clone().requires_grad_(True)
        rgb, _, _ = m.forward(opt, og, dg, white_bg=run["white_bg"], is_train=False, ndc_ray=ndc, N_samples=Sr)
        ((rgb - tgt) ** 2).mean().backward()
        torch.cuda.synchronize()
        m.grad_sync = None
        g = {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None}
        g.update(d_rays_o=og.grad.clone(), d_rays_d=dg.grad.clone())
        return g

    base = step(None)
    assert all(float(v.abs().max()) > 0 for v in base.values()), [k for k, v in base.items() if v.abs().max() == 0]
    errs, fails = {}, []
    for name, kws in SYNC_VARIANTS.items():
        sync = _StubSync(**kws)
        g = step(sync)
        assert sync.calls >= 2, name                 # the data-parallel branch ran
        assert g.keys() == base.keys()
        for k, ref in base.items():
            e = float((g[k] - ref).abs().max() / ref.abs().max().clamp_min(1e-30))
            errs[f"{name}/{k}"] = e
            if not e <= SYNC_NOISE:
                fails.append(f"{name}/{k}: {e:.3g}")
    record_err(f"dp_backward_sequences:{wl}", tol=SYNC_NOISE, **errs)
    assert not fails, fails
