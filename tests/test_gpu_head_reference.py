"""The tensor-core shading heads (and the strict-fp32 chain) against the float64 reference of tests/head_reference.py,
element by element, with bounds stated on each element's magnitude.

The heads run through the render op's own head classes (render._ShTcHead, _MlpTcHead, _WeakViewTcHead, _Fp32Head) on
a hand-built ops.Compacted, as render.shade_points drives them: the launches, staging-area sizing, operand split and
dcomps dtype are the render op's. The components come from a random VM field through the fused gathers; their float64
values are tests/vm_reference.py's (bf16-rounded factors for bf16 factor storage).

Sizes: A in {0, 1, 127, 128, 129, 255, 257, 148 x 128 - 1, 148 x 128, 148 x 128 + 1, 296 x 128 + 1} and the A of one
training step of cfg2_sh, cfg2 and cfg4; list capacity n_max in {A, A + 1, 2A} (at least 1, as in the render op); the
count always comes from the device. Inputs past the count are poisoned: sample records and components with NaN (their
list slots point at NaN records), dout with NaN. The staging area starts as 0xFF bytes (bf16 NaN). Outputs handed to
the kernels are views into larger buffers: the rows between the count and n_max and the tail past n_max hold sentinels
that must survive.

Forward: every element of feat and rgb within FWD_MULT x (operand unit) x magnitude (for rgb the pre-activation's),
the unit being 2^-16 for hi + lo bf16 operands, 2^-8 for bf16, 2^-11 for fp16 and 2^-24 for the fp32 chain. The
class path and a direct call of the same ops into sentinel-guarded views give the same bits.

Backward (dout non-zero only on rows without an ambiguous relu unit, see head_reference): every dcomps and weight-
gradient element within BWD_MULT x 2^-8 x its magnitude, accumulated onto a non-zero base; then the same with dout
restricted to single rows and tiles (rows 0, 127, 128, A - 1; the last tile; the second tile of wgrad CTA 0; the last
tile of the last CTA), where a dropped, repeated or misplaced tile moves a gradient by ~100 % of its magnitude; the
partition of the rows into those parts must sum to the full call's weight gradients within ADD_TOL of the magnitude
(the bf16 operands of a row do not depend on the other rows: only the fp32 accumulation order differs), and each part's
dcomps rows must equal the full call's bit for bit while rows outside the part are exactly zero."""
import pytest
import torch

import joint_tensorf_b200 as jt
from gpu_common import default_opt, record_err
from head_reference import head_backward, head_forward, view_dirs
from joint_tensorf_b200 import ops, render
from oracle import vm_oracle as vo
from vm_reference import vm_adjoint

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TM, NSM = 128, 148                   # rows per tile, SMs of a B200 (the wgrad kernels' persistent grid)
S, N_RAYS, GRID = 64, 97, (13, 11, 17)
REC_PAD = 41                         # NaN sample records past the live ones
TAIL = 3                             # rows of every output buffer past n_max
SENT_ROW, SENT_TAIL = -777.0, 12345.0
SIZES = [0, 1, 127, 128, 129, 255, 257, NSM * TM - 1, NSM * TM, NSM * TM + 1, 2 * NSM * TM + 1,
         "cfg2_sh", "cfg2", "cfg4"]
# (fea_prog, view_prog, normalize_dir), cycled over the sizes: every head sees progress 1, 0.65 and 0 on both PE
# inputs and both direction modes
PROGS = [(0.65, 0.65, True), (1.0, 0.0, False), (0.0, 1.0, True), (0.65, 1.0, False), (1.0, 0.65, True),
         (0.0, 0.65, False)]
UNIT = {1: 2.0 ** -8, 2: 2.0 ** -16, 3: 2.0 ** -11, "fp32": 2.0 ** -24}
# Bounds: |got - ref| <= MULT x unit x magnitude, per element, each multiple at least 4x the largest value measured
# over all sizes and n_max on one NVIDIA B200 (in the comments). The rgb bounds are stated on the magnitude of the
# pre-activation, which the MLP heads' cancelling sums make large: hence multiples below 1 there.
FWD_MULT = {   # variant: (feat, rgb); SH's tensor-core forward writes no features
    "sh_split2": (None, 0.5),              # rgb 0.099
    "sh_split2_bf16store": (None, 0.5),    # rgb 0.109
    "sh_split1": (None, 1.0),              # rgb 0.200
    "sh_infer": (None, 0.5),               # rgb 0.099
    "mlp_split2": (2.0, 1 / 64),           # feat 0.294, rgb 0.0034
    "mlp_split2_bf16store": (2.0, 1 / 64),  # feat 0.289, rgb 0.0030
    "mlp_split1": (2.0, 1 / 64),           # feat 0.493, rgb 0.0020
    "mlp_infer_fp16": (1 / 16, 1 / 32),    # feat 0.0092 (from the hi + lo basis kernel), rgb 0.0049
    "mlp_infer_hilo": (2.0, 1 / 64),       # feat 0.294, rgb 0.0034
    "wv": (2.0, 1 / 32),                   # feat 0.436, rgb 0.0052
    "wv_infer": (2.0, 1 / 32),             # feat 0.436, rgb 0.0052
    "fp32_sh": (32.0, 16.0),               # feat 6.34, rgb 2.05
    "fp32_mlp": (32.0, 2.0),               # feat 6.34, rgb 0.279
    "fp32_wv": (32.0, 8.0),                # feat 5.52, rgb 1.12
}
BWD_MULT = 8.0                       # backward, bf16 unit 2^-8: dcomps 1.96 (SH, bf16 rows), weight gradients 1.43
ADD_TOL = 2.0 ** -21                 # partition additivity of the weight gradients on the magnitude: 1.0e-7 (SH)
AMB = 2.0 ** -18                     # ambiguous relu unit: |pre| <= AMB x magnitude (the hi + lo forward's masks)
AMB_ROWS = 0.15                      # at most this fraction of rows may hold an ambiguous unit: 0.082 (MLP_Fea)

HEADS = {   # shading, components per plane, app_dim, hidden, head class
    "sh": ("SH", 48, 27, 0, render._ShTcHead),
    "mlp": ("MLP_Fea", 48, 27, 64, render._MlpTcHead),
    "wv": ("MLP_Fea_WeakView", 20, 20, 32, render._WeakViewTcHead),
}
PARAM_NAMES = {"MLP_Fea": [f"renderModule.mlp.{i}.{k}" for i in (0, 2, 4) for k in ("weight", "bias")],
               "MLP_Fea_WeakView": [f"renderModule.layer{i}.{k}" for i in (1, 2, 3) for k in ("weight", "bias")]}
# stage layout (bytes) per tile: the regions head_tc.cuh / weakview_tc.cu define, as (offset, size); `fwd` regions are
# written by the forward, `bwd` regions by the backward with weight gradients
STAGE = {
    "tc": dict(tile=161792, fwd=[(0, 36864), (36864, 40960), (77824, 20480), (98304, 20480)],
               bwd=[(118784, 16384), (135168, 16384), (151552, 8192), (159744, 2048)]),
    "wv": dict(tile=96256, fwd=[(0, 16384), (16384, 28672), (45056, 12288), (57344, 12288)],
               bwd=[(69632, 8192), (77824, 8192), (86016, 8192), (94208, 2048)]),
}


# ------------------------------------------------------------------ inputs
_CFG_A = {}


def _size(a):
    """A of one training step of a benchmark workload (VMRender.last_counts), or the literal size."""
    if isinstance(a, int):
        return a
    if a not in _CFG_A:
        kw, run = jt.synth.config(a)
        kw = dict(kw)
        ndc = bool(run["ndc"])
        if ndc:
            kw["near_far"] = [-1.0, 1.0]
        torch.manual_seed(0)
        m = jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), DEV, **kw)
        o, d, _ = jt.synth.llff_ndc_rays(4096, 1) if ndc else jt.synth.blender_rays(4096, 1)
        m.forward(default_opt(m.shadingMode, ndc), o.to(DEV), d.to(DEV), white_bg=run["white_bg"], is_train=True,
                  ndc_ray=ndc, N_samples=run["n_samples"])
        _CFG_A[a] = int(jt.VMRender.last_counts[1].item())
        del m
        torch.cuda.empty_cache()
    return _CFG_A[a]


def _n_maxes(A):
    return sorted({max(A, 1), A + 1, max(2 * A, 1)})


class _Inputs:
    """A random VM appearance field, a sample list of A appearance samples (slots into V = A + 37 records, in random
    order, plus NaN records past them), rays with non-unit directions, basis_mat and head weights, and the float64
    components of the live samples."""

    def __init__(self, head, A, storage="fp32", seed=0):
        shading, C, F, H, self.Head = HEADS[head]
        self.shading, self.A, self.F, self.H = shading, A, F, H
        gen = torch.Generator(device=DEV).manual_seed(seed)
        MAT, VEC = ((0, 1), (0, 2), (1, 2)), (2, 1, 0)
        planes = [torch.randn((GRID[MAT[i][1]], GRID[MAT[i][0]], C), device=DEV, generator=gen) for i in range(3)]
        lines = [torch.randn((GRID[VEC[i]], C), device=DEV, generator=gen) for i in range(3)]
        fs = ops.FactorSet([p.permute(2, 0, 1)[None] for p in planes], [l.t()[None, :, :, None] for l in lines])
        if storage == "bf16":
            fs = fs.with_bf16_store()
            planes, lines = [s.float() for s in fs.store[:3]], [s.float() for s in fs.store[3:]]
        self.afs = fs
        V = A + 37
        self.samp = torch.full((V + REC_PAD, 4), float("nan"), device=DEV)
        self.samp[:V, :3] = torch.rand((V, 3), device=DEV, generator=gen) * 2.2 - 1.1   # some taps off the grid
        self.samp[:V, 3] = 0.0
        self.sidx = (torch.randint(0, N_RAYS, (V + REC_PAD,), device=DEV, generator=gen) * S +
                     torch.randint(0, S, (V + REC_PAD,), device=DEV, generator=gen)).int()
        cap = 2 * A + 1
        self.aidx = torch.randint(V, V + REC_PAD, (cap,), device=DEV, generator=gen).int()   # NaN records
        self.aidx[:A] = torch.randperm(V, device=DEV, generator=gen)[:A].int()
        self.rays_d = torch.randn((N_RAYS, 3), device=DEV, generator=gen) * 1.7
        self.count = torch.tensor([A], device=DEV, dtype=torch.int32)
        p = vo.init_params(list(GRID), [16] * 3, [C] * 3, F, shading, max(H, 1), 2, 2, 0.1, 0.0, seed=seed)
        self.wb = p["basis_mat.weight"].to(DEV).contiguous()
        self.params = [p[k].to(DEV).contiguous() for k in PARAM_NAMES.get(shading, [])]
        gin = torch.zeros((1, sum(fs.C)), device=DEV).expand(A, -1)     # [A, sum C]: the appearance form
        r = vm_adjoint(planes, lines, self.samp, n=A, slot=self.aidx, gin=gin)
        self.comps_ref, self.comps_mag = r.value, r.value_bound
        self.comps = torch.full((cap, sum(fs.C)), float("nan"), device=DEV)     # WeakView's fp32 component rows
        ops.vm_gather_fwd(1, fs, self.samp, self.aidx, self.count, cap, self.comps)

    def cfg(self, fprog, vprog, ndc, split=2, head="tc", infer_fp16=True, storage="fp32"):
        return render.RenderCfg(shading=self.shading, app_dim=self.F, hidden=self.H, fea_pe=2, view_pe=2,
                                fea_prog=fprog, view_prog=vprog, n_samples=S, ndc=ndc, head=head, tc_fwd_split=split,
                                tc_infer_fp16=infer_fp16, storage=storage)

    def head(self, cfg, n_max, Head=None):
        comp = ops.Compacted()
        comp.samp, comp.sidx = self.samp, self.sidx
        return (Head or self.Head)(cfg, self.afs, comp, self.aidx, self.rays_d, self.wb, self.params, self.count,
                                   n_max)

    def reference(self, fprog, vprog, ndc, amb):
        dirs = view_dirs(self.rays_d, self.sidx, self.aidx, self.A, S, ndc)
        return head_forward(self.shading, self.comps_ref, dirs, self.wb, self.params, fprog, vprog,
                            comps_mag=self.comps_mag, amb=amb), dirs


@pytest.fixture
def ff_stage(monkeypatch):
    """The head classes' staging areas start as 0xFF bytes; returns the list of the areas handed out."""
    made = []

    def wrap(orig):
        def alloc(n_max, device):
            st = orig(n_max, device)
            st.fill_(0xFF)
            made.append(st)
            return st
        return alloc
    monkeypatch.setattr(ops, "head_tc_stage", wrap(ops.head_tc_stage))
    monkeypatch.setattr(ops, "wv_stage", wrap(ops.wv_stage))
    return made


def _guarded(n_max, A, cols, dtype=torch.float32):
    """[n_max + TAIL, cols] buffer, rows [A, n_max) holding SENT_ROW and the tail SENT_TAIL: (buffer, view [:n_max])."""
    buf = torch.full((n_max + TAIL, cols), SENT_TAIL, device=DEV, dtype=dtype)
    buf[A:n_max] = SENT_ROW
    return buf, buf[:n_max]


def _guard_ok(buf, A, n_max, dtype=torch.float32):
    return (bool((buf[A:n_max] == torch.tensor(SENT_ROW, dtype=dtype)).all()) and
            bool((buf[n_max:] == torch.tensor(SENT_TAIL, dtype=dtype)).all()))


def _rel(got, ref, mag):
    """max |got - ref| / mag (0 / 0 = 0; a non-zero difference over a zero magnitude is inf)."""
    if got.numel() == 0:
        return 0.0
    d = (got.double() - ref).abs()
    r = torch.where(d == 0, torch.zeros_like(d), d / mag)
    return float(r.nan_to_num(float("inf")).max())


def _stage_check(kind, stage, A, n_max, regions):
    """Tiles below ceil(A / 128): the given regions hold finite bf16 values (rows past A included); tiles past them up
    to ceil(n_max / 128) are untouched (0xFF)."""
    L = STAGE[kind]
    t_live = (A + TM - 1) // TM
    tiles = stage[: ((n_max + TM - 1) // TM) * L["tile"]].view(-1, L["tile"])
    for off, size in regions:
        if t_live and not bool(torch.isfinite(tiles[:t_live, off:off + size].view(torch.bfloat16).float()).all()):
            return f"non-finite staged operands in region at {off}"
    if not bool((tiles[t_live:] == 0xFF).all()):
        return "staging tiles past the count were written"
    return None


# ------------------------------------------------------------------ forward
# id -> (head, train, split, storage, infer_fp16, class): the render op's forward launches
FWD = {
    "sh_split2": ("sh", True, 2, "fp32", True, None),
    "sh_split2_bf16store": ("sh", True, 2, "bf16", True, None),
    "sh_split1": ("sh", True, 1, "fp32", True, None),
    "sh_infer": ("sh", False, 2, "fp32", True, None),
    "mlp_split2": ("mlp", True, 2, "fp32", True, None),
    "mlp_split2_bf16store": ("mlp", True, 2, "bf16", True, None),
    "mlp_split1": ("mlp", True, 1, "fp32", True, None),
    "mlp_infer_fp16": ("mlp", False, 3, "fp32", True, None),
    "mlp_infer_hilo": ("mlp", False, 2, "fp32", False, None),
    "wv": ("wv", True, 2, "fp32", True, None),
    "wv_infer": ("wv", False, 2, "fp32", True, None),
    "fp32_sh": ("sh", True, "fp32", "fp32", True, render._Fp32Head),
    "fp32_mlp": ("mlp", True, "fp32", "fp32", True, render._Fp32Head),
    "fp32_wv": ("wv", True, "fp32", "fp32", True, render._Fp32Head),
}


def _direct_forward(I, split, stage, fprog, vprog, ndc, n_max):
    """The class's forward launches called directly with sentinel-guarded output views: (featdir buffer, rgb buffer)."""
    A = I.A
    fbuf, fd = _guarded(n_max, A, 32)
    rbuf, rgb = _guarded(n_max, A, 4)
    if I.shading == "SH":
        ops.app_basis_sh_fwd_tc(split, I.afs, I.samp, I.aidx, I.sidx, I.rays_d, S, ndc, I.wb, I.count, n_max, fd, rgb,
                                stage)
    elif I.shading == "MLP_Fea":
        ops.app_basis_fwd_tc(min(split, 2), I.afs, I.samp, I.aidx, I.sidx, I.rays_d, S, ndc, I.wb, I.count, n_max, fd,
                             stage)
        ops.head_mlp_fwd_tc(split, fd, *I.params, I.count, n_max, fprog, vprog, rgb, stage)
    else:
        ops.wv_head_fwd_tc(I.comps, I.aidx, I.sidx, I.rays_d, S, ndc, I.wb, *I.params, I.count, n_max, fprog, vprog,
                           fd, rgb, stage)
    return fbuf, rbuf


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("variant", list(FWD))
def test_forward_matches_float64(variant, size, ff_stage):
    """feat, view direction and rgb of every live row against float64 at every n_max; the direct launches into
    sentinel-guarded views reproduce the class's bits and write nothing past the count; staged operand tiles are finite
    below the count and untouched past it."""
    head, train, split, storage, infer_fp16, Head = FWD[variant]
    A = _size(size)
    fprog, vprog, ndc = PROGS[SIZES.index(size) % len(PROGS)]
    I = _Inputs(head, A, storage, seed=SIZES.index(size))
    unit = UNIT[split]
    ref, dirs = I.reference(fprog, vprog, ndc, amb=16 * unit)
    errs, fails = {}, []
    for n_max in _n_maxes(A):
        cfg = I.cfg(fprog, vprog, ndc, split=2 if split == "fp32" else min(split, 2),
                    head="fp32" if split == "fp32" else "tc", infer_fp16=infer_fp16, storage=storage)
        h = I.head(cfg, n_max, Head)
        n_stage = len(ff_stage)
        rgb = h.forward(train, True)
        torch.cuda.synchronize()
        tag = f"n_max={n_max}"
        m_feat, m_rgb = FWD_MULT[variant]
        e_rgb = _rel(rgb[:A, :3], ref.rgb, ref.pre_mag) / unit
        e_feat = _rel(h.feat[:A, :I.F], ref.feat, ref.feat_mag) / unit if m_feat is not None else 0.0
        errs[f"rgb/{tag}"], errs[f"feat/{tag}"] = e_rgb, e_feat
        if not (e_rgb <= m_rgb and (m_feat is None or e_feat <= m_feat)):
            fails.append(f"{tag}: rgb {e_rgb:.3g}, feat {e_feat:.3g} units")
        if split == "fp32":
            continue
        e_dir = float((h.feat[:A, 28:31].double() - dirs).abs().max()) if A else 0.0
        if not e_dir <= 2.0 ** -21 * 3:
            fails.append(f"{tag}: view direction off by {e_dir:.3g}")
        if not bool((h.feat[:A, 31] == 0).all()) or (I.shading == "MLP_Fea" and not bool((h.feat[:A, 27] == 0).all())):
            fails.append(f"{tag}: pad columns of featdir not zero")
        stage = ff_stage[n_stage] if len(ff_stage) > n_stage else None
        assert (stage is not None) == train
        if stage is not None:
            bad = _stage_check("wv" if head == "wv" else "tc", stage, A, n_max,
                               STAGE["wv" if head == "wv" else "tc"]["fwd"][:1 if head == "sh" else 4])
            if bad:
                fails.append(f"{tag}: {bad}")
        # the same launches into guarded views; the staging area of this call starts as 0xFF too
        st2 = None
        if stage is not None:
            st2 = torch.full_like(stage, 0xFF)
        fbuf, rbuf = _direct_forward(I, split, st2, fprog, vprog, ndc, n_max)
        torch.cuda.synchronize()
        if not torch.equal(rbuf[:A], rgb[:A]):
            fails.append(f"{tag}: direct rgb differs from the class's")
        cols = [28, 29, 30] + ([] if I.shading == "SH" else list(range(I.F)))
        if not torch.equal(fbuf[:A, cols], h.feat[:A, cols]):
            fails.append(f"{tag}: direct featdir differs from the class's")
        if not (_guard_ok(rbuf, A, n_max) and _guard_ok(fbuf, A, n_max)):
            fails.append(f"{tag}: rows past the count or past n_max were written")
        if st2 is not None and not torch.equal(st2, stage):
            fails.append(f"{tag}: direct staging area differs from the class's")
    record_err(f"head_fwd:{variant}:{size}", A=A, **errs)
    assert not fails, fails


# ------------------------------------------------------------------ backward
BWD = {   # id -> (head, dcomps dtype)
    "sh": ("sh", torch.bfloat16),
    "mlp_bf16dc": ("mlp", torch.bfloat16),
    "mlp_fp32dc": ("mlp", torch.float32),
    "wv": ("wv", torch.float32),
}
GRAD_KEYS = ("wb", "w1", "b1", "w2", "b2", "w3", "b3")


def _row_sets(A, n_max):
    """Disjoint row parts: rows {0, 127, 128, A - 1}; the last tile; the second tile of wgrad CTA 0 (tile index =
    grid size); the last tile of the last CTA; the remaining rows in two random halves."""
    grid = min((n_max + TM - 1) // TM, NSM)
    ntiles = (A + TM - 1) // TM
    tile = lambda t: set(range(t * TM, min((t + 1) * TM, A))) if 0 <= t < ntiles else set()   # noqa: E731
    last_cta = [t for t in range(grid - 1, ntiles, grid)]
    sets = [{r for r in (0, 127, 128, A - 1) if 0 <= r < A}, tile(ntiles - 1), tile(grid),
            tile(last_cta[-1]) if last_cta else set()]
    parts, seen = [], set()
    for s in sets:
        s = s - seen
        seen |= s
        parts.append(sorted(s))
    rest = torch.tensor(sorted(set(range(A)) - seen), dtype=torch.long)
    perm = rest[torch.randperm(rest.numel(), generator=torch.Generator().manual_seed(A))]
    parts += [sorted(perm[: rest.numel() // 2].tolist()), sorted(perm[rest.numel() // 2:].tolist())]
    return [p for p in parts if p]


def _backward(h, I, dout, n_max, dc_dtype, base):
    """Class backward into guarded views; weight gradients accumulate onto `base`. Returns (dcomps buffer, grads
    {key: (buffer, view)})."""
    A, ctot = I.A, sum(I.afs.C)
    dbuf, dc = _guarded(n_max, A, ctot, dc_dtype)
    grads = {}
    for k, t in zip(GRAD_KEYS, [I.wb] + I.params):
        buf = torch.full((t.numel() + TAIL,), SENT_TAIL, device=DEV)
        buf[:t.numel()] = base[k].reshape(-1)
        grads[k] = (buf, buf[:t.numel()].view(t.shape))
    head_grads = [grads[k][1] for k in GRAD_KEYS[1:]] if I.params else None
    h.backward(dout, dc, grads["wb"][1], head_grads)
    torch.cuda.synchronize()
    return dbuf, grads


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("variant", list(BWD))
def test_backward_matches_float64(variant, size, ff_stage):
    """dcomps and the weight gradients against float64 at every n_max (full dout, onto a non-zero base), then dout
    restricted to row / tile parts: each part against its own float64 reference, the parts' sum against the full
    call, dcomps rows bit-equal to the full call's and exactly zero outside the part."""
    head, dc_dtype = BWD[variant]
    A = _size(size)
    fprog, vprog, ndc = PROGS[(SIZES.index(size) + 1) % len(PROGS)]
    I = _Inputs(head, A, seed=100 + SIZES.index(size))
    ref, _ = I.reference(fprog, vprog, ndc, amb=AMB)
    amb_rows = int(ref.ambiguous.sum())
    gen = torch.Generator(device=DEV).manual_seed(7)
    dout_live = torch.randn((A, 4), device=DEV, generator=gen) * (~ref.ambiguous)[:, None]
    dout_live[:, 3] = 0
    unit = 2.0 ** -8
    errs, fails = dict(amb_rows=amb_rows), []
    if amb_rows > AMB_ROWS * max(A, 1):
        fails.append(f"{amb_rows} of {A} rows hold an ambiguous relu unit")
    keys = GRAD_KEYS if I.params else GRAD_KEYS[:1]
    for n_max in _n_maxes(A):
        tag = f"n_max={n_max}"
        cfg = I.cfg(fprog, vprog, ndc)
        h = I.head(cfg, n_max)
        h.forward(True, True)
        stage = ff_stage[-1]

        def run(rows):
            """Backward with dout on `rows` (None: all live rows), NaN past the count; (dcomps, grads, ref)."""
            dout = torch.full((n_max, 4), float("nan"), device=DEV)
            d = dout_live if rows is None else torch.zeros_like(dout_live)
            if rows is not None:
                idx = torch.tensor(rows, device=DEV, dtype=torch.long)
                d[idx] = dout_live[idx]
            dout[:A] = d
            b = head_backward(ref, d)
            base = {k: torch.zeros_like(t) for k, t in zip(GRAD_KEYS, [I.wb] + I.params)}
            if rows is None:     # accumulation onto a non-zero base
                base = {k: torch.randn(t.shape, device=DEV, generator=gen) for k, t in base.items()}
            dbuf, grads = _backward(h, I, dout, n_max, dc_dtype, base)
            if not _guard_ok(dbuf, A, n_max, dc_dtype):
                fails.append(f"{tag} rows={'all' if rows is None else len(rows)}: dcomps written past the count")
            for k in keys:
                buf, v = grads[k]
                if not bool((buf[v.numel():] == SENT_TAIL).all()):
                    fails.append(f"{tag}: written past the end of d{k}")
            g = {k: grads[k][1].double() - base[k].double() for k in keys}
            slack = {k: base[k].double().abs() * 2.0 ** -23 for k in keys}     # rounding of base + gradient
            return dbuf[:A], g, b, slack

        dc_full, g_full, b_full, slack = run(None)
        e = _rel(dc_full, b_full.dcomps, b_full.dcomps_mag) / unit
        errs[f"full/{tag}/dcomps"] = e
        if not e <= BWD_MULT:
            fails.append(f"{tag}: dcomps {e:.3g} units")
        for k in keys:
            d = (g_full[k] - b_full.grads[k]).abs() - slack[k]
            e = _rel(d.clamp_min(0), torch.zeros_like(d), b_full.grads_mag[k]) / unit
            errs[f"full/{tag}/{k}"] = e
            if not e <= BWD_MULT:
                fails.append(f"{tag}: d{k} {e:.3g} units")
        bad = _stage_check("wv" if head == "wv" else "tc", stage, A, n_max,
                           [STAGE["tc"]["fwd"][0], STAGE["tc"]["bwd"][2]] if head == "sh" else
                           STAGE["wv" if head == "wv" else "tc"]["fwd"] + STAGE["wv" if head == "wv" else "tc"]["bwd"])
        if bad:
            fails.append(f"{tag}: {bad}")
        if A == 0:
            continue
        # localised dout and partition additivity (zero base)
        _, g_zero, _, _ = run(list(range(A)))
        total = {k: torch.zeros_like(g_zero[k]) for k in keys}
        worst_loc, worst_add = 0.0, 0.0
        for p, rows in enumerate(_row_sets(A, n_max)):
            dc, g, b, _ = run(rows)
            total = {k: total[k] + g[k] for k in keys}
            for k in keys:
                e = _rel(g[k], b.grads[k], b.grads_mag[k]) / unit
                worst_loc = max(worst_loc, e)
                if not e <= BWD_MULT:
                    fails.append(f"{tag} part {p} ({len(rows)} rows from {rows[0]}): d{k} {e:.3g} units")
            idx = torch.tensor(rows, device=DEV, dtype=torch.long)
            off = torch.ones(A, dtype=torch.bool, device=DEV)
            off[idx] = False
            if not torch.equal(dc[idx], dc_full[idx]):
                fails.append(f"{tag} part {p}: dcomps rows differ from the full call's")
            if not bool((dc[off] == 0).all()):
                fails.append(f"{tag} part {p}: dcomps non-zero on rows with zero dout")
        for k in keys:
            e = _rel(total[k], g_zero[k].double(), b_full.grads_mag[k])
            worst_add = max(worst_add, e)
            if not e <= ADD_TOL:
                fails.append(f"{tag}: sum over the parts of d{k} differs from the full call by {e:.3g}")
        errs[f"local/{tag}"], errs[f"additivity/{tag}"] = worst_loc, worst_add
    record_err(f"head_bwd:{variant}:{size}", A=A, mult=BWD_MULT, add_tol=ADD_TOL, **errs)
    assert not fails, f"{len(fails)} failures; first: " + "; ".join(fails[:6])


# ------------------------------------------------------------------ launch forms the classes do not reach
def test_fixed_count_and_ldf_forms():
    """The ops with n_dev = None (count = n_max) give the bits of the device-count launch; jt_head_bwd_tc on feature
    rows of pitch 28 gives the bits of pitch 32."""
    A = NSM * TM + 1
    fails = []
    for head in ("sh", "mlp", "wv"):
        I = _Inputs(head, A, seed=5)
        fprog, vprog = 0.65, 0.65
        stage = (ops.wv_stage if head == "wv" else ops.head_tc_stage)(A, DEV)
        outs = []
        for n_dev in (I.count, None):
            fd = torch.zeros((A, 32), device=DEV)
            rgb = torch.zeros((A, 4), device=DEV)
            if head == "sh":
                ops.app_basis_sh_fwd_tc(2, I.afs, I.samp, I.aidx, I.sidx, I.rays_d, S, True, I.wb, n_dev, A, fd, rgb,
                                        stage)
            elif head == "mlp":
                ops.app_basis_fwd_tc(2, I.afs, I.samp, I.aidx, I.sidx, I.rays_d, S, True, I.wb, n_dev, A, fd, stage)
                ops.head_mlp_fwd_tc(2, fd, *I.params, n_dev, A, fprog, vprog, rgb, stage)
            else:
                ops.wv_head_fwd_tc(I.comps, I.aidx, I.sidx, I.rays_d, S, True, I.wb, *I.params, n_dev, A, fprog, vprog,
                                   fd, rgb, stage)
            dout = torch.randn((A, 4), device=DEV, generator=torch.Generator(device=DEV).manual_seed(3))
            dc = torch.zeros((A, sum(I.afs.C)), device=DEV, dtype=torch.bfloat16 if head != "wv" else torch.float32)
            grads = [torch.zeros_like(t) for t in [I.wb] + I.params]
            if head == "sh":
                ops.sh_bwd_tc(dout, fd, I.wb, n_dev, A, dc, stage, grads[0])
            elif head == "mlp":
                ops.head_bwd_tc(dout, fd, I.wb, *I.params[0::2], n_dev, A, fprog, dc, stage, grads)
            else:
                ops.wv_head_bwd_tc(dout, fd, I.wb, *I.params[0::2], n_dev, A, fprog, dc, stage, grads)
            torch.cuda.synchronize()
            outs.append((fd.clone(), rgb.clone(), dc.clone()))
            if head == "mlp" and n_dev is not None:
                dc28 = torch.zeros_like(dc)
                fd28 = fd[:, :28].contiguous()
                ops.head_bwd_tc(dout, fd28, I.wb, *I.params[0::2], n_dev, A, fprog, dc28, stage, None)
                torch.cuda.synchronize()
                if not torch.equal(dc28, dc):
                    fails.append("mlp: dcomps from feature rows of pitch 28 differ from pitch 32")
        for name, a, b in zip(("featdir", "rgb", "dcomps"), outs[0], outs[1]):
            if not torch.equal(a, b):
                fails.append(f"{head}: {name} with a fixed count differs from the device count")
    assert not fails, fails
