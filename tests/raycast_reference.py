"""Float64 reference for the ray caster (jt_raycast, B200_VMSplit.raycast). It takes the kernel's fp32 sample depths and
points as input, applies the same first-sample and subdivision semantics as the kernel with a float64 predicate, and
ends with a float64 root of {alpha64(o + d t) >= level} (bisection of the predicate) in the final bracket.

The subdivision (`refine`) is written once for any dtype: run in float32 with the kernel's own predicate it replays
the kernel's rounds; run in float64 with alpha64 it is the reference."""
import torch

from density_grad_reference import density_and_grad


def field_alpha64(planes, lines, aabb, shift, act, length, inv=None, keep_fn=None):
    """alpha(xyz) = 1 - exp(-sigma64 * length) of the density field (density_grad_reference, float64), with the
    occupancy mask keep_fn(xyz) -> bool [n] applied as compute_alpha applies it. Returns (alpha_fn, grad_fn):
    grad_fn(xyz) = d alpha / d xyz."""
    def both(xyz):
        x = xyz.double()
        keep = keep_fn(x) if keep_fn is not None else None
        sigma, grad = density_and_grad(planes, lines, aabb, x, shift, act, inv=inv, keep=keep)
        a = 1.0 - torch.exp(-sigma * length)
        return a, (length * torch.exp(-sigma * length))[:, None] * grad
    return (lambda xyz: both(xyz)[0]), (lambda xyz: both(xyz)[1])


def in_box64(aabb, xyz):
    aabb = aabb.double()
    return ((xyz >= aabb[0]) & (xyz <= aabb[1])).all(dim=-1)


def first_inside(inside):
    """inside [n, S] bool -> index of the first True per row, -1 where there is none."""
    S = inside.shape[1]
    idx = torch.where(inside, torch.arange(S).expand_as(inside), torch.full_like(inside, S, dtype=torch.long))
    k = idx.min(dim=1).values
    return torch.where(k < S, k, torch.full_like(k, -1))


def _next_up(x):
    return torch.nextafter(x, torch.full_like(x, float("inf")))


def refine(lo, hi, inside_fn, P, max_rounds=64):
    """The kernel's refinement on brackets [lo, hi] (1-D tensors of one dtype; lo outside, hi inside): each round
    evaluates inside_fn at the P points t_j = min(lo + w j, hi), w = (hi - lo) / (P + 1), j = 1..P (every operation
    rounded in the tensors' dtype) and keeps the first inside point as hi and the point before it as lo, until
    hi - lo <= 2^-20 of the initial width or no value of the dtype lies strictly inside. inside_fn(rows [m], t [m, P])
    -> bool [m, P], rows indexing the brackets still refining. Returns (lo, hi, rounds)."""
    lo, hi = lo.clone(), hi.clone()
    stop = (hi - lo) * 2.0 ** -20
    rounds = torch.zeros(lo.shape, dtype=torch.long)
    j = torch.arange(1, P + 1, dtype=lo.dtype)
    inv = 1.0 / (P + 1)
    for _ in range(max_rounds):
        act = ((hi - lo) > stop) & (_next_up(lo) < hi)
        if not bool(act.any()):
            break
        a = act.nonzero().squeeze(1)
        l, h = lo[a], hi[a]
        w = (h - l) * inv
        tj = torch.minimum(l[:, None] + w[:, None] * j, h[:, None])
        ins = inside_fn(a, tj)
        first = first_inside(ins)
        got = first >= 0
        fi = first.clamp_min(0)
        new_hi = torch.where(got, tj.gather(1, fi[:, None]).squeeze(1), h)
        prev = tj.gather(1, (fi - 1).clamp_min(0)[:, None]).squeeze(1)
        new_lo = torch.where(got, torch.where(fi > 0, prev, l), tj[:, P - 1])
        lo[a], hi[a] = new_lo, new_hi
        rounds[a] += 1
    return lo, hi, rounds


def cast64(o, d, t_samp, pts_samp, inbox_samp, alpha_fn, aabb, level, P, bisect=80):
    """Float64 ray cast of rays o, d [n,3] on the marcher's fp32 samples: depths t_samp [n,S], points pts_samp [n,S,3]
    and box results inbox_samp [n,S]. A sample is inside iff inbox and alpha64(its fp32 point) >= level.
    k = the first inside sample (-1: miss); for k > 0 the bracket [t_{k-1}, t_k] is refined in float64 (inside iff
    in_box64 and alpha64 >= level at o + d t in float64), then t_star = the crossing of the predicate in the final
    bracket by bisection. k == 0: t_star = t_0. Returns dict(k, lo, hi (the refined bracket; lo = hi = t_0 for k == 0,
    hi = inf on a miss), t_star, alpha_samp [n,S]), float64."""
    o, d = o.double(), d.double()
    t_samp = t_samp.double()
    n, S = t_samp.shape
    pts = pts_samp.double()
    alpha_samp = torch.zeros((n, S), dtype=torch.float64)
    if inbox_samp.any():
        alpha_samp[inbox_samp] = alpha_fn(pts[inbox_samp])
    k = first_inside(inbox_samp & (alpha_samp >= level))
    lo = torch.full((n,), float("nan"), dtype=torch.float64)
    hi = torch.full((n,), float("inf"), dtype=torch.float64)
    got = k >= 0
    hi[got] = t_samp[got, k[got]]
    lo[got] = hi[got]
    t_star = hi.clone()

    def inside_at(rows, t):
        p = o[rows, None, :] + d[rows, None, :] * t[..., None]
        flat = p.reshape(-1, 3)
        ok = in_box64(aabb, flat)
        a = torch.zeros(flat.shape[0], dtype=torch.float64)
        if ok.any():
            a[ok] = alpha_fn(flat[ok])
        return (ok & (a >= level)).reshape(t.shape)

    ref = (k > 0).nonzero().squeeze(1)
    if ref.numel():
        lo_r, hi_r, _ = refine(t_samp[ref, k[ref] - 1], hi[ref], lambda a, t: inside_at(ref[a], t), P)
        lo[ref], hi[ref] = lo_r, hi_r
        for _ in range(bisect):
            mid = 0.5 * (lo_r + hi_r)
            ins = inside_at(ref, mid[:, None]).squeeze(1)
            lo_r, hi_r = torch.where(ins, lo_r, mid), torch.where(ins, mid, hi_r)
        t_star[ref] = hi_r
    return dict(k=k, lo=lo, hi=hi, t_star=t_star, alpha_samp=alpha_samp)
