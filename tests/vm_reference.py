"""float64 reference of the VM feature gather and of its adjoint (plain torch, CPU or CUDA).

One sample u (normalised coordinates in [-1, 1]^3) reads, for each of the three plane / line pairs i, a bilinear tap
of the channel-last plane P_i [H,W,C] at (u[MAT[i][0]], u[MAT[i][1]]) and a linear tap of the line L_i [L,C] at
u[VEC[i]] (ATen grid_sampler, align_corners=True, zero padding). The density feature is sum_i sum_c P_ic L_ic, the
appearance components are the products P_ic L_ic themselves. Given the upstream gradient `gin` this evaluates

  * the forward value,
  * the six factor gradients (what jt_vm_scatter_rays and jt_vm_gather_bwd accumulate),
  * the per-sample coordinate gradient du = dL/du (the dsamp output of jt_vm_gather_bwd),
  * the per-ray sums d_o = sum_j du_j * inv and d_d = sum_j du_j * t_j * inv (what jt_vm_scatter_rays adds into
    d/d rays_o and d/d rays_d),

each with the sum of the absolute values of its terms, against which tolerances are stated.

Tap positions (tap_dtype="fp32", the default) are formed in fp32 exactly as the kernels form them (make_tap in
jt_common.cuh, make_pos in vm_scatter.cu): x = (u + 1) * (0.5 (n - 1)), floor, fraction, the in-range masks, the
axis weights (1 - f) m0 and f m1, and the plane weight as the fp32 product of two axis weights. Everything after
that is float64, so what separates a correct kernel from this reference is the rounding of its fp32 sums.
tap_dtype="float64" forms the positions in float64, as float64 autograd of F.grid_sample does."""
from types import SimpleNamespace

import torch

MAT = ((0, 1), (0, 2), (1, 2))     # plane i: x axis (W) samples u[MAT[i][0]], y axis (H) samples u[MAT[i][1]]
VEC = (2, 1, 0)                    # line i samples u[VEC[i]]


def axis_taps(g, n, tap_dtype="fp32"):
    """Tap setup on an axis of n texels: clamped indices i0 / i1 (always safe to index), weights w0 / w1 (zero for
    an out-of-range tap), in-range masks m0 / m1 and d index / d g. fp32 positions follow make_tap (jt_common.cuh)."""
    dt = torch.float32 if tap_dtype == "fp32" else torch.float64
    g = g.to(dt)
    scale = torch.tensor(0.5 * (n - 1), dtype=dt, device=g.device)
    x = (g + 1.0) * scale
    xf = torch.floor(x)
    f = x - xf
    i0 = torch.clamp(torch.nan_to_num(xf, nan=-2.0), -2.0, float(n)).to(torch.int64)   # NaN -> -2: both out of range
    i1 = i0 + 1
    m0 = ((i0 >= 0) & (i0 < n)).to(dt)
    m1 = ((i1 >= 0) & (i1 < n)).to(dt)
    return SimpleNamespace(i0=i0.clamp(0, n - 1), i1=i1.clamp(0, n - 1), w0=(1.0 - f) * m0, w1=f * m1,
                           m0=m0, m1=m1, scale=0.5 * (n - 1))


def vm_adjoint(planes, lines, samp, n=None, slot=None, gin=None, sidx=None, S=None, n_rays=None, inv=(1.0, 1.0, 1.0),
               tap_dtype="fp32", chunk=1 << 17):
    """Reference of one VM factor group.

    planes: three [H,W,C] tensors, lines: three [L,C] tensors (any float dtype; read as float64).
    samp:   [V,4] records (u_x, u_y, u_z, t); element e of the list reads record slot[e] (or e without `slot`).
    n:      number of list elements (default: len(slot) or V).
    gin:    None (forward only), [n] (density: dL/d feature) or [n, sum C] (appearance: dL/d components), any dtype.
    sidx, S, n_rays: with these, d_o / d_d are summed per ray (ray = sidx[slot[e]] // S) and scaled by `inv`.

    Returns a SimpleNamespace of float64 tensors on samp's device:
      value [n] (gin None or 1-D) or [n, sum C]; value_mag: sum of |P_ic L_ic| terms; value_bound: the same with
        every interpolation expanded (sum |w P| * sum |w L|), a bound of every partial sum of the kernels' forward;
      gp / gl: the 6 factor gradients (lists of [H,W,C] / [L,C]) and gp_mag / gl_mag;
      du [n,3], du_mag; du_plane [3,n,3]: the contribution of plane / line pair i;
      d_o, d_d [n_rays,3] and their _mag; d_o_plane, d_d_plane [3,n_rays,3]."""
    dev = samp.device
    f64 = torch.float64
    n = n if n is not None else (slot.shape[0] if slot is not None else samp.shape[0])
    C = [p.shape[2] for p in planes]
    off = [0, C[0], C[0] + C[1]]
    app = gin is not None and gin.dim() == 2
    r = SimpleNamespace()
    vshape = (n, sum(C)) if app else (n,)
    r.value, r.value_mag, r.value_bound = (torch.zeros(vshape, dtype=f64, device=dev) for _ in range(3))
    if gin is not None:
        r.gp = [torch.zeros(p.shape, dtype=f64, device=dev) for p in planes]
        r.gl = [torch.zeros(l.shape, dtype=f64, device=dev) for l in lines]
        r.gp_mag = [torch.zeros_like(g) for g in r.gp]
        r.gl_mag = [torch.zeros_like(g) for g in r.gl]
        r.du_plane = torch.zeros((3, n, 3), dtype=f64, device=dev)
        r.du_mag_plane = torch.zeros((3, n, 3), dtype=f64, device=dev)
    for i in range(3):
        H, W, _ = planes[i].shape
        L = lines[i].shape[0]
        Pf = planes[i].reshape(H * W, C[i]).to(f64)
        Lf = lines[i].to(f64)
        ax, ay, al = MAT[i][0], MAT[i][1], VEC[i]
        for e0 in range(0, n, chunk):
            e1 = min(e0 + chunk, n)
            j = slot[e0:e1].long() if slot is not None else torch.arange(e0, e1, device=dev)
            u = samp[j, :3].float() if tap_dtype == "fp32" else samp[j, :3].to(f64)
            tx, ty, tl = axis_taps(u[:, ax], W, tap_dtype), axis_taps(u[:, ay], H, tap_dtype), axis_taps(u[:, al], L, tap_dtype)
            idx = [ty.i0 * W + tx.i0, ty.i0 * W + tx.i1, ty.i1 * W + tx.i0, ty.i1 * W + tx.i1]      # 00 10 01 11
            w = [(tx.w0 * ty.w0).to(f64), (tx.w1 * ty.w0).to(f64), (tx.w0 * ty.w1).to(f64), (tx.w1 * ty.w1).to(f64)]
            wl = [tl.w0.to(f64), tl.w1.to(f64)]
            p = [Pf[k] for k in idx]
            la, lb = Lf[tl.i0], Lf[tl.i1]
            pv = sum(wk[:, None] * pk for wk, pk in zip(w, p))
            pa = sum(wk[:, None] * pk.abs() for wk, pk in zip(w, p))
            lv = wl[0][:, None] * la + wl[1][:, None] * lb
            lva = wl[0][:, None] * la.abs() + wl[1][:, None] * lb.abs()
            prod = pv * lv
            if app:
                r.value[e0:e1, off[i]:off[i] + C[i]] = prod
                r.value_mag[e0:e1, off[i]:off[i] + C[i]] = prod.abs()
                r.value_bound[e0:e1, off[i]:off[i] + C[i]] = pa * lva
            else:
                r.value[e0:e1] += prod.sum(1)
                r.value_mag[e0:e1] += prod.abs().sum(1)
                r.value_bound[e0:e1] += (pa * lva).sum(1)
            if gin is None:
                continue
            gc = gin[e0:e1, off[i]:off[i] + C[i]].to(f64) if app else gin[e0:e1].to(f64)[:, None]
            g_pl, g_pl_a = gc * lv, gc.abs() * lva          # dL / d(interpolated plane value)
            g_ln, g_ln_a = gc * pv, gc.abs() * pa           # dL / d(interpolated line value)
            for k in range(4):
                r.gp[i].view(H * W, C[i]).index_add_(0, idx[k], w[k][:, None] * g_pl)
                r.gp_mag[i].view(H * W, C[i]).index_add_(0, idx[k], w[k][:, None] * g_pl_a)
            for k, ik in enumerate((tl.i0, tl.i1)):
                r.gl[i].index_add_(0, ik, wl[k][:, None] * g_ln)
                r.gl_mag[i].index_add_(0, ik, wl[k][:, None] * g_ln_a)
            # d/d index, ATen grid_sampler_2d_backward: an out-of-range tap reads as 0
            mx0, mx1, my0, my1 = (t.to(f64)[:, None] for t in (tx.m0, tx.m1, ty.m0, ty.m1))
            ml0, ml1 = tl.m0.to(f64)[:, None], tl.m1.to(f64)[:, None]
            wx0, wx1, wy0, wy1 = (t.to(f64)[:, None] for t in (tx.w0, tx.w1, ty.w0, ty.w1))
            p00, p10, p01, p11 = p
            dx = wy0 * (mx1 * p10 - mx0 * p00) + wy1 * (mx1 * p11 - mx0 * p01)
            dxa = wy0 * (mx1 * p10.abs() + mx0 * p00.abs()) + wy1 * (mx1 * p11.abs() + mx0 * p01.abs())
            dy = wx0 * (my1 * p01 - my0 * p00) + wx1 * (my1 * p11 - my0 * p10)
            dya = wx0 * (my1 * p01.abs() + my0 * p00.abs()) + wx1 * (my1 * p11.abs() + my0 * p10.abs())
            dl, dla = ml1 * lb - ml0 * la, ml1 * lb.abs() + ml0 * la.abs()
            for a, s, d, da, gg, gga in ((ax, tx.scale, dx, dxa, g_pl, g_pl_a), (ay, ty.scale, dy, dya, g_pl, g_pl_a),
                                         (al, tl.scale, dl, dla, g_ln, g_ln_a)):
                r.du_plane[i, e0:e1, a] = (gg * d).sum(1) * s
                r.du_mag_plane[i, e0:e1, a] = (gga * da).sum(1) * s
    if gin is None:
        return r
    r.du, r.du_mag = r.du_plane.sum(0), r.du_mag_plane.sum(0)
    if sidx is not None:
        j = slot[:n].long() if slot is not None else torch.arange(n, device=dev)
        ray = (sidx[j].long() // S)
        t = samp[j, 3].to(f64)[:, None]
        invt = torch.tensor(inv, dtype=f64, device=dev)
        r.d_o_plane, r.d_d_plane, r.d_o_mag_plane, r.d_d_mag_plane = (
            torch.zeros((3, n_rays, 3), dtype=f64, device=dev) for _ in range(4))
        for i in range(3):
            r.d_o_plane[i].index_add_(0, ray, r.du_plane[i] * invt)
            r.d_d_plane[i].index_add_(0, ray, r.du_plane[i] * t * invt)
            r.d_o_mag_plane[i].index_add_(0, ray, r.du_mag_plane[i] * invt.abs())
            r.d_d_mag_plane[i].index_add_(0, ray, r.du_mag_plane[i] * t.abs() * invt.abs())
        r.d_o, r.d_d = r.d_o_plane.sum(0), r.d_d_plane.sum(0)
        r.d_o_mag, r.d_d_mag = r.d_o_mag_plane.sum(0), r.d_d_mag_plane.sum(0)
    return r


def density_feature(planes, lines, u):
    """float64 density feature sum_i sum_c P_ic(u) L_ic(u) with fp32 tap weights, and the sum of |P_ic L_ic|."""
    samp = torch.zeros((u.shape[0], 4), dtype=torch.float32, device=u.device)
    samp[:, :3] = u
    r = vm_adjoint(planes, lines, samp)
    return r.value, r.value_mag
