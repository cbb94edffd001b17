"""float64 reference of the three shading heads and of their backward (plain torch, CPU or CUDA).

The heads map the appearance components of a sample to its colour:

  SH                feat = comps Wb^T [27];  pre = sum_k Y_k(dir) feat[c*9+k] + 0.5;          rgb = relu(pre)
  MLP_Fea           feat = comps Wb^T [27];  x = [feat | dir | PE(feat) | PE(dir)] [150];
                    pre = W3 relu(W2 relu(W1 x + b1) + b2) + b3;                           rgb = sigmoid(pre)
  MLP_Fea_WeakView  feat = comps Wb^T [20];  x = [feat | PE(feat)] [100];  h2 = relu(W2 relu(W1 x + b1) + b2);
                    pre = W3 [PE(dir) | h2] + b3;                                          rgb = sigmoid(pre)

PE is the reference's positional_encoding with two frequencies: per element [sin x, sin 2x, cos x, cos 2x] times the
annealing masks m_l = clamp(2 progress - l, 0, 1), formed in fp32 as both the kernels and the oracle form them.

Given `dout` = dL/d(pre) -- what jt_render_bwd hands the head, the output activation already folded in -- the
backward gives dcomps and the weight gradients dWb, dW1, db1, dW2, db2, dW3, db3.

Every output comes with its magnitude: the same chain evaluated on absolute values (|W| |x| per GEMM, the relu masks
applied, and |PE(x)| + 2^l m_l mag(x) per PE entry, as |PE'| <= 2^l m_l). A kernel whose operands
carry a relative error of u is then within a small multiple of u times the magnitude, element by element; the tests
state their bounds that way.

A relu unit whose float64 pre-activation lies within `amb` times its magnitude of 0 is ambiguous: a kernel with
operand unit u <= amb may take the other branch there. `ambiguous` flags the rows that hold such a unit. The forward
magnitudes keep such units (a kernel that takes the other branch stays within the bound); the backward uses the
exact float64 masks, so its callers give ambiguous rows a zero `dout`."""
from types import SimpleNamespace

import torch

F64 = torch.float64
SH_C0 = 0.28209479177387814
SH_C1 = 0.4886025119029199
SH_C2 = (1.0925484305920792, -1.0925484305920792, 0.31539156525252005, -1.0925484305920792, 0.5462742152960396)


def view_dirs(rays_d, sidx, aidx, n, S, normalize_dir):
    """View direction of appearance sample e < n: rays_d[sidx[aidx[e]] // S], divided by its norm when normalize_dir
    (NDC rays); float64."""
    ray = torch.div(sidx[aidx[:n].long()].long(), S, rounding_mode="floor")
    d = rays_d[ray].to(F64)
    if normalize_dir:
        d = d / torch.linalg.vector_norm(d, dim=1, keepdim=True)
    return d


def pe_masks(progress):
    """m_0, m_1 = clamp(2 progress - l, 0, 1), in fp32 (the kernels' fminf(fmaxf(p * 2.f - l, 0.f), 1.f))."""
    p2 = torch.tensor(progress, dtype=torch.float32) * 2
    return [float((p2 - l).clamp(0.0, 1.0)) for l in range(2)]


def pe(v, v_mag, progress):
    """PE of [n, E] values: [n, 4E] in element-major order [sin x, sin 2x, cos x, cos 2x] x masks, its magnitude, and
    the masks."""
    m0, m1 = pe_masks(progress)
    x2 = 2.0 * v
    val = torch.stack([torch.sin(v) * m0, torch.sin(x2) * m1, torch.cos(v) * m0, torch.cos(x2) * m1], -1)
    mag = val.abs() + torch.stack([m0 * v_mag, 2 * m1 * v_mag, m0 * v_mag, 2 * m1 * v_mag], -1)
    n, E = v.shape
    return val.reshape(n, 4 * E), mag.reshape(n, 4 * E), (m0, m1)


def pe_backward(g, g_mag, v, masks):
    """d/dv of sum(g * PE(v)) for g [n, 4E] (element-major), and its magnitude."""
    m0, m1 = masks
    g = g.reshape(*v.shape, 4)
    gm = g_mag.reshape(*v.shape, 4)
    s, c = torch.sin(v), torch.cos(v)
    s2, c2 = torch.sin(2 * v), torch.cos(2 * v)
    d = m0 * (c * g[..., 0] - s * g[..., 2]) + 2 * m1 * (c2 * g[..., 1] - s2 * g[..., 3])
    dm = m0 * (gm[..., 0] + gm[..., 2]) + 2 * m1 * (gm[..., 1] + gm[..., 3])
    return d, dm


def sh_basis(d):
    """The 9 real SH bases of degree 2 (eval_sh_bases) at directions d [n, 3]."""
    x, y, z = d.unbind(-1)
    return torch.stack([torch.full_like(x, SH_C0), -SH_C1 * y, SH_C1 * z, -SH_C1 * x, SH_C2[0] * x * y,
                        SH_C2[1] * y * z, SH_C2[2] * (2 * z * z - x * x - y * y), SH_C2[3] * x * z,
                        SH_C2[4] * (x * x - y * y)], -1)


def _lin(x, x_mag, w, b):
    w = w.to(F64)
    y, y_mag = x @ w.T, x_mag @ w.abs().T
    if b is not None:
        y, y_mag = y + b.to(F64), y_mag + b.to(F64).abs()
    return y, y_mag


def head_forward(shading, comps, dirs, wb, params=(), fprog=1.0, vprog=1.0, comps_mag=None, amb=2.0 ** -12):
    """Forward of one head on n samples.

    comps [n, sum C], dirs [n, 3] (view_dirs), wb [F, sum C], params (w1, b1, w2, b2, w3, b3) or () for SH; comps_mag
    (default |comps|) bounds the rounding of the components, e.g. vm_reference's value_bound for gathered components.
    Returns a SimpleNamespace of float64 tensors: feat, feat_mag, pre, pre_mag, rgb, ambiguous [n] (bool), and the
    intermediates head_backward needs."""
    f = SimpleNamespace(shading=shading, params=params, fprog=fprog, vprog=vprog)
    f.comps = comps.to(F64)
    f.comps_mag = f.comps.abs() if comps_mag is None else comps_mag.to(F64)
    f.dirs = dirs.to(F64)
    f.wb = wb.to(F64)
    f.feat, f.feat_mag = _lin(f.comps, f.comps_mag, f.wb, None)
    n = f.comps.shape[0]
    if shading == "SH":
        f.Y = sh_basis(f.dirs)
        fv = f.feat.view(n, 3, 9)
        fm = f.feat_mag.view(n, 3, 9)
        f.pre = (fv * f.Y[:, None]).sum(-1) + 0.5
        f.pre_mag = (fm * f.Y.abs()[:, None]).sum(-1) + 0.5
        f.rgb = torch.relu(f.pre)
        f.ambiguous = torch.zeros(n, dtype=torch.bool, device=f.comps.device)
        return f
    w1, b1, w2, b2, w3, b3 = params
    pf, pf_mag, f.fmasks = pe(f.feat, f.feat_mag, fprog)
    pd, pd_mag, _ = pe(f.dirs, f.dirs.abs(), vprog)
    if shading == "MLP_Fea":
        f.x = torch.cat([f.feat, f.dirs, pf, pd], 1)
        f.x_mag = torch.cat([f.feat_mag, f.dirs.abs(), pf_mag, pd_mag], 1)
    elif shading == "MLP_Fea_WeakView":
        f.x = torch.cat([f.feat, pf], 1)
        f.x_mag = torch.cat([f.feat_mag, pf_mag], 1)
    else:
        raise ValueError(shading)
    f.p1, f.p1_mag = _lin(f.x, f.x_mag, w1, b1)
    keep1 = f.p1 > -amb * f.p1_mag
    f.h1, f.h1_mag = torch.relu(f.p1), f.p1_mag * keep1
    f.p2, f.p2_mag = _lin(f.h1, f.h1_mag, w2, b2)
    keep2 = f.p2 > -amb * f.p2_mag
    f.h2, f.h2_mag = torch.relu(f.p2), f.p2_mag * keep2
    if shading == "MLP_Fea":
        f.mid, f.mid_mag = f.h2, f.h2_mag
    else:
        f.mid, f.mid_mag = torch.cat([pd, f.h2], 1), torch.cat([pd_mag, f.h2_mag], 1)
    f.pre, f.pre_mag = _lin(f.mid, f.mid_mag, w3, b3)
    f.rgb = torch.sigmoid(f.pre)
    f.ambiguous = ((f.p1.abs() <= amb * f.p1_mag).any(1) | (f.p2.abs() <= amb * f.p2_mag).any(1))
    return f


def head_backward(f, dout):
    """Backward of head_forward's head for dout = dL/d(pre) [n, >= 3] (columns past 3 ignored). The relu masks are
    the exact float64 ones (p > 0). Returns a SimpleNamespace: dcomps, dfeat and the weight gradients `grads` (a dict
    with keys wb, w1, b1, w2, b2, w3, b3; wb alone for SH), each with its magnitude (dcomps_mag, grads_mag)."""
    g = dout[:, :3].to(F64)
    ga = g.abs()
    b = SimpleNamespace(grads={}, grads_mag={})
    if f.shading == "SH":
        b.dfeat = (g[:, :, None] * f.Y[:, None]).reshape(g.shape[0], 27)
        b.dfeat_mag = (ga[:, :, None] * f.Y.abs()[:, None]).reshape(g.shape[0], 27)
    else:
        w1, _, w2, _, w3, _ = (t.to(F64) for t in f.params)
        m1, m2 = (f.p1 > 0).to(F64), (f.p2 > 0).to(F64)
        nv = f.mid.shape[1] - f.h2.shape[1]          # PE(dir) columns ahead of h2 in layer 3's input (WeakView)
        dh2 = (g @ w3)[:, nv:] * m2
        dh2_mag = (ga @ w3.abs())[:, nv:] * m2
        dh1, dh1_mag = (dh2 @ w2) * m1, (dh2_mag @ w2.abs()) * m1
        dx, dx_mag = dh1 @ w1, dh1_mag @ w1.abs()
        F = f.feat.shape[1]
        o = F + (3 if f.shading == "MLP_Fea" else 0)  # PE(feat) columns start after [feat | dir] or [feat]
        dpe, dpe_mag = pe_backward(dx[:, o:o + 4 * F], dx_mag[:, o:o + 4 * F], f.feat, f.fmasks)
        b.dfeat, b.dfeat_mag = dx[:, :F] + dpe, dx_mag[:, :F] + dpe_mag
        b.grads.update(w1=dh1.T @ f.x, b1=dh1.sum(0), w2=dh2.T @ f.h1, b2=dh2.sum(0), w3=g.T @ f.mid, b3=g.sum(0))
        b.grads_mag.update(w1=dh1_mag.T @ f.x_mag, b1=dh1_mag.sum(0), w2=dh2_mag.T @ f.h1_mag, b2=dh2_mag.sum(0),
                           w3=ga.T @ f.mid_mag, b3=ga.sum(0))
    b.dcomps, b.dcomps_mag = b.dfeat @ f.wb, b.dfeat_mag @ f.wb.abs()
    b.grads["wb"], b.grads_mag["wb"] = b.dfeat.T @ f.comps, b.dfeat_mag.T @ f.comps_mag
    return b
