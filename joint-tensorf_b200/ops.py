"""Torch-tensor wrappers over the C ABI (include/jt_vm.h) + the autograd glue.

PyTorch is plumbing here: it owns device memory and the CUDA stream, and its
autograd engine calls our backward kernels. All arithmetic of the hot path is in
csrc/*.cu. Nothing in this file computes on the CPU or falls back to ATen
operators for the hot path.
"""
import contextlib
import ctypes
import math

import torch

from . import _lib
from ._lib import check, floats, ints, longlongs, ptrs

MAT_MODE = ((0, 1), (0, 2), (1, 2))   # reference tensorBase.py:405
VEC_MODE = (2, 1, 0)                  # reference tensorBase.py:406


# ------------------------------------------------------------------ per-kernel timing (bench.py)
class KernelTimer:
    """Optional CUDA-event timing around each C-ABI call (enabled by bench.py for the
    roofline breakdown; off in normal runs so the hot path records no events)."""

    def __init__(self):
        self.enabled = False
        self.records = []      # (name, start_event, end_event)

    @contextlib.contextmanager
    def span(self, name):
        if not self.enabled:
            yield
            return
        s = torch.cuda.Event(enable_timing=True)
        e = torch.cuda.Event(enable_timing=True)
        s.record()
        yield
        e.record()
        self.records.append((name, s, e))

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for name, s, e in self.records:
            tot, cnt = out.get(name, (0.0, 0))
            out[name] = (tot + s.elapsed_time(e), cnt + 1)
        self.records = []
        return out


TIMER = KernelTimer()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return 0 if t is None else t.data_ptr()


def _need_cuda(t, name):
    if not t.is_cuda:
        raise _lib.JtError(f"{name} must be a CUDA tensor: this path has no CPU implementation")


# ------------------------------------------------------------------ factors
def phys_cl(x):
    """[1,C,H,W] tensor -> its channel-last physical view [H,W,C] (contiguous fp32)."""
    assert x.dim() == 4 and x.shape[0] == 1, x.shape
    xp = x.permute(0, 2, 3, 1)
    if not xp.is_contiguous():
        xp = xp.contiguous()
    if xp.dtype != torch.float32:
        xp = xp.float()
    return xp[0]


class FactorSet:
    """Three planes + three lines in channel-last physical form and their dims. `store` (optional) is a list of
    six bf16 buffers holding the same values: the kernels then gather from those (dims[12] = 1) while `planes` /
    `lines` stay the fp32 tensors the gradients belong to."""

    def __init__(self, planes, lines, store=None):
        self.planes = [phys_cl(p) for p in planes]            # [H,W,C]
        self.lines = [phys_cl(l)[:, 0, :] for l in lines]     # [L,C]
        self.C = [p.shape[2] for p in self.planes]
        for i in range(3):
            if self.C[i] % 4 != 0 or self.lines[i].shape[1] != self.C[i]:
                raise _lib.JtError(f"component count {self.C[i]} must be a multiple of 4 and match its line")
        self.store = store
        self.dims = ints([p.shape[0] for p in self.planes] + [p.shape[1] for p in self.planes] +
                         [l.shape[0] for l in self.lines] + self.C + [1 if store is not None else 0])
        src = store if store is not None else self.planes + self.lines
        self.ptrs = ptrs([t.data_ptr() for t in src])
        self.ctot = sum(self.C)

    def with_bf16_store(self, cache=None):
        """The same factors with a bf16 gather-side copy (one jt_cast_bf16_multi launch). `cache`: dict reused
        across calls; an entry is valid while the source tensor's storage and version counter are unchanged
        (inference renders thousands of chunks from the same factors)."""
        srcs = self.planes + self.lines
        key = tuple((t.data_ptr(), t._version, tuple(t.shape)) for t in srcs)
        if cache is not None and cache.get("key") == key:
            store = cache["store"]
        else:
            store = [torch.empty(t.shape, device=t.device, dtype=torch.bfloat16) for t in srcs]
            cast_bf16_multi(srcs, store)
            if cache is not None:
                cache["key"], cache["store"] = key, store
        fs = FactorSet.__new__(FactorSet)
        fs.planes, fs.lines, fs.C, fs.ctot, fs.store = self.planes, self.lines, self.C, self.ctot, store
        fs.dims = ints(list(self.dims)[:12] + [1])
        fs.ptrs = ptrs([t.data_ptr() for t in store])
        return fs

    def zero_grads(self):
        gp = [torch.zeros_like(p) for p in self.planes]
        gl = [torch.zeros_like(l) for l in self.lines]
        return gp, gl

    @staticmethod
    def grads_as_nchw(gp, gl):
        """physical [H,W,C] / [L,C] gradients -> logical [1,C,H,W] / [1,C,L,1] views."""
        return ([g.unsqueeze(0).permute(0, 3, 1, 2) for g in gp],
                [g.unsqueeze(0).unsqueeze(2).permute(0, 3, 1, 2) for g in gl])


def cast_bf16_multi(srcs, dsts):
    """dsts[i] = bf16(srcs[i]) for up to 12 contiguous fp32 arrays in one launch (csrc/factor_store.cu)."""
    for a, b in zip(srcs, dsts):
        _need_cuda(a, "factor")
        assert a.is_contiguous() and b.is_contiguous() and a.dtype == torch.float32 and b.dtype == torch.bfloat16
    with TIMER.span("cast_bf16"):
        check(_lib.lib().jt_cast_bf16_multi(len(srcs), ptrs([a.data_ptr() for a in srcs]),
                                            ptrs([b.data_ptr() for b in dsts]), longlongs([a.numel() for a in srcs]),
                                            _stream()), "jt_cast_bf16_multi")


# ------------------------------------------------------------------ K1
def sample_ray_dense(rays_o, rays_d, aux, ndc, n_samples, geom, mask=None):
    _need_cuda(rays_o, "rays_o")
    n = rays_o.shape[0]
    dev = rays_o.device
    pts = torch.empty((n, n_samples, 3), device=dev)
    z = torch.empty((n, n_samples), device=dev)
    valid = torch.empty((n, n_samples), device=dev, dtype=torch.uint8)
    mb, md, mg = (mask.bits, mask.h_dims, mask.h_geom) if mask is not None else (None, None, None)
    with TIMER.span("sample_ray_dense"):
        check(_lib.lib().jt_sample_ray_dense(_p(rays_o), _p(rays_d), _p(aux), int(ndc), n, n_samples, geom,
                                             _p(mb), md, mg, _p(pts), _p(z), _p(valid), _stream()),
              "jt_sample_ray_dense")
    return pts, z, valid.bool()


class Compacted:
    """Result of jt_march_compact (all device tensors, capacity N*S)."""
    __slots__ = ("n_rays", "n_samples", "cap", "ray_off", "sidx", "samp", "dist", "count")


def march_compact(rays_o, rays_d, aux, ndc, n_samples, geom, mask=None):
    _need_cuda(rays_o, "rays_o")
    n = rays_o.shape[0]
    dev = rays_o.device
    cap = max(n * n_samples, 1)
    c = Compacted()
    c.n_rays, c.n_samples, c.cap = n, n_samples, cap
    ray_cnt = torch.empty((max(n, 1),), device=dev, dtype=torch.int32)
    c.ray_off = torch.zeros((n + 1,), device=dev, dtype=torch.int32)
    c.sidx = torch.empty((cap,), device=dev, dtype=torch.int32)
    c.samp = torch.empty((cap, 4), device=dev)
    c.dist = torch.empty((cap,), device=dev)
    mb, md, mg = (mask.bits, mask.h_dims, mask.h_geom) if mask is not None else (None, None, None)
    with TIMER.span("march_compact"):
        check(_lib.lib().jt_march_compact(_p(rays_o), _p(rays_d), _p(aux), int(ndc), n, n_samples, geom,
                                          _p(mb), md, mg, _p(ray_cnt), _p(c.ray_off), _p(c.sidx), _p(c.samp),
                                          _p(c.dist), _stream()), "jt_march_compact")
    c.count = c.ray_off[n:n + 1]          # device scalar V (never read on the host in the hot path)
    return c


# ------------------------------------------------------------------ K2
def vm_gather_fwd(app, fs, samp, slot, n_dev, n_max, out):
    with TIMER.span("vm_app_fwd" if app else "vm_density_fwd"):
        check(_lib.lib().jt_vm_gather_fwd(int(app), fs.ptrs, fs.dims, _p(samp), _p(slot), _p(n_dev), int(n_max),
                                          _p(out), _stream()), "jt_vm_gather_fwd")


def vm_gather_bwd(app, fs, gp, gl, samp, slot, n_dev, n_max, gin, dsamp, accumulate):
    gptrs = ptrs([g.data_ptr() for g in gp] + [g.data_ptr() for g in gl])
    with TIMER.span("vm_app_bwd" if app else "vm_density_bwd"):
        check(_lib.lib().jt_vm_gather_bwd(int(app), fs.ptrs, gptrs, fs.dims, _p(samp), _p(slot), _p(n_dev),
                                          int(n_max), _p(gin), _p(dsamp), int(accumulate), _stream()),
              "jt_vm_gather_bwd")


def vm_scatter_rays(app, fs, gp, gl, samp, slot, sidx, n_dev, n_max, gin, n_samples, h_inv, d_o, d_d, max_ctas=0,
                    plane_mask=7):
    """Run-merged factor-gradient scatter + per-ray pose-path gradients (vm_scatter.cu). plane_mask: which of the
    three plane / line pairs this launch walks (7 = all). gp = gl = None: coordinate-only walk (d_o / d_d alone)."""
    gptrs = None if gp is None else ptrs([g.data_ptr() for g in gp] + [g.data_ptr() for g in gl])
    with TIMER.span("vm_app_bwd" if app else "vm_density_bwd"):
        check(_lib.lib().jt_vm_scatter_rays(int(app), fs.ptrs, gptrs, fs.dims, _p(samp), _p(slot), _p(sidx),
                                            _p(n_dev), int(n_max), _p(gin), int(gin.dtype == torch.bfloat16),
                                            int(n_samples), h_inv, _p(d_o), _p(d_d), int(max_ctas), int(plane_mask),
                                            _stream()),
              "jt_vm_scatter_rays")


# ------------------------------------------------------------------ K3
def gemm_nt(x, ldx, w, ldw, w_kn, bias, y, ldy, mask, ldm, m_dev, m_max, n, k, act, name="gemm_nt",
            x_off=0, w_off=0, y_off=0, mask_off=0):
    """offsets are in floats (used to address column blocks of a wider buffer)."""
    with TIMER.span(name):
        check(_lib.lib().jt_gemm_nt(_p(x) + 4 * x_off, ldx, _p(w) + 4 * w_off, ldw, int(w_kn), _p(bias),
                                    _p(y) + 4 * y_off, ldy, (_p(mask) + 4 * mask_off) if mask is not None else 0,
                                    ldm, _p(m_dev), int(m_max), n, k, act, _stream()), "jt_gemm_nt")


def gemm_tn(dy, ldy, x, ldx, m_dev, m_max, n, k, dw, ldw, db, name="gemm_tn", dy_off=0, x_off=0, dw_off=0):
    with TIMER.span(name):
        check(_lib.lib().jt_gemm_tn(_p(dy) + 4 * dy_off, ldy, _p(x) + 4 * x_off, ldx, _p(m_dev), int(m_max), n, k,
                                    _p(dw) + 4 * dw_off, ldw, _p(db), _stream()), "jt_gemm_tn")


def pe_encode(bwd, app_dim, fea_pe, view_pe, mode, fprog, vprog, n_samples, normalize_dir, feat, ldf, aidx, sidx,
              rays_d, n_dev, n_max, out, ldo, out2=None, ldo2=0, din=None, ldi=0):
    with TIMER.span("pe_bwd" if bwd else "pe_fwd"):
        check(_lib.lib().jt_pe_encode(int(bwd), app_dim, fea_pe, view_pe, mode, float(fprog), float(vprog),
                                      n_samples, int(normalize_dir), _p(feat), ldf, _p(aidx), _p(sidx), _p(rays_d),
                                      _p(n_dev), int(n_max), _p(out), ldo, _p(out2), ldo2, _p(din), ldi, _stream()),
              "jt_pe_encode")


def sh_shade(bwd, feat, ldf, aidx, sidx, rays_d, n_samples, normalize_dir, n_dev, n_max, rgb, dout, dfeat, ldd):
    with TIMER.span("sh_bwd" if bwd else "sh_fwd"):
        check(_lib.lib().jt_sh_shade(int(bwd), _p(feat), ldf, _p(aidx), _p(sidx), _p(rays_d), n_samples,
                                     int(normalize_dir), _p(n_dev), int(n_max), _p(rgb), _p(dout), _p(dfeat), ldd,
                                     _stream()), "jt_sh_shade")


# ------------------------------------------------------------------ K3 tensor-core path
def tc_selftest(mode, a, b, k, n, ma=0):
    d = torch.zeros((128, n), device=a.device)
    check(_lib.lib().jt_tc_selftest(mode, _p(a), a.shape[1], _p(b), b.shape[1], _p(d), k, n, ma, _stream()),
          "jt_tc_selftest")
    return d


def head_tc_stage(n_max, device):
    """Scratch for the bf16 operand tiles exchanged between the tensor-core head kernels."""
    nbytes = int(_lib.lib().jt_head_tc_stage_bytes(int(n_max)))
    return torch.empty((nbytes,), device=device, dtype=torch.uint8)


def app_basis_fwd_tc(split, fs, samp, aidx, sidx, rays_d, n_samples, normalize_dir, wb, n_dev, n_max, featdir,
                     stage=None):
    """appearance gather + basis_mat on tensor cores -> featdir [A][32] (feat | dir)."""
    with TIMER.span("app_basis_fwd_tc"):
        check(_lib.lib().jt_app_basis_fwd_tc(split, fs.ptrs, fs.dims, _p(samp), _p(aidx), _p(sidx), _p(rays_d),
                                             int(n_samples), int(normalize_dir), _p(wb), _p(n_dev), int(n_max),
                                             _p(featdir), _p(stage), _stream()), "jt_app_basis_fwd_tc")


def app_basis_sh_fwd_tc(split, fs, samp, aidx, sidx, rays_d, n_samples, normalize_dir, wb, n_dev, n_max, featdir, rgb,
                        stage=None):
    """appearance gather + basis_mat + SHRender in one kernel -> rgb [A][4]; featdir [A][32] keeps the view dir."""
    with TIMER.span("app_basis_sh_fwd_tc"):
        check(_lib.lib().jt_app_basis_sh_fwd_tc(split, fs.ptrs, fs.dims, _p(samp), _p(aidx), _p(sidx), _p(rays_d),
                                                int(n_samples), int(normalize_dir), _p(wb), _p(n_dev), int(n_max),
                                                _p(featdir), _p(rgb), _p(stage), _stream()), "jt_app_basis_sh_fwd_tc")


def sh_bwd_tc(dout, featdir, wb, n_dev, n_max, dcomps, stage, g_basis):
    """g_basis [27][144] zero-initialised by the caller (accumulated), or None (frozen basis_mat; stage may be None)."""
    with TIMER.span("sh_bwd_tc"):
        check(_lib.lib().jt_sh_bwd_tc(_p(dout), _p(featdir), int(featdir.shape[1]), _p(wb), _p(n_dev), int(n_max),
                                      _p(dcomps), int(dcomps.dtype == torch.bfloat16), _p(stage), _p(g_basis),
                                      _stream()), "jt_sh_bwd_tc")


def head_mlp_fwd_tc(split, featdir, w1, b1, w2, b2, w3, b3, n_dev, n_max, fprog, vprog, rgb, stage=None):
    with TIMER.span("head_mlp_fwd_tc"):
        check(_lib.lib().jt_head_mlp_fwd_tc(split, _p(featdir), _p(w1), _p(b1), _p(w2), _p(b2), _p(w3), _p(b3),
                                            _p(n_dev), int(n_max), float(fprog), float(vprog), _p(rgb), _p(stage),
                                            _stream()), "jt_head_mlp_fwd_tc")


def head_bwd_tc(dout, feat, wb, w1, w2, w3, n_dev, n_max, fprog, dcomps, stage, grads):
    """grads = (gWb, gW1, gb1, gW2, gb2, gW3, gb3), zero-initialised by the caller, or None (no weight gradients).
    feat: [A][ldf] rows whose first 27 floats are the basis projection (ldf = 28 or 32)."""
    grads = grads if grads is not None else (None,) * 7
    with TIMER.span("head_bwd_tc"):
        check(_lib.lib().jt_head_bwd_tc(_p(dout), _p(feat), int(feat.shape[1]), _p(wb), _p(w1), _p(w2), _p(w3), _p(n_dev), int(n_max),
                                        float(fprog), _p(dcomps), int(dcomps.dtype == torch.bfloat16), _p(stage),
                                        *[_p(g) for g in grads], _stream()),
              "jt_head_bwd_tc")


def wv_stage(n_max, device):
    """Scratch for the bf16 operand tiles exchanged between the WeakView tensor-core head kernels."""
    nbytes = int(_lib.lib().jt_wv_stage_bytes(int(n_max)))
    return torch.empty((nbytes,), device=device, dtype=torch.uint8)


def wv_head_fwd_tc(comps, aidx, sidx, rays_d, n_samples, normalize_dir, wb, w1, b1, w2, b2, w3, b3, n_dev, n_max, fprog,
                   vprog, featdir, rgb, stage=None):
    """basis_mat + PE + MLPRender_Fea_WeakView on tensor cores (csrc/weakview_tc.cu): comps [A][60] -> rgb [A][4]."""
    with TIMER.span("wv_head_fwd_tc"):
        check(_lib.lib().jt_wv_head_fwd_tc(_p(comps), _p(aidx), _p(sidx), _p(rays_d), int(n_samples), int(normalize_dir),
                                           _p(wb), _p(w1), _p(b1), _p(w2), _p(b2), _p(w3), _p(b3), _p(n_dev), int(n_max),
                                           float(fprog), float(vprog), _p(featdir), _p(rgb), _p(stage), _stream()),
              "jt_wv_head_fwd_tc")


def wv_head_bwd_tc(dout, featdir, wb, w1, w2, w3, n_dev, n_max, fprog, dcomps, stage, grads):
    """grads = (gWb, gW1, gb1, gW2, gb2, gW3, gb3), zero-initialised by the caller, or None (no weight gradients);
    dcomps [A][60] fp32."""
    grads = grads if grads is not None else (None,) * 7
    with TIMER.span("wv_head_bwd_tc"):
        check(_lib.lib().jt_wv_head_bwd_tc(_p(dout), _p(featdir), _p(wb), _p(w1), _p(w2), _p(w3), _p(n_dev), int(n_max),
                                           float(fprog), _p(dcomps), _p(stage), *[_p(g) for g in grads], _stream()),
              "jt_wv_head_bwd_tc")


# ------------------------------------------------------------------ K5
def host_taps(kernel):
    """Blur taps as a host float array (they travel in the kernel parameters / constant bank).
    `B200_VMSplit.get_kernel` computes the taps on the host and attaches them to the device tensor it
    returns (`_jt_host`); a foreign tensor costs one device->host copy."""
    if isinstance(kernel, (list, tuple)):
        vals = list(kernel)
    else:
        vals = getattr(kernel, "_jt_host", None)
        if vals is None:
            vals = kernel.detach().reshape(-1).float().cpu().tolist()
    return floats(vals), len(vals)


def blur_cl(x_phys, h, w, c, taps, axes, adjoint):
    """x_phys: contiguous fp32 buffer holding h*w*c floats, interpreted as [h][w][c]; taps = host_taps(...)."""
    out = torch.empty_like(x_phys)
    tmp = torch.empty_like(x_phys) if axes == 3 else None
    h_taps, ntaps = taps
    with TIMER.span("blur_adj" if adjoint else "blur_fwd"):
        check(_lib.lib().jt_blur_cl(_p(x_phys), _p(out), _p(tmp), h, w, c, h_taps, ntaps, axes,
                                    int(adjoint), _stream()), "jt_blur_cl")
    return out


def blur_multi(arrays, metas, tapsets, adjoint):
    """arrays: contiguous fp32 buffers; metas[i] = (h, w, c, axes, tapset); tapsets: list of host tap lists of
    equal length (<= 2). One C-ABI call, two launches (csrc/blur.cu). Returns the blurred buffers."""
    outs = [torch.empty_like(a) for a in arrays]
    tmps = [torch.empty_like(a) if m[3] == 3 else None for a, m in zip(arrays, metas)]
    ntaps = len(tapsets[0])
    assert all(len(t) == ntaps for t in tapsets)
    flat = floats([v for t in tapsets for v in t])
    dims = ints([v for m in metas for v in m[:4]])
    sets = ints([m[4] for m in metas])
    with TIMER.span("blur_adj" if adjoint else "blur_fwd"):
        check(_lib.lib().jt_blur_multi(len(arrays), ptrs([a.data_ptr() for a in arrays]),
                                       ptrs([o.data_ptr() for o in outs]), ptrs([_p(t) for t in tmps]), dims, sets,
                                       flat, len(tapsets), ntaps, int(adjoint), _stream()), "jt_blur_multi")
    return outs


class BlurGroup(torch.autograd.Function):
    """All blurred factors of a step as ONE autograd node: forward = two launches (W passes, then H passes) over
    up to 12 arrays, backward = two launches of the adjoint. `metas[i] = (hq, wq, axes, tapset)` per factor
    (see BlurFactor for the (hq, wq) re-interpretation); `tapsets` = host tap lists (density, colour)."""

    @staticmethod
    def forward(ctx, metas, tapsets, *factors):
        xs, full = [], []
        for x, (hq, wq, axes, ts) in zip(factors, metas):
            _need_cuda(x, "factor")
            xp = phys_cl(x)
            c = xp.shape[2]
            assert xp.shape[0] * xp.shape[1] == hq * wq
            xs.append(xp)
            full.append((hq, wq, c, axes, ts))
        ys = blur_multi(xs, full, tapsets, 0)
        ctx.meta = (full, tapsets, [tuple(xp.shape) for xp in xs])
        outs = tuple(y.view(1, m[0], m[1], m[2]).permute(0, 3, 1, 2) for y, m in zip(ys, full))
        # a blurred copy of a frozen factor is frozen too, so that the render op sees which factors need a gradient
        ctx.mark_non_differentiable(*[y for i, y in enumerate(outs) if not ctx.needs_input_grad[2 + i]])
        return outs

    @staticmethod
    def backward(ctx, *gys):
        full, tapsets, shapes = ctx.meta
        idx = [i for i, g in enumerate(gys) if g is not None and ctx.needs_input_grad[2 + i]]
        gxs = blur_multi([phys_cl(gys[i]) for i in idx], [full[i] for i in idx], tapsets, 1) if idx else []
        out = [None] * len(gys)
        for i, gx in zip(idx, gxs):
            out[i] = gx.view(1, *shapes[i]).permute(0, 3, 1, 2)
        return (None, None, *out)


class BlurFactor(torch.autograd.Function):
    """Separable blur of one VM factor ([1,C,H,W] logical shape, channel-last memory).

    `hq, wq` are the (H', W') the reference passes to convolute_plane
    (bateRF.py:68,76,117): (g[m0], g[m1]) although storage is [g[m1], g[m0]] -- a
    re-interpretation of the buffer on non-cubic grids (SURVEY.md Appendix B-3).
    In channel-last memory the re-interpretation is the same statement: treat the
    [H][W][C] buffer as [H'][W'][C]. Output logical shape: [1,C,H',W']."""

    @staticmethod
    def forward(ctx, x, taps, hq, wq, axes):
        _need_cuda(x, "factor")
        xp = phys_cl(x)
        c = xp.shape[2]
        assert xp.shape[0] * xp.shape[1] == hq * wq
        ht = host_taps(taps)
        y = blur_cl(xp, hq, wq, c, ht, axes, 0)
        ctx.meta = (tuple(xp.shape), hq, wq, c, axes, ht)
        return y.view(1, hq, wq, c).permute(0, 3, 1, 2)

    @staticmethod
    def backward(ctx, gy):
        shape, hq, wq, c, axes, ht = ctx.meta
        gp = phys_cl(gy)
        gx = blur_cl(gp, hq, wq, c, ht, axes, 1)
        return gx.view(1, *shape).permute(0, 3, 1, 2), None, None, None, None


# ------------------------------------------------------------------ standalone feature ops (API parity)
def _samp_from_xyz(xyz_norm):
    n = xyz_norm.shape[0]
    samp = torch.zeros((max(n, 1), 4), device=xyz_norm.device)
    samp[:n, :3] = xyz_norm.detach()
    return samp


class DensityFeature(torch.autograd.Function):
    """compute_densityfeature(xyz_norm) as a differentiable op (bateRF.py:41-94)."""

    @staticmethod
    def forward(ctx, xyz, *factors):
        _need_cuda(xyz, "xyz_sampled")
        fs = FactorSet(factors[:3], factors[3:])
        n = xyz.shape[0]
        samp = _samp_from_xyz(xyz)
        out = torch.empty((max(n, 1),), device=xyz.device)
        vm_gather_fwd(0, fs, samp, None, None, n, out)
        ctx.fs, ctx.samp, ctx.n = fs, samp, n
        return out[:n]

    @staticmethod
    def backward(ctx, g):
        fs, samp, n = ctx.fs, ctx.samp, ctx.n
        gp, gl = fs.zero_grads()
        dsamp = torch.zeros_like(samp)
        vm_gather_bwd(0, fs, gp, gl, samp, None, None, n, g.contiguous().float(), dsamp, 0)
        gpn, gln = FactorSet.grads_as_nchw(gp, gl)
        return (dsamp[:n, :3], *gpn, *gln)


class AppComponents(torch.autograd.Function):
    """plane*line products [A, sum C_app] feeding basis_mat (bateRF.py:97-128)."""

    @staticmethod
    def forward(ctx, xyz, *factors):
        _need_cuda(xyz, "xyz_sampled")
        fs = FactorSet(factors[:3], factors[3:])
        n = xyz.shape[0]
        samp = _samp_from_xyz(xyz)
        out = torch.empty((max(n, 1), fs.ctot), device=xyz.device)
        vm_gather_fwd(1, fs, samp, None, None, n, out)
        ctx.fs, ctx.samp, ctx.n = fs, samp, n
        return out[:n]

    @staticmethod
    def backward(ctx, g):
        fs, samp, n = ctx.fs, ctx.samp, ctx.n
        gp, gl = fs.zero_grads()
        dsamp = torch.zeros_like(samp)
        vm_gather_bwd(1, fs, gp, gl, samp, None, None, n, g.contiguous().float(), dsamp, 0)
        gpn, gln = FactorSet.grads_as_nchw(gp, gl)
        return (dsamp[:n, :3], *gpn, *gln)


class Linear(torch.autograd.Function):
    """y = x W^T (+ b) through jt_gemm_nt / jt_gemm_tn (used by compute_appfeature's basis_mat)."""

    @staticmethod
    def forward(ctx, x, w, b):
        m, k = x.shape
        n = w.shape[0]
        ldx, ldy = (k + 3) & ~3, (n + 3) & ~3
        xp = x if (ldx == k and x.is_contiguous()) else torch.nn.functional.pad(x, (0, ldx - k)).contiguous()
        y = torch.empty((max(m, 1), ldy), device=x.device)
        wc = w.contiguous()
        gemm_nt(xp, ldx, wc, k, 0, b, y, ldy, None, 0, None, m, n, k, 0, name="basis_fwd")
        ctx.save_for_backward(xp, wc)
        ctx.meta = (m, n, k, ldx, ldy, b is not None)
        return y[:m, :n]

    @staticmethod
    def backward(ctx, gy):
        xp, wc = ctx.saved_tensors
        m, n, k, ldx, ldy, has_b = ctx.meta
        g = torch.zeros((max(m, 1), ldy), device=gy.device)
        g[:m, :n] = gy
        gx = torch.empty((max(m, 1), ldx), device=gy.device)
        gemm_nt(g, ldy, wc, k, 1, None, gx, ldx, None, 0, None, m, k, n, 0, name="basis_bwd_x")
        gw = torch.zeros_like(wc)
        gb = torch.zeros((n,), device=gy.device) if has_b else None
        gemm_tn(g, ldy, xp, ldx, None, m, n, k, gw, k, gb, name="basis_bwd_w")
        return gx[:m, :k], gw, gb


# ------------------------------------------------------------------ field maintenance (section 8f-3)
def field_alpha(fs, geom, shift, act, length, xyz=None, lin=None, grid=None, mask=None):
    """alpha at explicit points (xyz [n,3]) or on the dense grid (lin = 3 device linspace tables, grid = (gx,gy,gz);
    result [gz,gy,gx]). fs: FactorSet of the density factors."""
    mb, md, mg = (mask.bits, mask.h_dims, mask.h_geom) if mask is not None else (None, None, None)
    if xyz is not None:
        _need_cuda(xyz, "xyz")
        xyz = xyz.reshape(-1, 3).contiguous().float()
        n = xyz.shape[0]
        out = torch.empty((n,), device=xyz.device)
        lx = ly = lz = None
        g3 = None
    else:
        lx, ly, lz = lin
        _need_cuda(lx, "linspace table")
        n = 0
        out = torch.empty((grid[2], grid[1], grid[0]), device=lx.device)
        g3 = ints(grid)
    with TIMER.span("field_alpha"):
        check(_lib.lib().jt_field_alpha(fs.ptrs, fs.dims, geom, _p(xyz), n, _p(lx), _p(ly), _p(lz), g3, _p(mb), md, mg,
                                        float(shift), int(act), float(length), _p(out), _stream()), "jt_field_alpha")
    return out


def field_density_grad(fs, geom, shift, act, xyz=None, samp=None, slot=None, n_dev=None, n_max=None, mask=None,
                       normals=False, want_sigma=True):
    """sigma = feature2density(sigma_feature(p)) and grad = d sigma / d p (jt_field_density_grad, no autograd): at world
    points xyz [n,3] (tested against the occupancy mask) -> (sigma [n], grad [n,3]), or at compacted samples samp
    [cap,4] (normalised coordinates; element e reads samp[slot[e]] when slot is given; count n_dev on the device, at
    most n_max; no mask). normals=True: the second
    output holds the unit outward normals -grad/|grad| (0 where grad is 0 or not finite). want_sigma=False: sigma is
    not written and None is returned in its place. fs: FactorSet of the fp32 density factors."""
    mb, md, mg = (mask.bits, mask.h_dims, mask.h_geom) if mask is not None else (None, None, None)
    if xyz is not None:
        _need_cuda(xyz, "xyz")
        xyz = xyz.reshape(-1, 3).contiguous().float()
        n = xyz.shape[0]
        dev = xyz.device
        if n == 0:
            return (torch.empty((0,), device=dev) if want_sigma else None), torch.empty((0, 3), device=dev)
    else:
        _need_cuda(samp, "samp")
        n, dev = int(n_max), samp.device
    sigma = torch.empty((n,), device=dev) if want_sigma else None
    grad = torch.empty((n, 3), device=dev)
    with TIMER.span("field_density_grad"):
        check(_lib.lib().jt_field_density_grad(fs.ptrs, fs.dims, geom, _p(xyz), _p(samp), _p(slot), _p(n_dev), n,
                                               _p(mb), md, mg, float(shift), int(act), int(bool(normals)),
                                               _p(sigma), _p(grad), _stream()), "jt_field_density_grad")
    return sigma, grad


def raycast(fs, geom, shift, act, length, level, rays_o, rays_d, n_samples, ztab=None, mask=None, rounds=False,
            counter=True):
    """First hit of rays_o / rays_d [n,3] on {compute_alpha(p, length) >= level} (jt_raycast, no autograd), on the
    no-grad forward's sample depths (metric rays, or the NDC depth table ztab [n_samples]) refined to the first
    crossing -> (t [n] (+inf: miss), xyz [n,3] (0: miss), k [n] int32 hit sample (-1: miss)), plus the refinement
    rounds per ray [n] int32 with rounds=True. counter=False hands rays to warps by a static grid stride instead of an
    atomic counter (the same results; for timing the two schedules). fs: FactorSet of the fp32 density factors."""
    if not 0.0 < float(level) < 1.0:
        raise _lib.JtError(f"raycast: level {level} must lie in (0, 1)")
    _need_cuda(rays_o, "rays_o")
    _need_cuda(rays_d, "rays_d")
    rays_o = rays_o.reshape(-1, 3).contiguous().float()
    rays_d = rays_d.reshape(-1, 3).contiguous().float()
    n, dev = rays_o.shape[0], rays_o.device
    t = torch.empty((n,), device=dev)
    xyz = torch.empty((n, 3), device=dev)
    k = torch.empty((n,), device=dev, dtype=torch.int32)
    rnd = torch.empty((n,), device=dev, dtype=torch.int32) if rounds else None
    if n > 0:
        mb, md, mg = (mask.bits, mask.h_dims, mask.h_geom) if mask is not None else (None, None, None)
        work = torch.zeros((1,), device=dev, dtype=torch.int32) if counter else None
        with TIMER.span("raycast"):
            check(_lib.lib().jt_raycast(fs.ptrs, fs.dims, geom, _p(mb), md, mg, float(shift), int(act), float(length),
                                        float(level), _p(rays_o), _p(rays_d), n, _p(ztab), int(n_samples), _p(work),
                                        _p(t), _p(xyz), _p(k), _p(rnd), _stream()), "jt_raycast")
    return (t, xyz, k, rnd) if rounds else (t, xyz, k)


def alpha_mask_build(alpha_zyx, thres):
    """alpha [D,H,W] -> (vol [D,H,W] float {0,1}, bits int32 words, stats int32[7])."""
    _need_cuda(alpha_zyx, "alpha")
    assert alpha_zyx.is_contiguous() and alpha_zyx.dtype == torch.float32
    d, h, w = alpha_zyx.shape
    dev = alpha_zyx.device
    tmp = torch.empty_like(alpha_zyx)
    vol = torch.empty_like(alpha_zyx)
    bits = torch.empty(((d * h * w + 31) // 32,), device=dev, dtype=torch.int32)
    stats = torch.empty((7,), device=dev, dtype=torch.int32)
    with TIMER.span("alpha_mask_build"):
        check(_lib.lib().jt_alpha_mask_build(_p(alpha_zyx), w, h, d, float(thres), _p(tmp), _p(vol), _p(bits),
                                             _p(stats), _stream()), "jt_alpha_mask_build")
    return vol, bits, stats


def marching_cubes(vol_zyx, level, lin, aabb, normals=False):
    """Marching cubes on a dense volume: vol_zyx [gz,gy,gx] fp32 (contiguous, CUDA), inside where value > level.
    lin = the three device tables [x, y, z] with s = torch.linspace(0, 1, g); aabb [2,3] (host values). Lattice
    point (i, j, k) is aabb[0]*(1-s) + aabb[1]*s, the dense_xyz of getDenseAlpha.
    Returns (verts [V,3] fp32, faces [F,3] int32) on the volume's device; [0,3] tensors when nothing crosses.
    One vertex per lattice edge whose ends straddle the level, interpolated linearly along the edge, so the
    vertices are those of any marching cubes; the triangulation inside a cell comes from the project's generated
    case table (csrc/gen_mc_tables.py) and may differ from PyMCubes or skimage. The mesh is closed where the
    surface does not reach the volume's border, and normals point toward decreasing value. Order: vertices by the
    linear index of the edge's lower end, then axis x < y < z; faces by cell, then table order. One 16-byte host
    read of the counts sizes the outputs.
    normals=True also returns normals [V,3] fp32 (jt_mc_normals): per vertex -normalize((1-t) g(p0) + t g(p1)), g the
    volume's central-difference gradient in world units at the two ends of the vertex's edge (one-sided at the
    border), t the vertex's position on the edge; (0,0,0) where that vector is zero. They point toward decreasing
    value, as the faces do."""
    if not isinstance(vol_zyx, torch.Tensor):
        raise _lib.JtError("marching_cubes: the volume must be a tensor")
    _need_cuda(vol_zyx, "volume")
    if vol_zyx.dtype != torch.float32 or vol_zyx.dim() != 3 or not vol_zyx.is_contiguous():
        raise _lib.JtError(f"marching_cubes: the volume must be a contiguous fp32 [gz,gy,gx] tensor, got "
                           f"{vol_zyx.dtype} {tuple(vol_zyx.shape)}")
    gz, gy, gx = vol_zyx.shape
    if min(gx, gy, gz) < 2:
        raise _lib.JtError(f"marching_cubes: every dimension must be >= 2, got {tuple(vol_zyx.shape)}")
    lv = ctypes.c_float(float(level)).value
    if not math.isfinite(lv):
        raise _lib.JtError(f"marching_cubes: level {level!r} is not a finite fp32 value")
    for t, g, name in zip(lin, (gx, gy, gz), "xyz"):
        if t.device != vol_zyx.device or t.dtype != torch.float32 or t.shape != (g,) or not t.is_contiguous():
            raise _lib.JtError(f"marching_cubes: lin_{name} must be a contiguous fp32 [{g}] tensor on the volume's device")
    h_aabb = torch.as_tensor(aabb, dtype=torch.float32).reshape(6).tolist()
    nbytes = int(_lib.lib().jt_mc_scratch_bytes(gx, gy, gz))
    if nbytes < 0:
        raise _lib.JtError(f"marching_cubes: grid {gx}x{gy}x{gz} has 2^31 or more points")
    dev = vol_zyx.device
    scratch = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    totals = torch.empty((2,), dtype=torch.int64, device=dev)
    with TIMER.span("mc_count"):
        check(_lib.lib().jt_mc_count(_p(vol_zyx), gx, gy, gz, lv, _p(scratch), _p(totals), _stream()), "jt_mc_count")
    nv, nf = totals.tolist()
    if max(nv, nf) > 2 ** 31 - 1:
        raise _lib.JtError(f"marching_cubes: {nv} vertices / {nf} triangles do not fit int32 indices")
    verts = torch.empty((nv, 3), dtype=torch.float32, device=dev)
    faces = torch.empty((nf, 3), dtype=torch.int32, device=dev)
    if nv > 0 or nf > 0:
        with TIMER.span("mc_emit"):
            check(_lib.lib().jt_mc_emit(_p(vol_zyx), gx, gy, gz, lv, _p(lin[0]), _p(lin[1]), _p(lin[2]),
                                        floats(h_aabb), _p(scratch), _p(totals), _p(verts), _p(faces), _stream()),
                  "jt_mc_emit")
    if not normals:
        return verts, faces
    nrm = torch.empty((nv, 3), dtype=torch.float32, device=dev)
    if nv > 0:
        with TIMER.span("mc_normals"):
            check(_lib.lib().jt_mc_normals(_p(vol_zyx), gx, gy, gz, lv, _p(lin[0]), _p(lin[1]), _p(lin[2]),
                                           floats(h_aabb), _p(scratch), _p(totals), _p(nrm), _stream()),
                  "jt_mc_normals")
    return verts, faces, nrm


def resize_bilinear_cl(x, h2, w2):
    """[1,C,H,W] channel-last factor -> [1,C,h2,w2] channel-last (bilinear, align_corners=True)."""
    _need_cuda(x, "factor")
    xp = phys_cl(x)
    h, w, c = xp.shape
    out = torch.empty((h2, w2, c), device=x.device, dtype=torch.float32)
    with TIMER.span("resize_bilinear"):
        check(_lib.lib().jt_resize_bilinear_cl(_p(xp), h, w, c, _p(out), int(h2), int(w2), _stream()),
              "jt_resize_bilinear_cl")
    return out.unsqueeze(0).permute(0, 3, 1, 2)
