"""The fused render op: one autograd node for the whole L1 forward/backward.

Sequence of C-ABI calls for one batch of rays (all on the current stream, no
host synchronisation anywhere -- the reference syncs at every boolean-mask
index, SURVEY.md section 2b):

  forward   jt_march_compact -> jt_vm_gather_fwd(density) -> jt_alpha_fwd -> appearance + shading:
              tcgen05, SH shading        jt_app_basis_sh_fwd_tc          (gather + basis_mat + SHRender, one kernel)
              tcgen05, MLP_Fea head      jt_app_basis_fwd_tc -> jt_head_mlp_fwd_tc
              strict fp32 (any head)     jt_vm_gather_fwd(app) -> jt_gemm_nt(basis) -> jt_pe_encode / jt_gemm_nt / jt_sh_shade
            -> jt_composite_fwd
  normals   jt_march_compact -> jt_vm_gather_fwd(density) -> jt_alpha_fwd -> jt_field_density_grad(samples)
            -> jt_normal_composite   (render_normals: no grad, no appearance stage)
  backward  jt_render_bwd -> jt_ray_init -> head backward (jt_sh_bwd_tc | jt_head_bwd_tc | fp32 GEMM chain)
            -> jt_vm_scatter_rays(app) -> jt_vm_scatter_rays(density)
            (pose-path gradients accumulate inside the scatters; with a gradient synchroniser attached the
            appearance part of the flat gradient bucket is all-reduced while the density scatter runs)

The backward computes only the gradients autograd asks for (ctx.needs_input_grad). With a frozen scene (test-time
pose optimisation: freeze_scene()) it runs the head backward without weight gradients and both scatters
coordinate-only, and allocates no factor-gradient bucket.

Sample counts (V valid samples, A appearance samples) stay on the device; the
kernels read them from `ray_off[N]` / `app_off[N]` and run persistent grids.
"""
import copy

import torch

from . import _lib, ops, parallel
from ._lib import check
from .ops import FactorSet, TIMER, _p, _stream


def _r4(n):
    return (n + 3) & ~3


class RenderCfg:
    """Host-side description of one forward call (plain Python, no tensors)."""

    def __init__(self, **kw):
        self.n_samples = 0
        self.ndc = False
        self.white_bg = True
        self.h_geom = None          # ctypes float[12]
        self.h_inv = None           # ctypes float[3]
        self.mask = None            # PackedMask or None
        self.density_shift = -10.0
        self.act = 0                # 0 softplus, 1 relu
        self.distance_scale = 25.0
        self.thres = 1e-4
        self.depth_bias = 0.0       # -near + 0.05
        self.shading = "MLP_Fea"
        self.app_dim = 27
        self.fea_pe = 2
        self.view_pe = 2
        self.hidden = 64
        self.fea_prog = 1.0
        self.view_prog = 1.0
        self.head = "fp32"          # "fp32": SIMT GEMMs (strict parity) | "tc": tcgen05 fused head
        self.tc_fwd_split = 2       # 2: hi+lo bf16 operands (fp32-class forward), 1: plain bf16
        self.grad_enabled = True    # torch.is_grad_enabled() at the call site (B200_VMSplit.forward sets it)
        self.tc_infer_fp16 = True   # no-grad forward of the MLP_Fea head: single-term fp16 operands (rgb within ~2e-5)
        self.storage = "fp32"       # "bf16": the kernels gather from a bf16 copy of the factors (fp32 masters / gradients)
        self.store_cache = (None, None)
        self.bf16_backward_taps = False
        self.app_cap = None         # capacity of the appearance-stage buffers for training calls (None: N*S)
        self.app_monitor = None     # callable(a_total_dev, app_used_dev, n_rays): B200_VMSplit's capacity tracker
        self.infer_exact_alloc = True   # no-grad calls read A on the host and allocate exactly
        self.__dict__.update(kw)


class _HeadImpl:
    """One implementation of the shading head on the compacted appearance samples. `forward` returns rgb [cap,4] and
    keeps, as attributes, what its `backward` needs; `backward` writes dcomps [cap, sum C_app] (dtype `dcomps_dtype`)
    for the appearance scatter and the basis_mat / head weight gradients into `g_basis` / `head_grads` (None: not
    wanted)."""
    dcomps_dtype = torch.float32

    def __init__(self, cfg, afs, comp, aidx, rays_d, basis_w, params, a_count, cap):
        self.cfg, self.afs, self.comp, self.aidx, self.rays_d = cfg, afs, comp, aidx, rays_d
        self.basis_w, self.params, self.a_count, self.cap = basis_w, params, a_count, cap
        self.dev = rays_d.device
        self.shade_act = 2 if cfg.shading == "SH" else 1      # output activation jt_render_bwd differentiates

    @classmethod
    def supports(cls, shading, app_dim, hidden, fea_pe, view_pe, comps):
        """The tensor-core heads are specialised for the shipped configurations (class attributes)."""
        return (shading == cls.shading and app_dim == cls.app_dim and all(int(c) == cls.comps for c in comps) and
                (cls.mlp is None or (hidden, fea_pe, view_pe) == cls.mlp))

    def _wgrads(self, g_basis, head_grads):
        """The tensor-core MLP heads write all seven weight gradients or none: a frozen group gets dropped scratch."""
        if g_basis is None and head_grads is None:
            return None
        return (g_basis if g_basis is not None else torch.zeros_like(self.basis_w),
                *(head_grads if head_grads is not None else [torch.zeros_like(t) for t in self.params]))


class _Fp32Head(_HeadImpl):
    """Strict fp32 SIMT chain, any head: appearance gather -> basis_mat GEMM -> SH shading or PE + MLP GEMMs."""
    consumed = False

    def forward(self, train, basis_grad):
        cfg, afs, comp, aidx, a_count, cap = self.cfg, self.afs, self.comp, self.aidx, self.a_count, self.cap
        F, H, ldf, dev = cfg.app_dim, cfg.hidden, _r4(cfg.app_dim), self.dev
        self.comps = torch.empty((cap, afs.ctot), device=dev)
        ops.vm_gather_fwd(1, afs, comp.samp, aidx, a_count, cap, self.comps)
        self.feat = feat = torch.empty((cap, ldf), device=dev)
        ops.gemm_nt(self.comps, afs.ctot, self.basis_w, afs.ctot, 0, None, feat, ldf, None, 0, a_count, cap, F,
                    afs.ctot, 0, name="basis_fwd")
        rgb = torch.empty((cap, 4), device=dev)
        if cfg.shading == "SH":
            ops.sh_shade(0, feat, ldf, aidx, comp.sidx, self.rays_d, cfg.n_samples, cfg.ndc, a_count, cap, rgb, None,
                         None, 0)
            return rgb
        w1, b1, w2, b2, w3, b3 = self.params
        if cfg.shading == "MLP_Fea":
            self.in_dim = in_dim = F + 3 + 2 * cfg.fea_pe * F + 6 * cfg.view_pe
            self.ldi = ldi = _r4(in_dim)
            self.x = x = torch.empty((cap, ldi), device=dev)
            ops.pe_encode(0, F, cfg.fea_pe, cfg.view_pe, 0, cfg.fea_prog, cfg.view_prog, cfg.n_samples, cfg.ndc,
                          feat, ldf, aidx, comp.sidx, self.rays_d, a_count, cap, x, ldi)
            self.h1 = h1 = torch.empty((cap, H), device=dev)
            ops.gemm_nt(x, ldi, w1, in_dim, 0, b1, h1, H, None, 0, a_count, cap, H, in_dim, 1, name="mlp_l1_fwd")
            self.h2 = h2 = torch.empty((cap, H), device=dev)
            ops.gemm_nt(h1, H, w2, H, 0, b2, h2, H, None, 0, a_count, cap, H, H, 1, name="mlp_l2_fwd")
            ops.gemm_nt(h2, H, w3, H, 0, b3, rgb, 4, None, 0, a_count, cap, 3, H, 2, name="mlp_l3_fwd")
        elif cfg.shading == "MLP_Fea_WeakView":
            self.in_dim = in_dim = F + 2 * cfg.fea_pe * F
            self.ldi = ldi = _r4(in_dim)
            self.nv = nv = 6 * cfg.view_pe
            assert nv % 4 == 0, "view_pe must be even for the WeakView layout"
            self.ldm = ldm = nv + H
            self.x = x = torch.empty((cap, ldi), device=dev)
            self.mid = mid = torch.empty((cap, ldm), device=dev)
            ops.pe_encode(0, F, cfg.fea_pe, cfg.view_pe, 1, cfg.fea_prog, cfg.view_prog, cfg.n_samples, cfg.ndc,
                          feat, ldf, aidx, comp.sidx, self.rays_d, a_count, cap, x, ldi, mid, ldm)
            self.h1 = h1 = torch.empty((cap, H), device=dev)
            ops.gemm_nt(x, ldi, w1, in_dim, 0, b1, h1, H, None, 0, a_count, cap, H, in_dim, 1, name="mlp_l1_fwd")
            ops.gemm_nt(h1, H, w2, H, 0, b2, mid, ldm, None, 0, a_count, cap, H, H, 1, name="mlp_l2_fwd", y_off=nv)
            ops.gemm_nt(mid, ldm, w3, ldm, 0, b3, rgb, 4, None, 0, a_count, cap, 3, ldm, 2, name="mlp_l3_fwd")
        else:
            raise _lib.JtError(f"shading model {cfg.shading!r} is not implemented by the B200 path")
        return rgb

    def backward(self, dout, dcomps, g_basis, head_grads):
        if self.consumed:
            raise _lib.JtError("second backward through the same render call: the strict-fp32 MLP head reuses its "
                               "encoded-input buffer for the input gradient (2.6 GB at 4096 x 1000 samples); call "
                               "forward again, or use head_precision='tc' / SH shading, whose backward is re-entrant")
        cfg, afs, feat, a_count, cap, dev = self.cfg, self.afs, self.feat, self.a_count, self.cap, self.dev
        F, H, ldf = cfg.app_dim, cfg.hidden, _r4(cfg.app_dim)
        dfeat = torch.empty((cap, ldf), device=dev)
        if cfg.shading == "SH":
            ops.sh_shade(1, feat, ldf, self.aidx, self.comp.sidx, self.rays_d, cfg.n_samples, cfg.ndc, a_count, cap,
                         None, dout, dfeat, ldf)
        else:
            self.consumed = True
            w1, b1, w2, b2, w3, b3 = self.params
            # the bucket views are zero-filled: the weight-gradient GEMMs write into them directly
            gw1, gb1, gw2, gb2, gw3, gb3 = head_grads if head_grads is not None else [None] * 6
            x, ldi, in_dim, h1 = self.x, self.ldi, self.in_dim, self.h1
            dh2 = torch.empty((cap, H), device=dev)
            dh1 = torch.empty((cap, H), device=dev)
            # layer 3 reads h2 (MLP_Fea) or [view PE | h2] (WeakView, whose dh2 skips the view columns)
            l3, ld3, off = (self.h2, H, 0) if cfg.shading == "MLP_Fea" else (self.mid, self.ldm, self.nv)
            if gw3 is not None:
                ops.gemm_tn(dout, 4, l3, ld3, a_count, cap, 3, ld3, gw3, ld3, gb3, name="mlp_l3_bwd_w")
            ops.gemm_nt(dout, 4, w3, ld3, 1, None, dh2, H, l3, ld3, a_count, cap, H, 3, 0, name="mlp_l3_bwd_x",
                        w_off=off, mask_off=off)
            if gw2 is not None:
                ops.gemm_tn(dh2, H, h1, H, a_count, cap, H, H, gw2, H, gb2, name="mlp_l2_bwd_w")
            ops.gemm_nt(dh2, H, w2, H, 1, None, dh1, H, h1, H, a_count, cap, H, H, 0, name="mlp_l2_bwd_x")
            if gw1 is not None:
                ops.gemm_tn(dh1, H, x, ldi, a_count, cap, H, in_dim, gw1, in_dim, gb1, name="mlp_l1_bwd_w")
            # the encoded input is dead after dW1: reuse its buffer for its own gradient
            ops.gemm_nt(dh1, H, w1, in_dim, 1, None, x, ldi, None, 0, a_count, cap, in_dim, H, 0, name="mlp_l1_bwd_x")
            ops.pe_encode(1, F, cfg.fea_pe, cfg.view_pe, int(cfg.shading != "MLP_Fea"), cfg.fea_prog, cfg.view_prog,
                          cfg.n_samples, cfg.ndc, feat, ldf, None, None, None, a_count, cap, dfeat, ldf, None, 0, x, ldi)
        if g_basis is not None:
            ops.gemm_tn(dfeat, ldf, self.comps, afs.ctot, a_count, cap, F, afs.ctot, g_basis, afs.ctot, None,
                        name="basis_bwd_w")
        ops.gemm_nt(dfeat, ldf, self.basis_w, afs.ctot, 1, None, dcomps, afs.ctot, None, 0, a_count, cap, afs.ctot, F,
                    0, name="basis_bwd_x")


class _ShTcHead(_HeadImpl):
    """tcgen05 SH head: appearance gather + basis_mat + SHRender in one kernel; bf16 dcomps (bf16 GEMM operands)."""
    shading, app_dim, comps, mlp = "SH", 27, 48, None           # Blender: 3 x 48 components, app_dim 27
    dcomps_dtype = torch.bfloat16

    def forward(self, train, basis_grad):
        cfg, cap = self.cfg, self.cap
        rgb = torch.empty((cap, 4), device=self.dev)
        self.feat = torch.empty((cap, 32), device=self.dev)       # feat 0..26 | 0 | view dir 28..30 | 0
        # the staged component tile only feeds the basis_mat weight gradient
        self.stage = ops.head_tc_stage(cap, self.dev) if train and basis_grad else None
        ops.app_basis_sh_fwd_tc(cfg.tc_fwd_split, self.afs, self.comp.samp, self.aidx, self.comp.sidx, self.rays_d,
                                cfg.n_samples, cfg.ndc, self.basis_w, self.a_count, cap, self.feat, rgb, self.stage)
        return rgb

    def backward(self, dout, dcomps, g_basis, head_grads):
        # no staged component tile when basis_mat was frozen in the forward: no weight gradient either
        ops.sh_bwd_tc(dout, self.feat, self.basis_w, self.a_count, self.cap, dcomps, self.stage,
                      g_basis if self.stage is not None else None)


class _MlpTcHead(_HeadImpl):
    """tcgen05 MLP_Fea head: appearance gather + basis_mat, then the MLP; bf16 dcomps."""
    shading, app_dim, comps, mlp = "MLP_Fea", 27, 48, (64, 2, 2)    # mlp: (hidden, fea_pe, view_pe)
    dcomps_dtype = torch.bfloat16

    def forward(self, train, basis_grad):
        cfg, cap = self.cfg, self.cap
        rgb = torch.empty((cap, 4), device=self.dev)
        self.feat = torch.empty((cap, 32), device=self.dev)       # feat 0..26 | 0 | view dir 28..30 | 0
        # the data backward reads the staged relu tiles as well as the component tile
        self.stage = ops.head_tc_stage(cap, self.dev) if train else None
        ops.app_basis_fwd_tc(cfg.tc_fwd_split, self.afs, self.comp.samp, self.aidx, self.comp.sidx, self.rays_d,
                             cfg.n_samples, cfg.ndc, self.basis_w, self.a_count, cap, self.feat, self.stage)
        # inference: fp16 operand tiles (one MMA per product, half the shared memory, two CTAs per SM); the
        # training forward keeps the hi+lo bf16 split because its staged tiles feed the bf16 backward GEMMs
        split = 3 if (not train and cfg.tc_infer_fp16 and cfg.tc_fwd_split == 2) else cfg.tc_fwd_split
        ops.head_mlp_fwd_tc(split, self.feat, *self.params, self.a_count, cap, cfg.fea_prog, cfg.view_prog, rgb,
                            self.stage)
        return rgb

    def backward(self, dout, dcomps, g_basis, head_grads):
        w1, b1, w2, b2, w3, b3 = self.params
        ops.head_bwd_tc(dout, self.feat, self.basis_w, w1, w2, w3, self.a_count, self.cap, self.cfg.fea_prog, dcomps,
                        self.stage, self._wgrads(g_basis, head_grads))


class _WeakViewTcHead(_HeadImpl):
    """tcgen05 MLP_Fea_WeakView head (csrc/weakview_tc.cu): fp32 appearance gather, then basis_mat + PE + MLP."""
    shading, app_dim, comps, mlp = "MLP_Fea_WeakView", 20, 20, (32, 2, 2)    # LLFF: 3 x 20 components

    def forward(self, train, basis_grad):
        cfg, cap = self.cfg, self.cap
        comps = torch.empty((cap, self.afs.ctot), device=self.dev)   # the staged bf16 tile replaces it in the backward
        ops.vm_gather_fwd(1, self.afs, self.comp.samp, self.aidx, self.a_count, cap, comps)
        self.feat = torch.empty((cap, 32), device=self.dev)       # feat 0..19 | 0 | view dir 28..30 | 0
        rgb = torch.empty((cap, 4), device=self.dev)
        self.stage = ops.wv_stage(cap, self.dev) if train else None
        ops.wv_head_fwd_tc(comps, self.aidx, self.comp.sidx, self.rays_d, cfg.n_samples, cfg.ndc, self.basis_w,
                           *self.params, self.a_count, cap, cfg.fea_prog, cfg.view_prog, self.feat, rgb, self.stage)
        return rgb

    def backward(self, dout, dcomps, g_basis, head_grads):
        w1, b1, w2, b2, w3, b3 = self.params
        ops.wv_head_bwd_tc(dout, self.feat, self.basis_w, w1, w2, w3, self.a_count, self.cap, self.cfg.fea_prog,
                           dcomps, self.stage, self._wgrads(g_basis, head_grads))


def tc_head(shading, app_dim, hidden, fea_pe, view_pe, comps):
    """The tensor-core head implementation covering this configuration, or None."""
    return next((h for h in (_ShTcHead, _MlpTcHead, _WeakViewTcHead)
                 if h.supports(shading, app_dim, hidden, fea_pe, view_pe, comps)), None)


def head_class(cfg, comps):
    """The head implementation a call with `cfg` runs on appearance components `comps`: the tensor-core head under
    cfg.head == "tc" (an error when none covers the configuration), else the strict fp32 chain."""
    if cfg.head != "tc":
        return _Fp32Head
    Head = tc_head(cfg.shading, cfg.app_dim, cfg.hidden, cfg.fea_pe, cfg.view_pe, comps)
    if Head is None:
        raise _lib.JtError("head='tc' needs 3 x 48 appearance components, app_dim 27 and MLP_Fea (hidden 64, "
                           "pe 2) or SH shading, or 3 x 20 components, app_dim 20 and MLP_Fea_WeakView (hidden "
                           "32, pe 2); use head='fp32'")
    return Head


def shade_points(cfg, afs, xyz_norm, viewdirs, basis_w, params):
    """Colour of the field at n points: rgb [n,3] of the head head_class(cfg, afs.C) runs, for normalised coordinates
    xyz_norm [n,3] (zero components outside [-1,1], as grid_sample's zero padding) and view directions viewdirs [n,3]
    taken as given (no normalisation). Each point is a one-sample ray whose sample is its own appearance sample, so
    the head's no-grad forward shades it exactly as it shades a render sample; rows are independent of each other.
    cfg supplies the head fields (shading, sizes, head, tc_fwd_split, tc_infer_fp16, PE progress)."""
    n = xyz_norm.shape[0]
    dev = xyz_norm.device
    Head = head_class(cfg, afs.C)
    cfg = copy.copy(cfg)
    cfg.n_samples, cfg.ndc = 1, False
    comp = ops.Compacted()
    comp.samp = ops._samp_from_xyz(xyz_norm)
    comp.sidx = torch.arange(max(n, 1), device=dev, dtype=torch.int32)
    count = torch.full((1,), n, device=dev, dtype=torch.int32)
    h = Head(cfg, afs, comp, comp.sidx, viewdirs.contiguous().float(), basis_w, params, count, max(n, 1))
    return h.forward(train=False, basis_grad=False)[:n, :3]


def render_normals(cfg, dfs, dfs32, rays_o, rays_d, aux):
    """Normal map of N rays (no grad): (normal_map [N,3], depth [N], opacity [N]). The samples, the density gather
    (on `dfs`, the factors forward gathers from) and jt_alpha_fwd run exactly as in VMRender.forward, so depth and
    opacity are the no-grad forward's bit for bit; jt_field_density_grad then gives every valid sample's unit outward
    normal from the fp32 factors `dfs32`, and jt_normal_composite sums weight x normal per ray over all valid samples.
    No appearance stage runs. cfg supplies n_samples, ndc, h_geom, mask, density_shift, act, distance_scale, thres and
    depth_bias."""
    lib = _lib.lib()
    dev = rays_o.device
    N, S = rays_o.shape[0], cfg.n_samples
    comp = ops.march_compact(rays_o, rays_d, aux, cfg.ndc, S, cfg.h_geom, cfg.mask)
    cap = comp.cap
    sigfeat = torch.empty((cap,), device=dev)
    ops.vm_gather_fwd(0, dfs, comp.samp, None, comp.count, cap, sigfeat)
    weight = torch.empty((cap,), device=dev)
    trans = torch.empty((cap,), device=dev)
    acc = torch.empty((N,), device=dev)
    wz = torch.empty((N,), device=dev)
    app_cnt = torch.empty((N,), device=dev, dtype=torch.int32)
    app_off = torch.zeros((N + 1,), device=dev, dtype=torch.int32)
    aidx = torch.empty((1,), device=dev, dtype=torch.int32)       # appearance list capped at one entry: not used here
    app_of = torch.empty((cap,), device=dev, dtype=torch.int32)
    with TIMER.span("alpha_fwd"):
        check(lib.jt_alpha_fwd(_p(comp.ray_off), N, _p(sigfeat), _p(comp.dist), _p(comp.samp),
                               float(cfg.density_shift), cfg.act, float(cfg.distance_scale), float(cfg.thres),
                               _p(weight), _p(trans), _p(acc), _p(wz), _p(app_cnt), _p(app_off), _p(aidx),
                               _p(app_of), 1, None, _stream()), "jt_alpha_fwd")
    _, nrm = ops.field_density_grad(dfs32, cfg.h_geom, cfg.density_shift, cfg.act, samp=comp.samp, n_dev=comp.count,
                                    n_max=cap, normals=True, want_sigma=False)
    normal_map = torch.empty((N, 3), device=dev)
    depth = torch.empty((N,), device=dev)
    opacity = torch.empty((N,), device=dev)
    with TIMER.span("normal_composite"):
        check(lib.jt_normal_composite(_p(comp.ray_off), N, _p(weight), _p(nrm), _p(acc), _p(wz), _p(rays_d),
                                      float(cfg.depth_bias), _p(normal_map), _p(depth), _p(opacity), _stream()),
              "jt_normal_composite")
    return normal_map, depth, opacity


# VMRender.apply's inputs as ctx.needs_input_grad indexes them: cfg, rays_o, rays_d, aux, then these groups
_RAYS, _DENS, _APP, _BASIS, _HEAD = slice(1, 3), slice(4, 10), slice(10, 16), slice(16, 17), slice(17, None)


def _full_backward(cfg):
    """An active gradient synchroniser (data parallel, outside `sync.paused()`) runs the full backward on every rank."""
    sync = getattr(cfg, "grad_sync", None)
    return sync is not None and sync._active()


class VMRender(torch.autograd.Function):
    """rgb_map, depth_map, opacity = render(rays, factors, basis, head).

    Inputs after cfg: rays_o [N,3], rays_d [N,3], aux (jitter [N] | NDC depth
    table [S] | None), 6 density factors (3 planes, 3 lines), 6 appearance
    factors, basis weight, then the head parameters (w1,b1,w2,b2,w3,b3) or none
    for SH. Factors are logical [1,C,H,W] / [1,C,L,1] tensors in channel-last
    memory (B200_VMSplit stores its parameters that way)."""

    @staticmethod
    def forward(ctx, cfg, rays_o, rays_d, aux, *tensors):
        ops._need_cuda(rays_o, "rays_o")
        lib = _lib.lib()
        dev = rays_o.device
        rays_o = rays_o.detach().contiguous().float()
        rays_d = rays_d.detach().contiguous().float()
        inputs = (cfg, rays_o, rays_d, aux) + tensors
        dens, app, basis_w, head = inputs[_DENS], inputs[_APP], inputs[_BASIS][0], inputs[_HEAD]
        head = [t.detach().contiguous() for t in head]
        basis_w = basis_w.detach().contiguous()
        dfs = FactorSet([t.detach() for t in dens[:3]], [t.detach() for t in dens[3:]])
        afs = FactorSet([t.detach() for t in app[:3]], [t.detach() for t in app[3:]])
        # bf16 factor storage: the forward gathers read the bf16 copy. The backward walks the fp32 factors unless
        # cfg.bf16_backward_taps: the coordinate (pose) gradient is a DIFFERENCE of neighbouring texels, and on a blurred
        # field bf16 rounding of two nearly equal neighbours costs more than the 2e-2 class allows (measured 2.7e-2 on
        # d/d rays_o); the staged taps are not what binds the scatter kernel either (same time with 8-byte taps).
        dfs32, afs32 = dfs, afs
        if cfg.storage == "bf16":
            dfs = dfs.with_bf16_store(cfg.store_cache[0])
            afs = afs.with_bf16_store(cfg.store_cache[1])
            if cfg.bf16_backward_taps:
                dfs32, afs32 = dfs, afs
        N, S = rays_o.shape[0], cfg.n_samples
        F = cfg.app_dim
        if basis_w.shape != (F, afs.ctot):
            raise _lib.JtError(f"basis_mat weight {tuple(basis_w.shape)} != ({F}, {afs.ctot})")
        Head = head_class(cfg, afs.C)

        comp = ops.march_compact(rays_o, rays_d, aux, cfg.ndc, S, cfg.h_geom, cfg.mask)
        cap = comp.cap
        sigfeat = torch.empty((cap,), device=dev)
        ops.vm_gather_fwd(0, dfs, comp.samp, None, comp.count, cap, sigfeat)

        weight = torch.empty((cap,), device=dev)
        trans = torch.empty((cap,), device=dev)
        acc = torch.empty((N,), device=dev)
        wz = torch.empty((N,), device=dev)
        app_cnt = torch.empty((N,), device=dev, dtype=torch.int32)
        app_off = torch.zeros((N + 1,), device=dev, dtype=torch.int32)
        aidx = torch.empty((cap,), device=dev, dtype=torch.int32)
        app_of = torch.empty((cap,), device=dev, dtype=torch.int32)
        # needs_input_grad mirrors requires_grad of the inputs even under torch.no_grad(), and grad mode is always
        # off inside Function.forward: the caller records it in cfg.grad_enabled. Without this test every
        # full-frame render ran the training forward (staging tiles written for a backward that never comes).
        train = cfg.grad_enabled and any(ctx.needs_input_grad)
        # Memory model of the appearance stage (INTEGRATION.md): the number of appearance samples A only exists on
        # the device. Training sizes the appearance-stage buffers (features, staged operand tiles, dcomps) to
        # `acap` = cfg.app_cap, a host-side bound kept by B200_VMSplit from the counts of earlier steps (read back
        # asynchronously; N*S when there is no history) -- jt_alpha_fwd clamps the list to it and raises a device flag
        # that the module checks at its next call. No-grad calls read A on the host (the reference synchronises at
        # the same place: boolean-mask indexing, batBase.py:128) and allocate exactly.
        acap = cap if (cfg.app_cap is None or not train) else max(1, min(cap, int(cfg.app_cap)))
        app_used = torch.zeros((2,), device=dev, dtype=torch.int32)
        with TIMER.span("alpha_fwd"):
            check(lib.jt_alpha_fwd(_p(comp.ray_off), N, _p(sigfeat), _p(comp.dist), _p(comp.samp),
                                   float(cfg.density_shift), cfg.act, float(cfg.distance_scale), float(cfg.thres),
                                   _p(weight), _p(trans), _p(acc), _p(wz), _p(app_cnt), _p(app_off), _p(aidx),
                                   _p(app_of), int(acap), _p(app_used), _stream()), "jt_alpha_fwd")
        a_count = app_used[0:1]                   # min(A, acap); the true A stays in app_off[N]
        if not train and cfg.infer_exact_alloc:
            acap = max(int(a_count.item()), 1)
        cap_v, cap = cap, acap                    # from here on `cap` sizes the APPEARANCE stage; cap_v = N*S

        h = Head(cfg, afs, comp, aidx, rays_d, basis_w, head, a_count, cap)
        rgb = h.forward(train, any(ctx.needs_input_grad[_BASIS]) or _full_backward(cfg))

        rgb_pre = torch.empty((N, 3), device=dev)
        rgb_map = torch.empty((N, 3), device=dev)
        depth = torch.empty((N,), device=dev)
        opacity = torch.empty((N,), device=dev)
        with TIMER.span("composite_fwd"):
            check(lib.jt_composite_fwd(_p(app_off), N, _p(aidx), _p(weight), _p(rgb), _p(acc), _p(wz), _p(rays_d),
                                       int(cfg.white_bg), float(cfg.depth_bias), _p(rgb_pre), _p(rgb_map),
                                       _p(depth), _p(opacity), int(cap), _stream()), "jt_composite_fwd")

        ctx.cfg, ctx.comp, ctx.dfs, ctx.afs, ctx.head = cfg, comp, dfs32, afs32, h
        ctx.bufs = dict(sigfeat=sigfeat, weight=weight, trans=trans, app_of=app_of, rgb=rgb, rgb_pre=rgb_pre)
        # version check only: the kernels read the parameters' storage directly, so an in-place update between
        # forward and backward (an optimizer step, load_state_dict) must raise as it does for the reference's ATen
        # nodes instead of silently differentiating the new values
        ctx.save_for_backward(*tensors)
        ctx.mark_non_differentiable(depth)
        VMRender.last_counts = (comp.count, app_off[N:N + 1])      # device scalars V, A (diagnostics / bench)
        VMRender.last_app_used = app_used                           # {min(A, capacity), overflow flag}
        if cfg.app_monitor is not None and train:
            cfg.app_monitor(app_off[N:N + 1], app_used, N)
        return rgb_map, depth, opacity

    @staticmethod
    def backward(ctx, g_rgb, g_depth, g_acc):
        lib = _lib.lib()
        cfg, comp, dfs, afs, h, b = ctx.cfg, ctx.comp, ctx.dfs, ctx.afs, ctx.head, ctx.bufs
        _ = ctx.saved_tensors                                 # raises if a parameter was modified in place since forward
        dev = g_rgb.device
        N, cap_v, cap = comp.n_rays, comp.cap, h.cap          # cap: appearance-stage capacity, cap_v = N*S
        g_rgb = g_rgb.contiguous().float()
        g_acc = g_acc.contiguous().float() if g_acc is not None else None

        dout = torch.empty((cap, 4), device=dev)
        dsig = torch.empty((cap_v,), device=dev)
        dnorm = torch.empty((N,), device=dev) if cfg.ndc else None
        with TIMER.span("render_bwd"):
            check(lib.jt_render_bwd(_p(comp.ray_off), N, _p(b["sigfeat"]), _p(comp.dist), _p(b["weight"]),
                                    _p(b["trans"]), _p(b["app_of"]), _p(b["rgb"]), _p(b["rgb_pre"]), _p(g_rgb),
                                    _p(g_acc), float(cfg.density_shift), cfg.act, float(cfg.distance_scale),
                                    int(cfg.white_bg), h.shade_act, _p(dout), _p(dsig), _p(dnorm), _stream()),
                  "jt_render_bwd")

        if VMRender.debug_capture is not None:            # diagnostics (scripts/debug_cfg4_grad.py): per-sample gradients
            VMRender.debug_capture.update(dsig=dsig.clone(), dout=dout.clone(), count=comp.count.clone(),
                                          weight=b["weight"].clone(), trans=b["trans"].clone(), rgb=b["rgb"].clone(),
                                          sigfeat=b["sigfeat"].clone(), a_count=h.a_count.clone())

        # Only the gradients autograd asks for. With an active gradient synchroniser every rank runs the full backward,
        # so that all ranks issue the same collectives whatever their parameters' requires_grad.
        sync = cfg.grad_sync if _full_backward(cfg) else None      # None: world size 1, or inside `sync.paused()`
        need = [sync is not None or any(ctx.needs_input_grad[s]) for s in (_RAYS, _DENS, _APP, _BASIS, _HEAD)]
        need_rays, need_dens, need_app, need_basis, need_head = need

        # One flat zero-filled bucket for every gradient this node produces (one memset; also the unit the
        # data-parallel all-reduce works on): [app planes, app lines | density planes, density lines | basis, head],
        # each group present only when it is needed. The appearance part comes first and is complete first, so a
        # gradient synchroniser (parallel.OverlappedGradSync) can reduce it across ranks while the density scatter
        # still runs.
        shapes = ([p.shape for p in afs.planes] + [l.shape for l in afs.lines] if need_app else []) + \
                 ([p.shape for p in dfs.planes] + [l.shape for l in dfs.lines] if need_dens else []) + \
                 ([h.basis_w.shape] if need_basis else []) + ([t.shape for t in h.params] if need_head else [])
        sizes = [int(torch.Size(s).numel()) for s in shapes]
        flat = torch.zeros((sum(sizes),), device=dev)
        it = iter([v.view(s) for v, s in zip(flat.split(sizes), shapes)])
        gap, gal = ([next(it) for _ in range(3)], [next(it) for _ in range(3)]) if need_app else (None, None)
        gdp, gdl = ([next(it) for _ in range(3)], [next(it) for _ in range(3)]) if need_dens else (None, None)
        g_basis = next(it) if need_basis else None
        head_grads = [next(it) for _ in h.params] if need_head else None
        n_app = sum(sizes[0:6]) if need_app else 0

        d_o = torch.empty((N, 3), device=dev)
        d_d = torch.empty((N, 3), device=dev)
        with TIMER.span("ray_init"):
            check(lib.jt_ray_init(_p(h.rays_d), _p(dnorm), N, _p(d_o), _p(d_d), _stream()), "jt_ray_init")

        # the head backward and dcomps feed the appearance scatter (factor or ray gradients) and the weight gradients
        dcomps = None
        if need_app or need_rays or need_basis or need_head:
            dcomps = torch.empty((cap, afs.ctot), device=dev, dtype=h.dcomps_dtype)
            h.backward(dout, dcomps, g_basis, head_grads)
        o = 0
        for app, max_ctas, plane_mask, cut in parallel.scatter_schedule(sync, need_app, need_dens, need_rays, sizes,
                                                                        n_app, 4 if dfs.C[0] == 16 else 3):
            fs, gp, gl, slot, n_dev, n_max, gin = ((afs, gap, gal, h.aidx, h.a_count, cap, dcomps) if app else
                                                   (dfs, gdp, gdl, None, comp.count, cap_v, dsig))
            ops.vm_scatter_rays(app, fs, gp, gl, comp.samp, slot, comp.sidx, n_dev, n_max, gin, cfg.n_samples,
                                cfg.h_inv, d_o, d_d, max_ctas=max_ctas, plane_mask=plane_mask)
            if cut is not None:
                sync.on_app_grads(flat[o:cut])
                o = cut
        if sync is not None:
            # the current stream waits here for all reductions: whatever autograd does with the views next (hand
            # them to p.grad, clone them, feed the adjoint blur) sees the cross-rank sums
            sync.on_rest(flat[n_app:])

        gdpn, gdln = FactorSet.grads_as_nchw(gdp, gdl) if need_dens else ([None] * 3, [None] * 3)
        gapn, galn = FactorSet.grads_as_nchw(gap, gal) if need_app else ([None] * 3, [None] * 3)
        VMRender.last_grad_bucket = flat
        return (None, d_o if need_rays else None, d_d if need_rays else None, None, *gdpn, *gdln, *gapn, *galn, g_basis,
                *(head_grads if need_head else [None] * len(h.params)))


VMRender.last_grad_bucket = None
VMRender.debug_capture = None
VMRender.last_counts = None
