"""The fused render op: one autograd node for the whole L1 forward/backward.

Sequence of C-ABI calls for one batch of rays (all on the current stream, no
host synchronisation anywhere -- the reference syncs at every boolean-mask
index, SURVEY.md section 2b):

  forward   jt_march_compact -> jt_vm_gather_fwd(density) -> jt_alpha_fwd -> appearance + shading:
              tcgen05, SH shading        jt_app_basis_sh_fwd_tc          (gather + basis_mat + SHRender, one kernel)
              tcgen05, MLP_Fea head      jt_app_basis_fwd_tc -> jt_head_mlp_fwd_tc
              strict fp32 (any head)     jt_vm_gather_fwd(app) -> jt_gemm_nt(basis) -> jt_pe_encode / jt_gemm_nt / jt_sh_shade
            -> jt_composite_fwd
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
import torch

from . import _lib, ops
from ._lib import check, floats
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


def tc_supported(cfg, afs=None, raise_if_not=False, comps=None):
    """The tensor-core heads are specialised for the shipped configurations: Blender = 3 x 48 appearance
    components, app_dim 27, MLP_Fea (hidden 64, fea_pe = view_pe = 2) or SH shading."""
    comps = list(afs.C) if afs is not None else (list(comps) if comps is not None else None)
    c48 = comps is None or all(int(c) == 48 for c in comps)
    ok = (cfg.shading == "MLP_Fea" and cfg.app_dim == 27 and cfg.hidden == 64 and cfg.fea_pe == 2 and
          cfg.view_pe == 2 and c48)
    ok = ok or (cfg.shading == "SH" and cfg.app_dim == 27 and c48)
    # LLFF = 3 x 20 components, app_dim 20, MLP_Fea_WeakView (hidden 32, fea_pe = view_pe = 2): csrc/weakview_tc.cu
    c20 = comps is None or all(int(c) == 20 for c in comps)
    ok = ok or (cfg.shading == "MLP_Fea_WeakView" and cfg.app_dim == 20 and cfg.hidden == 32 and cfg.fea_pe == 2 and
                cfg.view_pe == 2 and c20)
    if not ok and raise_if_not:
        raise _lib.JtError("head='tc' needs 3 x 48 appearance components, app_dim 27 and MLP_Fea (hidden 64, pe 2) or "
                           "SH shading, or 3 x 20 components, app_dim 20 and MLP_Fea_WeakView (hidden 32, pe 2); "
                           "use head='fp32'")
    return ok


class _Head:
    """Forward/backward of the shading head on compacted appearance samples."""

    @staticmethod
    def forward(cfg, ws, feat, ldf, aidx, sidx, rays_d, a_count, cap, params, dev):
        F, H = cfg.app_dim, cfg.hidden
        rgb = torch.empty((cap, 4), device=dev)
        if cfg.shading == "SH":
            ops.sh_shade(0, feat, ldf, aidx, sidx, rays_d, cfg.n_samples, cfg.ndc, a_count, cap, rgb, None, None, 0)
            return rgb
        w1, b1, w2, b2, w3, b3 = params
        if cfg.shading == "MLP_Fea":
            in_dim = F + 3 + 2 * cfg.fea_pe * F + 6 * cfg.view_pe
            ldi = _r4(in_dim)
            x = torch.empty((cap, ldi), device=dev)
            ops.pe_encode(0, F, cfg.fea_pe, cfg.view_pe, 0, cfg.fea_prog, cfg.view_prog, cfg.n_samples, cfg.ndc,
                          feat, ldf, aidx, sidx, rays_d, a_count, cap, x, ldi)
            h1 = torch.empty((cap, H), device=dev)
            ops.gemm_nt(x, ldi, w1, in_dim, 0, b1, h1, H, None, 0, a_count, cap, H, in_dim, 1, name="mlp_l1_fwd")
            h2 = torch.empty((cap, H), device=dev)
            ops.gemm_nt(h1, H, w2, H, 0, b2, h2, H, None, 0, a_count, cap, H, H, 1, name="mlp_l2_fwd")
            ops.gemm_nt(h2, H, w3, H, 0, b3, rgb, 4, None, 0, a_count, cap, 3, H, 2, name="mlp_l3_fwd")
            ws.update(x=x, ldi=ldi, in_dim=in_dim, h1=h1, h2=h2)
        elif cfg.shading == "MLP_Fea_WeakView":
            in_dim = F + 2 * cfg.fea_pe * F
            ldi = _r4(in_dim)
            nv = 6 * cfg.view_pe
            assert nv % 4 == 0, "view_pe must be even for the WeakView layout"
            ldm = nv + H
            x = torch.empty((cap, ldi), device=dev)
            mid = torch.empty((cap, ldm), device=dev)
            ops.pe_encode(0, F, cfg.fea_pe, cfg.view_pe, 1, cfg.fea_prog, cfg.view_prog, cfg.n_samples, cfg.ndc,
                          feat, ldf, aidx, sidx, rays_d, a_count, cap, x, ldi, mid, ldm)
            h1 = torch.empty((cap, H), device=dev)
            ops.gemm_nt(x, ldi, w1, in_dim, 0, b1, h1, H, None, 0, a_count, cap, H, in_dim, 1, name="mlp_l1_fwd")
            ops.gemm_nt(h1, H, w2, H, 0, b2, mid, ldm, None, 0, a_count, cap, H, H, 1, name="mlp_l2_fwd", y_off=nv)
            ops.gemm_nt(mid, ldm, w3, ldm, 0, b3, rgb, 4, None, 0, a_count, cap, 3, ldm, 2, name="mlp_l3_fwd")
            ws.update(x=x, ldi=ldi, in_dim=in_dim, h1=h1, mid=mid, ldm=ldm, nv=nv)
        else:
            raise _lib.JtError(f"shading model {cfg.shading!r} is not implemented by the B200 path")
        return rgb

    @staticmethod
    def backward(cfg, ws, dout, feat, ldf, aidx, sidx, rays_d, a_count, cap, params, dev, wgrad=True):
        """dout [cap,4] -> dfeat [cap, ldf]; returns (dfeat, param grads list). wgrad=False (frozen head): the weight
        gradient GEMMs are skipped and the list is empty."""
        F, H = cfg.app_dim, cfg.hidden
        dfeat = torch.empty((cap, ldf), device=dev)
        if cfg.shading == "SH":
            ops.sh_shade(1, feat, ldf, aidx, sidx, rays_d, cfg.n_samples, cfg.ndc, a_count, cap, None, dout, dfeat, ldf)
            return dfeat, []
        w1, b1, w2, b2, w3, b3 = params
        gw1, gb1, gw2, gb2, gw3, gb3 = [torch.zeros_like(t) for t in params] if wgrad else [None] * 6
        x, ldi, in_dim, h1 = ws["x"], ws["ldi"], ws["in_dim"], ws["h1"]
        dh2 = torch.empty((cap, H), device=dev)
        dh1 = torch.empty((cap, H), device=dev)
        if cfg.shading == "MLP_Fea":
            h2 = ws["h2"]
            if wgrad:
                ops.gemm_tn(dout, 4, h2, H, a_count, cap, 3, H, gw3, H, gb3, name="mlp_l3_bwd_w")
            ops.gemm_nt(dout, 4, w3, H, 1, None, dh2, H, h2, H, a_count, cap, H, 3, 0, name="mlp_l3_bwd_x")
        else:
            mid, ldm, nv = ws["mid"], ws["ldm"], ws["nv"]
            if wgrad:
                ops.gemm_tn(dout, 4, mid, ldm, a_count, cap, 3, ldm, gw3, ldm, gb3, name="mlp_l3_bwd_w")
            ops.gemm_nt(dout, 4, w3, ldm, 1, None, dh2, H, mid, ldm, a_count, cap, H, 3, 0, name="mlp_l3_bwd_x",
                        w_off=nv, mask_off=nv)
        if wgrad:
            ops.gemm_tn(dh2, H, h1, H, a_count, cap, H, H, gw2, H, gb2, name="mlp_l2_bwd_w")
        ops.gemm_nt(dh2, H, w2, H, 1, None, dh1, H, h1, H, a_count, cap, H, H, 0, name="mlp_l2_bwd_x")
        if wgrad:
            ops.gemm_tn(dh1, H, x, ldi, a_count, cap, H, in_dim, gw1, in_dim, gb1, name="mlp_l1_bwd_w")
        # the encoded input is dead after dW1: reuse its buffer for its own gradient
        ops.gemm_nt(dh1, H, w1, in_dim, 1, None, x, ldi, None, 0, a_count, cap, in_dim, H, 0, name="mlp_l1_bwd_x")
        mode = 0 if cfg.shading == "MLP_Fea" else 1
        ops.pe_encode(1, F, cfg.fea_pe, cfg.view_pe, mode, cfg.fea_prog, cfg.view_prog, cfg.n_samples, cfg.ndc,
                      feat, ldf, None, None, None, a_count, cap, dfeat, ldf, None, 0, x, ldi)
        return dfeat, ([gw1, gb1, gw2, gb2, gw3, gb3] if wgrad else [])


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
        dens, app, basis_w, head = tensors[0:6], tensors[6:12], tensors[12], tensors[13:]
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
        ldf = _r4(F)
        if basis_w.shape != (F, afs.ctot):
            raise _lib.JtError(f"basis_mat weight {tuple(basis_w.shape)} != ({F}, {afs.ctot})")

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

        ws = {}
        comps = None
        if cfg.head == "tc" and cfg.shading == "MLP_Fea_WeakView":
            tc_supported(cfg, afs, raise_if_not=True)
            comps = torch.empty((cap, afs.ctot), device=dev)
            ops.vm_gather_fwd(1, afs, comp.samp, aidx, a_count, cap, comps)
            feat = torch.empty((cap, 32), device=dev)             # feat 0..19 | 0 | view dir 28..30 | 0
            rgb = torch.empty((cap, 4), device=dev)
            ws["stage"] = ops.wv_stage(cap, dev) if train else None
            ops.wv_head_fwd_tc(comps, aidx, comp.sidx, rays_d, S, cfg.ndc, basis_w, *head, a_count, cap, cfg.fea_prog,
                               cfg.view_prog, feat, rgb, ws["stage"])
            comps = None                                          # the staged bf16 tile replaces it in the backward
        elif cfg.head == "tc":
            tc_supported(cfg, afs, raise_if_not=True)
            rgb = torch.empty((cap, 4), device=dev)
            feat = torch.empty((cap, 32), device=dev)             # feat 0..26 | 0 | view dir 28..30 | 0
            # SH: the staged component tile only feeds the basis_mat weight gradient (MLP_Fea: the data backward
            # reads the staged relu tiles as well)
            sh_stage = ctx.needs_input_grad[16] or _full_backward(cfg)
            ws["stage"] = ops.head_tc_stage(cap, dev) if train and (cfg.shading != "SH" or sh_stage) else None
            if cfg.shading == "SH":
                ops.app_basis_sh_fwd_tc(cfg.tc_fwd_split, afs, comp.samp, aidx, comp.sidx, rays_d, S, cfg.ndc,
                                        basis_w, a_count, cap, feat, rgb, ws["stage"])
            else:
                ops.app_basis_fwd_tc(cfg.tc_fwd_split, afs, comp.samp, aidx, comp.sidx, rays_d, S, cfg.ndc, basis_w,
                                     a_count, cap, feat, ws["stage"])
                # inference: fp16 operand tiles (one MMA per product, half the shared memory, two CTAs per SM); the
                # training forward keeps the hi+lo bf16 split because its staged tiles feed the bf16 backward GEMMs
                mlp_split = 3 if (not train and cfg.tc_infer_fp16 and cfg.tc_fwd_split == 2) else cfg.tc_fwd_split
                ops.head_mlp_fwd_tc(mlp_split, feat, *head, a_count, cap, cfg.fea_prog, cfg.view_prog, rgb,
                                    ws["stage"])
        else:
            comps = torch.empty((cap, afs.ctot), device=dev)
            ops.vm_gather_fwd(1, afs, comp.samp, aidx, a_count, cap, comps)
            feat = torch.empty((cap, ldf), device=dev)
            ops.gemm_nt(comps, afs.ctot, basis_w, afs.ctot, 0, None, feat, ldf, None, 0, a_count, cap, F, afs.ctot, 0,
                        name="basis_fwd")
            rgb = _Head.forward(cfg, ws, feat, ldf, aidx, comp.sidx, rays_d, a_count, cap, head, dev)

        rgb_pre = torch.empty((N, 3), device=dev)
        rgb_map = torch.empty((N, 3), device=dev)
        depth = torch.empty((N,), device=dev)
        opacity = torch.empty((N,), device=dev)
        with TIMER.span("composite_fwd"):
            check(lib.jt_composite_fwd(_p(app_off), N, _p(aidx), _p(weight), _p(rgb), _p(acc), _p(wz), _p(rays_d),
                                       int(cfg.white_bg), float(cfg.depth_bias), _p(rgb_pre), _p(rgb_map),
                                       _p(depth), _p(opacity), int(cap), _stream()), "jt_composite_fwd")

        ctx.cfg, ctx.comp, ctx.dfs, ctx.afs, ctx.ws = cfg, comp, dfs32, afs32, ws
        ctx.bufs = dict(rays_d=rays_d, sigfeat=sigfeat, weight=weight, trans=trans, app_off=app_off, aidx=aidx,
                        app_of=app_of, comps=comps, feat=feat, rgb=rgb, rgb_pre=rgb_pre, basis_w=basis_w, head=head,
                        a_count=a_count)
        ctx.n_head = len(head)
        ctx.acap = cap
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
        cfg, comp, dfs, afs, ws, b = ctx.cfg, ctx.comp, ctx.dfs, ctx.afs, ctx.ws, ctx.bufs
        _ = ctx.saved_tensors                                 # raises if a parameter was modified in place since forward
        if ws.get("consumed"):
            raise _lib.JtError("second backward through the same render call: the strict-fp32 MLP head reuses its "
                               "encoded-input buffer for the input gradient (2.6 GB at 4096 x 1000 samples); call "
                               "forward again, or use head_precision='tc' / SH shading, whose backward is re-entrant")
        dev = g_rgb.device
        N, cap_v, cap = comp.n_rays, comp.cap, ctx.acap       # cap: appearance-stage capacity, cap_v = N*S
        F = cfg.app_dim
        ldf = _r4(F)
        g_rgb = g_rgb.contiguous().float()
        g_acc = g_acc.contiguous().float() if g_acc is not None else None
        shade_act = 2 if cfg.shading == "SH" else 1

        dout = torch.empty((cap, 4), device=dev)
        dsig = torch.empty((cap_v,), device=dev)
        dnorm = torch.empty((N,), device=dev) if cfg.ndc else None
        with TIMER.span("render_bwd"):
            check(lib.jt_render_bwd(_p(comp.ray_off), N, _p(b["sigfeat"]), _p(comp.dist), _p(b["weight"]),
                                    _p(b["trans"]), _p(b["app_of"]), _p(b["rgb"]), _p(b["rgb_pre"]), _p(g_rgb),
                                    _p(g_acc), float(cfg.density_shift), cfg.act, float(cfg.distance_scale),
                                    int(cfg.white_bg), shade_act, _p(dout), _p(dsig), _p(dnorm), _stream()),
                  "jt_render_bwd")

        if VMRender.debug_capture is not None:            # diagnostics (scripts/debug_cfg4_grad.py): per-sample gradients
            VMRender.debug_capture.update(dsig=dsig.clone(), dout=dout.clone(), count=comp.count.clone(),
                                          weight=b["weight"].clone(), trans=b["trans"].clone(), rgb=b["rgb"].clone(),
                                          sigfeat=b["sigfeat"].clone(), a_count=b["a_count"].clone())

        # Only the gradients autograd asks for. Input order: cfg, rays_o, rays_d, aux, 6 density factors, 6 appearance
        # factors, basis_mat, head parameters. With an active gradient synchroniser every rank runs the full backward,
        # so that all ranks issue the same collectives whatever their parameters' requires_grad.
        sync = cfg.grad_sync if _full_backward(cfg) else None      # None: world size 1, or inside `sync.paused()`
        ng = ctx.needs_input_grad
        if sync is not None:
            need_rays = need_dens = need_app = need_basis = need_head = True
        else:
            need_rays, need_dens, need_app = ng[1] or ng[2], any(ng[4:10]), any(ng[10:16])
            need_basis, need_head = ng[16], any(ng[17:])
        need_wgrad = need_basis or need_head

        # One flat zero-filled bucket for every gradient this node produces (one memset; also the unit the
        # data-parallel all-reduce works on): [app planes, app lines | density planes, density lines | basis, head],
        # each group present only when it is needed. The appearance part comes first and is complete first, so a
        # gradient synchroniser (parallel.OverlappedGradSync) can reduce it across ranks while the density scatter
        # still runs.
        shapes = ([p.shape for p in afs.planes] + [l.shape for l in afs.lines] if need_app else []) + \
                 ([p.shape for p in dfs.planes] + [l.shape for l in dfs.lines] if need_dens else []) + \
                 ([b["basis_w"].shape] if need_basis else []) + ([t.shape for t in b["head"]] if need_head else [])
        sizes = [int(torch.Size(s).numel()) for s in shapes]
        flat = torch.zeros((sum(sizes),), device=dev)
        views, o = [], 0
        for s, n in zip(shapes, sizes):
            views.append(flat[o:o + n].view(s))
            o += n
        it = iter(views)
        gap, gal = ([next(it) for _ in range(3)], [next(it) for _ in range(3)]) if need_app else (None, None)
        gdp, gdl = ([next(it) for _ in range(3)], [next(it) for _ in range(3)]) if need_dens else (None, None)
        g_basis = next(it) if need_basis else None
        head_grads = [next(it) for _ in b["head"]] if need_head else None
        n_app = sum(sizes[0:6]) if need_app else 0

        d_o = torch.empty((N, 3), device=dev)
        d_d = torch.empty((N, 3), device=dev)
        with TIMER.span("ray_init"):
            check(lib.jt_ray_init(_p(b["rays_d"]), _p(dnorm), N, _p(d_o), _p(d_d), _stream()), "jt_ray_init")

        # the head backward and dcomps feed the appearance scatter (factor or ray gradients) and the weight gradients
        dcomps = None
        if need_app or need_rays or need_wgrad:
            # the tensor-core heads produce all weight gradients or none: a frozen one gets scratch that is dropped
            wgrads = None
            if need_wgrad:
                wgrads = (g_basis if need_basis else torch.zeros_like(b["basis_w"]),
                          *(head_grads if need_head else [torch.zeros_like(t) for t in b["head"]]))
            # tensor-core head: dcomps crosses HBM as bf16 (its GEMM operands are bf16 already)
            wv_tc = cfg.head == "tc" and cfg.shading == "MLP_Fea_WeakView"
            dcomps = torch.empty((cap, afs.ctot), device=dev,
                                 dtype=torch.bfloat16 if (cfg.head == "tc" and not wv_tc) else torch.float32)
            if wv_tc:
                w1, b1, w2, b2, w3, b3 = b["head"]
                ops.wv_head_bwd_tc(dout, b["feat"], b["basis_w"], w1, w2, w3, b["a_count"], cap, cfg.fea_prog, dcomps,
                                   ws["stage"], wgrads)
            elif cfg.head == "tc" and cfg.shading == "SH":
                # no staged component tile when basis_mat was frozen in the forward: no weight gradient either
                sh_gb = g_basis if (need_basis and ws["stage"] is not None) else None
                ops.sh_bwd_tc(dout, b["feat"], b["basis_w"], b["a_count"], cap, dcomps, ws["stage"], sh_gb)
            elif cfg.head == "tc":
                w1, b1, w2, b2, w3, b3 = b["head"]
                ops.head_bwd_tc(dout, b["feat"], b["basis_w"], w1, w2, w3, b["a_count"], cap, cfg.fea_prog, dcomps,
                                ws["stage"], wgrads)
            else:
                dfeat, hg = _Head.backward(cfg, ws, dout, b["feat"], ldf, b["aidx"], comp.sidx, b["rays_d"],
                                           b["a_count"], cap, b["head"], dev, wgrad=need_head)
                if cfg.shading != "SH":
                    ws["consumed"] = True
                for dst, src in zip(head_grads or [], hg):
                    dst.copy_(src)
                if need_basis:
                    ops.gemm_tn(dfeat, ldf, b["comps"], afs.ctot, b["a_count"], cap, F, afs.ctot, g_basis, afs.ctot,
                                None, name="basis_bwd_w")
                ops.gemm_nt(dfeat, ldf, b["basis_w"], afs.ctot, 1, None, dcomps, afs.ctot, None, 0, b["a_count"], cap,
                            afs.ctot, F, 0, name="basis_bwd_x")
        # a frozen factor group is walked coordinate-only (no factor gradients) when the rays need a gradient
        if sync is None:
            if need_app or need_rays:
                ops.vm_scatter_rays(1, afs, gap, gal, comp.samp, b["aidx"], comp.sidx, b["a_count"], cap, dcomps,
                                    cfg.n_samples, cfg.h_inv, d_o, d_d)
            if need_dens or need_rays:
                ops.vm_scatter_rays(0, dfs, gdp, gdl, comp.samp, None, comp.sidx, comp.count, cap_v, dsig,
                                    cfg.n_samples, cfg.h_inv, d_o, d_d)
        elif getattr(sync, "per_plane", False):
            # variant (OverlappedGradSync(per_plane=True)): the appearance planes are walked one launch per plane and
            # each plane's gradients are all-reduced while the next launches run -- [plane 0] [plane 1] [plane 2 + the
            # three lines] [density + basis_mat + head]. Measured at N = 2 (profiles/r02e): the exposed wait halves
            # (0.21 -> 0.12 ms) but the non-persistent per-plane launches cost 0.11 ms more than they save.
            o = 0
            for i in range(3):
                ops.vm_scatter_rays(1, afs, gap, gal, comp.samp, b["aidx"], comp.sidx, b["a_count"], cap, dcomps,
                                    cfg.n_samples, cfg.h_inv, d_o, d_d, max_ctas=-80, plane_mask=1 << i)
                end = o + sizes[i] if i < 2 else n_app
                sync.on_app_grads(flat[o:end])
                o = end
            ops.vm_scatter_rays(0, dfs, gdp, gdl, comp.samp, None, comp.sidx, comp.count, cap_v, dsig, cfg.n_samples,
                                cfg.h_inv, d_o, d_d, max_ctas=-80)
            sync.on_rest(flat[n_app:])
        elif sync.use_split21(n_app, flat.numel()):
            # data parallel, 4+ ranks with an appearance-dominated bucket: [appearance planes 0+1: one persistent launch] -> all-reduce of their 2/4 of the
            # bucket starts -> [appearance plane 2] -> all-reduce of plane 2 + the three lines -> [density scatter] ->
            # all-reduce of the rest. The collectives get a 0.7 ms window (plane 2 + density) instead of the 0.4 ms of the
            # density scatter alone, which at N = 8 is shorter than the 69 MB all-reduce itself; the two launches that run
            # next to a collective use fixed 80-sample segments on a non-persistent grid, because NCCL's CTAs can only
            # get onto an SM when scatter CTAs retire (a persistent wave holds every SM until its kernel ends).
            # Measured (profiles/r02l_*, r02n8c_*): N = 8: exposed wait 0.36 -> 0.16 ms, the two scatters that share the
            # SMs with a collective lose 0.10 ms, step 3.21 -> 3.12 ms; N = 2: 3.04 vs 3.04 ms; cfg4 at N = 2 gets slower
            # (2.15 -> 2.29: its bucket is half density) -- hence OverlappedGradSync.use_split21.
            ops.vm_scatter_rays(1, afs, gap, gal, comp.samp, b["aidx"], comp.sidx, b["a_count"], cap, dcomps,
                                cfg.n_samples, cfg.h_inv, d_o, d_d, plane_mask=3)
            n01 = sizes[0] + sizes[1]
            sync.on_app_grads(flat[:n01])
            ops.vm_scatter_rays(1, afs, gap, gal, comp.samp, b["aidx"], comp.sidx, b["a_count"], cap, dcomps,
                                cfg.n_samples, cfg.h_inv, d_o, d_d, max_ctas=-80, plane_mask=4)
            sync.on_app_grads(flat[n01:n_app])
            ops.vm_scatter_rays(0, dfs, gdp, gdl, comp.samp, None, comp.sidx, comp.count, cap_v, dsig, cfg.n_samples,
                                cfg.h_inv, d_o, d_d, max_ctas=-80)
            # the current stream waits here for all reductions: whatever autograd does with the views next (hand
            # them to p.grad, clone them, feed the adjoint blur) sees the cross-rank sums
            sync.on_rest(flat[n_app:])
        else:
            # 2 ranks / density-heavy buckets: the appearance part of the bucket is all-reduced while the density
            # scatter runs (non-persistent grid, or a persistent wave that leaves sync.reserve_sms SMs to the collective)
            ops.vm_scatter_rays(1, afs, gap, gal, comp.samp, b["aidx"], comp.sidx, b["a_count"], cap, dcomps,
                                cfg.n_samples, cfg.h_inv, d_o, d_d)
            sync.on_app_grads(flat[:n_app])
            reserve = int(getattr(sync, "reserve_sms", 0))
            resident = 4 if dfs.C[0] == 16 else 3
            ops.vm_scatter_rays(0, dfs, gdp, gdl, comp.samp, None, comp.sidx, comp.count, cap_v, dsig, cfg.n_samples,
                                cfg.h_inv, d_o, d_d, max_ctas=((148 - reserve) * resident if reserve > 0 else -80))
            # the current stream waits here for both reductions: whatever autograd does with the views next (hand
            # them to p.grad, clone them, feed the adjoint blur) sees the cross-rank sums
            sync.on_rest(flat[n_app:])

        gdpn, gdln = FactorSet.grads_as_nchw(gdp, gdl) if need_dens else ([None] * 3, [None] * 3)
        gapn, galn = FactorSet.grads_as_nchw(gap, gal) if need_app else ([None] * 3, [None] * 3)
        VMRender.last_grad_bucket = flat
        return (None, d_o if need_rays else None, d_d if need_rays else None, None, *gdpn, *gdln, *gapn, *galn, g_basis,
                *(head_grads if need_head else [None] * ctx.n_head))


VMRender.last_grad_bucket = None
VMRender.debug_capture = None
VMRender.last_counts = None
