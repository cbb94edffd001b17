"""Frozen-scene backward of the fused render op: only the gradients autograd asks for.

With the scene frozen (freeze_scene(), or requires_grad_(False) on any subset of the field parameters) the render
op's backward skips the factor-gradient bucket, runs the scatter walkers coordinate-only and the tensor-core head
backwards without weight gradients. The ray gradients it returns are the same as with a trainable scene, up to the
order of fp32 atomic sums."""
import pytest
import torch

import joint_tensorf_b200 as jt
from common import golden_names, load_golden, rel_err
from gpu_common import default_opt, forward_kwargs, module_from_golden, record_err
from joint_tensorf_b200 import ops
from joint_tensorf_b200._lib import floats
from vm_reference import vm_adjoint

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GRAD_REL_TOL = 1e-4
TC_GRAD_REL_TOL = 2e-2
NOISE = 1e-5                 # frozen vs trainable scene: fp32 atomic-order noise only


def _group(name):
    if name.startswith(("density_plane", "density_line")):
        return "density"
    if name.startswith(("app_plane", "app_line")):
        return "app"
    return "head"                                   # basis_mat + the shading MLP


def _run(g, head, freeze=()):
    m = module_from_golden(g, DEV)
    m.head_precision = head
    if freeze == "all":
        m.freeze_scene()
    else:
        for k, p in m.named_parameters():
            if _group(k) in freeze:
                p.requires_grad_(False)
    o = g["rays_o"].to(DEV).requires_grad_(True)
    d = g["rays_d"].to(DEV).requires_grad_(True)
    rgb, depth, acc = m.forward(default_opt(g["case"]["shading"], g["case"].get("ndc", False)), o, d,
                                **forward_kwargs(g, DEV))
    ((rgb * g["w_rgb"].to(DEV)).sum() + (acc * g["w_acc"].to(DEV)).sum()).backward()
    return dict(d_rays_o=o.grad, d_rays_d=d.grad, bucket=jt.VMRender.last_grad_bucket.numel(),
                grads={k: (p.grad.detach().clone() if p.grad is not None else None) for k, p in m.named_parameters()})


def _noise(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


@pytest.mark.parametrize("name,head", [(n, "fp32") for n in golden_names()] +
                         [(n, "tc") for n in ["cubic_mlp", "sh_vm48", "ndc_weakview", "ndc_weakview_blur"]])
def test_frozen_scene_ray_gradients_on_reference_golden(name, head):
    g = load_golden(name)
    tol = GRAD_REL_TOL if head == "fp32" else TC_GRAD_REL_TOL
    full, frozen = _run(g, head), _run(g, head, "all")
    errs = {k: rel_err(frozen[k].cpu(), g[k]) for k in ("d_rays_o", "d_rays_d")}
    noise = {k + "|vs_trainable": _noise(frozen[k], full[k]) for k in ("d_rays_o", "d_rays_d")}
    record_err("frozen:" + name, head=head, **errs, **noise)
    assert all(v <= tol for v in errs.values()), errs
    assert all(v <= NOISE for v in noise.values()), noise
    assert all(v is None for v in frozen["grads"].values()), [k for k, v in frozen["grads"].items() if v is not None]
    assert frozen["bucket"] == 0


@pytest.mark.parametrize("frozen_group", ["density", "app", "head"])
@pytest.mark.parametrize("head", ["fp32", "tc"])
@pytest.mark.parametrize("name", ["sh_vm48", "cubic_mlp"])
def test_partially_frozen_scene(name, head, frozen_group):
    g = load_golden(name)
    full, part = _run(g, head), _run(g, head, (frozen_group,))
    errs = {}
    for k, ref in full["grads"].items():
        if _group(k) == frozen_group:
            assert part["grads"][k] is None, k
        else:
            assert part["grads"][k] is not None, k
            errs[k] = _noise(part["grads"][k], ref)
    for k in ("d_rays_o", "d_rays_d"):
        errs[k] = _noise(part[k], full[k])
    record_err(f"partial:{name}:{frozen_group}", head=head, **errs)
    assert all(v <= NOISE for v in errs.values()), errs


# ------------------------------------------------------------------ C ABI
def _scatter_inputs(seed=0):
    g = load_golden("sh_vm48")               # 3 x 16 density / 3 x 48 appearance components
    m = module_from_golden(g, DEV)
    o, d = g["rays_o"].to(DEV).contiguous(), g["rays_d"].to(DEV).contiguous()
    S = g["n_samples"]
    aux = g["jitter"].to(DEV).reshape(-1).contiguous() if g["jitter"] is not None else None
    comp = ops.march_compact(o, d, aux, False, S, m._h_geom(), None)
    dfs = ops.FactorSet([p.detach() for p in m.density_plane], [p.detach() for p in m.density_line])
    afs = ops.FactorSet([p.detach() for p in m.app_plane], [p.detach() for p in m.app_line])
    gen = torch.Generator(device=DEV).manual_seed(seed)
    gin_app = torch.randn((comp.cap, afs.ctot), device=DEV, generator=gen) * 0.1
    gin_dens = torch.randn((comp.cap,), device=DEV, generator=gen) * 0.1
    return m, comp, dfs, afs, gin_app, gin_dens, S, floats(m._h_inv.tolist())


@pytest.mark.parametrize("plane_mask", [1, 3, 7])
@pytest.mark.parametrize("bf16_factors", [False, True])
@pytest.mark.parametrize("app,gin_bf16", [(0, False), (1, False), (1, True)])
def test_coordinate_only_scatter_matches_full_scatter(app, gin_bf16, bf16_factors, plane_mask):
    m, comp, dfs, afs, gin_app, gin_dens, S, h_inv = _scatter_inputs()
    fs = afs if app else dfs
    if bf16_factors:
        fs = fs.with_bf16_store()
    gin = gin_app if app else gin_dens
    if gin_bf16:
        gin = gin.to(torch.bfloat16)
    N = comp.n_rays
    outs = []
    for with_grads in (True, False):
        gp = [torch.zeros_like(p) for p in fs.planes] if with_grads else None
        gl = [torch.zeros_like(p) for p in fs.lines] if with_grads else None
        d_o, d_d = torch.zeros((N, 3), device=DEV), torch.zeros((N, 3), device=DEV)
        ops.vm_scatter_rays(app, fs, gp, gl, comp.samp, None, comp.sidx, comp.count, comp.cap, gin, S, h_inv, d_o, d_d,
                            plane_mask=plane_mask)
        outs.append((d_o, d_d, gp))
    torch.cuda.synchronize()
    (fo, fd, gp), (co, cd, _) = outs
    assert float(fo.abs().max()) > 0 and float(sum(float(x.abs().max()) for x in gp)) > 0
    # The two walks size their persistent grids differently (the coordinate-only variant fits more CTAs per SM), so
    # their segments, and with them the fp32 partial sums of every ray, differ. A ray's d_o / d_d is a sum of terms
    # that cancel, so that rounding is stated per entry against the sum of |terms| of the float64 reference: each walk
    # is within 1e-6 of it from the exact value, and the two are within 1e-6 of it from each other. (Relative to the
    # largest entry of the tensor the difference reaches 1.2e-6 on the 3 x 48 appearance factors, run to run.)
    n = int(comp.count.item())
    planes, lines = ((fs.planes, fs.lines) if fs.store is None else
                     ([t.float() for t in fs.store[:3]], [t.float() for t in fs.store[3:]]))
    ref = vm_adjoint(planes, lines, comp.samp, n=n, gin=gin[:n], sidx=comp.sidx, S=S, n_rays=N, inv=list(h_inv))
    on = [i for i in range(3) if plane_mask >> i & 1]
    errs = {}
    for name, full, coord, r, mag in (("d_o", fo, co, ref.d_o_plane, ref.d_o_mag_plane),
                                      ("d_d", fd, cd, ref.d_d_plane, ref.d_d_mag_plane)):
        r, mag = sum(r[i] for i in on), sum(mag[i] for i in on).clamp_min(1e-300)
        errs[name + "|coord_vs_full"] = float(((coord.double() - full.double()).abs() / mag).max())
        errs[name + "|full_vs_f64"] = float(((full.double() - r).abs() / mag).max())
        errs[name + "|coord_vs_f64"] = float(((coord.double() - r).abs() / mag).max())
        errs[name + "|coord_vs_full_of_max"] = _noise(coord, full)
    record_err(f"coordinate_only_scatter:app{app}:gin_bf16={gin_bf16}:bf16={bf16_factors}:mask{plane_mask}", **errs)
    assert all(v <= 1e-6 for k, v in errs.items() if not k.endswith("_of_max")), errs


def _weights(shape_list, seed):
    gen = torch.Generator().manual_seed(seed)
    return [(torch.randn(s, generator=gen) * 0.2).to(DEV) for s in shape_list]


def test_sh_bwd_tc_without_weight_gradient_is_bit_identical():
    A, gen = 20000, torch.Generator().manual_seed(1)
    dout = torch.zeros((A, 4), device=DEV)
    dout[:, :3] = (torch.randn(A, 3, generator=gen) * 0.1).to(DEV)
    featdir = torch.zeros((A, 32), device=DEV)
    featdir[:, 28:31] = torch.nn.functional.normalize(torch.randn(A, 3, generator=gen), dim=-1).to(DEV)
    (wb,) = _weights([(27, 144)], 2)
    cnt = torch.tensor([A], device=DEV, dtype=torch.int32)
    stage = ops.head_tc_stage(A, DEV).zero_()
    dc_full = torch.empty((A, 144), device=DEV, dtype=torch.bfloat16)
    dc_frozen = torch.empty_like(dc_full)
    ops.sh_bwd_tc(dout, featdir, wb, cnt, A, dc_full, stage, torch.zeros((27, 144), device=DEV))
    ops.sh_bwd_tc(dout, featdir, wb, cnt, A, dc_frozen, None, None)
    torch.cuda.synchronize()
    assert torch.equal(dc_full, dc_frozen)


@pytest.mark.parametrize("dc_dtype", [torch.float32, torch.bfloat16])
def test_head_bwd_tc_without_weight_gradients_is_bit_identical(dc_dtype):
    A, S, n_rays = 20000, 64, 37
    gen = torch.Generator().manual_seed(3)
    comps = (torch.rand(A, 144, generator=gen) * 0.05).to(DEV)
    rays_d = torch.randn(n_rays, 3, generator=gen).to(DEV)
    sidx = (torch.randint(0, n_rays, (A,), generator=gen) * S + torch.randint(0, S, (A,), generator=gen)).int().to(DEV)
    aidx = torch.randperm(A, generator=gen).int().to(DEV)
    wb, w1, b1, w2, b2, w3, b3 = _weights([(27, 144), (64, 150), (64,), (64, 64), (64,), (3, 64), (3,)], 4)
    cnt = torch.tensor([A], device=DEV, dtype=torch.int32)
    rgb, feat = torch.zeros((A, 4), device=DEV), torch.zeros((A, 28), device=DEV)
    stage = ops.head_tc_stage(A, DEV)
    ops.head_fwd_tc(2, comps, aidx, sidx, rays_d, S, False, wb, w1, b1, w2, b2, w3, b3, cnt, A, 0.8, 0.6, rgb, feat, stage)
    dout = torch.zeros((A, 4), device=DEV)
    dout[:, :3] = (torch.randn(A, 3, generator=gen) * 0.1).to(DEV)
    dc_full, dc_frozen = torch.empty((A, 144), device=DEV, dtype=dc_dtype), torch.empty((A, 144), device=DEV, dtype=dc_dtype)
    grads = [torch.zeros_like(t) for t in (wb, w1, b1, w2, b2, w3, b3)]
    ops.head_bwd_tc(dout, feat, wb, w1, w2, w3, cnt, A, 0.8, dc_full, stage, grads)
    ops.head_bwd_tc(dout, feat, wb, w1, w2, w3, cnt, A, 0.8, dc_frozen, stage, None)
    torch.cuda.synchronize()
    assert torch.equal(dc_full, dc_frozen)
    assert float(grads[1].abs().max()) > 0


def test_wv_head_bwd_tc_without_weight_gradients_is_bit_identical():
    A, S, n_rays = 20000, 64, 37
    gen = torch.Generator().manual_seed(5)
    comps = (torch.rand(A, 60, generator=gen) * 0.05).to(DEV)
    rays_d = torch.randn(n_rays, 3, generator=gen).to(DEV)
    sidx = (torch.randint(0, n_rays, (A,), generator=gen) * S + torch.randint(0, S, (A,), generator=gen)).int().to(DEV)
    aidx = torch.randperm(A, generator=gen).int().to(DEV)
    wb, w1, b1, w2, b2, w3, b3 = _weights([(20, 60), (32, 100), (32,), (32, 32), (32,), (3, 44), (3,)], 6)
    cnt = torch.tensor([A], device=DEV, dtype=torch.int32)
    rgb, featdir = torch.zeros((A, 4), device=DEV), torch.zeros((A, 32), device=DEV)
    stage = ops.wv_stage(A, DEV)
    ops.wv_head_fwd_tc(comps, aidx, sidx, rays_d, S, True, wb, w1, b1, w2, b2, w3, b3, cnt, A, 1.0, 1.0, featdir, rgb,
                       stage)
    dout = torch.zeros((A, 4), device=DEV)
    dout[:, :3] = (torch.randn(A, 3, generator=gen) * 0.1).to(DEV)
    dc_full, dc_frozen = torch.empty((A, 60), device=DEV), torch.empty((A, 60), device=DEV)
    grads = [torch.zeros_like(t) for t in (wb, w1, b1, w2, b2, w3, b3)]
    ops.wv_head_bwd_tc(dout, featdir, wb, w1, w2, w3, cnt, A, 1.0, dc_full, stage, grads)
    ops.wv_head_bwd_tc(dout, featdir, wb, w1, w2, w3, cnt, A, 1.0, dc_frozen, stage, None)
    torch.cuda.synchronize()
    assert torch.equal(dc_full, dc_frozen)
    assert float(grads[1].abs().max()) > 0


# ------------------------------------------------------------------ full size
@pytest.mark.parametrize("wl", ["cfg2_sh", "cfg4"])
def test_full_size_frozen_scene_step(wl):
    """One test-time step at the benchmark's field sizes (4096 rays of one view): the frozen scene's ray gradients
    are the trainable scene's, no factor-gradient bucket is allocated, and the backward's peak memory drops by at
    least the factor bytes."""
    kw, run = jt.synth.config(wl)
    kw = dict(kw)
    ndc = bool(run["ndc"])
    if ndc:
        kw["near_far"] = [-1.0, 1.0]
    torch.manual_seed(0)
    m = jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), DEV, **kw)
    m.head_precision = "tc"
    S = run["n_samples"]
    o, d, _ = jt.synth.llff_ndc_rays(4096, 1) if ndc else jt.synth.blender_rays(4096, 1)
    o, d = o.to(DEV), d.to(DEV)
    tgt = torch.rand((4096, 3), generator=torch.Generator().manual_seed(5)).to(DEV)
    opt = default_opt(m.shadingMode, ndc)
    factor_bytes = sum(p.numel() * 4 for p in [*m.density_plane, *m.density_line, *m.app_plane, *m.app_line])

    def step():
        og, dg = o.clone().requires_grad_(True), d.clone().requires_grad_(True)
        rgb, _, _ = m.forward(opt, og, dg, white_bg=run["white_bg"], is_train=False, ndc_ray=ndc, N_samples=S)
        loss = ((rgb - tgt) ** 2).mean()
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        loss.backward()
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - base
        for p in m.parameters():
            p.grad = None
        return og.grad, dg.grad, peak, jt.VMRender.last_grad_bucket.numel()

    go_full, gd_full, peak_full, nb_full = step()
    m.freeze_scene()
    go, gd, peak, nb = step()
    errs = dict(d_rays_o=_noise(go, go_full), d_rays_d=_noise(gd, gd_full))
    record_err(f"frozen_full:{wl}", head="tc", peak_full_mb=peak_full / 2**20, peak_frozen_mb=peak / 2**20,
               factor_mb=factor_bytes / 2**20, **errs)
    assert nb == 0 and nb_full > 0
    assert all(v <= NOISE for v in errs.values()), errs
    assert peak_full - peak >= factor_bytes, (peak_full, peak, factor_bytes)


# ------------------------------------------------------------------ end to end
@pytest.mark.parametrize("head", ["tc", "fp32"])
def test_test_time_pose_optimisation_on_frozen_scene(head):
    """se3 -> rays (jt_pose_rays) -> render -> photometric loss, on a seeded 128^3 Blender field (SH shading):
    the frozen scene gives the trainable scene's d se3, Adam on se3 lowers the loss, and the tc / SH backward is
    re-entrant on a frozen scene as well."""
    kw, run = jt.synth.config("cfg2_sh")
    kw = dict(kw)
    kw["gridSize"] = [128] * 3
    torch.manual_seed(0)
    m = jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), DEV, **kw)
    m.head_precision = head
    with torch.no_grad():
        for p in [*m.density_plane, *m.density_line]:
            p.mul_(3.0)
    S = run["n_samples"]
    opt = default_opt(m.shadingMode, False)
    H = W = 800
    pose, intr = jt.synth.blender_views(1, (H, W), seed=3)
    pose, kinv = pose.to(DEV), intr.inverse().to(DEV)
    cam = jt.options.Namespace(H=H, W=W, camera=dict(model="perspective", ndc=False), arch=dict())
    pix = torch.randperm(H * W, generator=torch.Generator().manual_seed(9))[:4096].to(torch.int32).to(DEV)
    with torch.no_grad():
        c, r = jt.camera.get_center_and_ray(cam, pose, kinv, ray_idx=pix)
        target = m.forward(opt, c.view(-1, 3), r.view(-1, 3), white_bg=True, is_train=False, N_samples=S)[0]
    noise = torch.tensor([[0.02, -0.015, 0.01, 0.03, -0.02, 0.025]], device=DEV)
    start = jt.camera.refined_pose(noise, pose)
    se3 = torch.nn.Parameter(torch.zeros((1, 6), device=DEV))

    def loss_fn():
        c, r = jt.camera.get_center_and_ray(cam, start, kinv, ray_idx=pix, se3_refine=se3)
        rgb = m.forward(opt, c.view(-1, 3), r.view(-1, 3), white_bg=True, is_train=False, N_samples=S)[0]
        return ((rgb - target) ** 2).mean()

    loss_fn().backward()
    g_full = se3.grad.clone()
    se3.grad = None
    for p in m.parameters():
        p.grad = None
    m.freeze_scene()
    loss0 = loss_fn()
    loss0.backward()
    g_frozen = se3.grad.clone()
    assert all(p.grad is None for p in m.parameters())
    noise_err = _noise(g_frozen, g_full)
    if head == "tc":                                 # re-entrant backward through the same frozen render call
        se3.grad = None
        loss = loss_fn()
        loss.backward(retain_graph=True)
        loss.backward()
        assert _noise(se3.grad, 2 * g_frozen) <= NOISE, _noise(se3.grad, 2 * g_frozen)
    se3.grad = None
    adam = torch.optim.Adam([se3], lr=2e-3)
    for _ in range(20):
        adam.zero_grad()
        loss_fn().backward()
        adam.step()
    with torch.no_grad():
        loss20 = loss_fn()
    record_err(f"tto:{head}", d_se3=noise_err, loss0=loss0.item(), loss20=loss20.item())
    assert noise_err <= NOISE, (g_frozen, g_full)
    assert float(loss20) < float(loss0), (float(loss0), float(loss20))
