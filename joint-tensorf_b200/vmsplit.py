"""B200_VMSplit -- drop-in for the reference field classes `BAT_VMSplit` /
`TensorVMSplit` (model/tensorf_repr/bateRF.py:7, tensoRF.py:145).

Same constructor, parameter names / logical shapes (so reference checkpoints
load), `forward` signature and maintenance methods as the reference
(SURVEY.md section 8b); selected by the reference engine with
`--arch.tensorf.model=B200_VMSplit` (model/tensorf.py:375). The hot path runs in
csrc/*.cu through the C ABI; VM factors are stored channel-last in memory
(logical shape stays [1,C,H,W]) so the kernels gather whole channel vectors.
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

from . import _lib, ops
from ._lib import floats, ints
from .ops import MAT_MODE, VEC_MODE
from .render import RenderCfg, VMRender, render_normals, shade_points, tc_head

CL = torch.channels_last


# ------------------------------------------------------------------ blur taps (host side, 65 numbers)
def gaussian_taps(t, kernel_size):
    """reference model/kernels.py:16-22 (taps clamped to <= 1, not normalised)."""
    ns = torch.arange(-(kernel_size // 2), kernel_size // 2 + 1, dtype=torch.float32)
    tt = max(t, 0.0001)
    q = ns / tt
    k = 1 / (tt * math.sqrt(2 * math.pi)) * torch.exp(-0.5 * q * q)
    return torch.clamp(k, max=1.0)


def average_taps(t, kernel_size):
    """reference model/kernels.py:24-41 (box filter blended between floor/ceil widths)."""
    if kernel_size % 2 == 0:
        kernel_size += 1
    t = float(t)
    half = kernel_size // 2
    out = torch.zeros(kernel_size)
    for width, wgt in ((min(math.floor(t), half), 1 - t % 1.0), (min(math.ceil(t), half), t % 1.0)):
        box = torch.zeros(kernel_size)
        box[half - width:half + width + 1] = 1 / (width * 2 + 1)
        out = out + wgt * box
    return out


# ------------------------------------------------------------------ occupancy mask
class AlphaGridMask(torch.nn.Module):
    """Binary occupancy volume (reference tensorBase.py:80-98) + its bit-packed
    device copy used by the ray-march kernel."""

    def __init__(self, device, aabb, alpha_volume, packed_bits=None):
        super().__init__()
        self.device = device
        self.aabb = aabb.to(device)
        self.aabbSize = self.aabb[1] - self.aabb[0]
        self.invgridSize = 1.0 / self.aabbSize * 2
        self.alpha_volume = alpha_volume.view(1, 1, *alpha_volume.shape[-3:]).to(device)
        d, h, w = self.alpha_volume.shape[-3:]
        self.gridSize = torch.LongTensor([w, h, d]).to(device)
        self._pack(packed_bits)

    def _pack(self, packed_bits=None):
        d, h, w = self.alpha_volume.shape[-3:]
        if packed_bits is not None:          # already bit-packed by jt_alpha_mask_build
            self.bits = packed_bits
            self.h_dims = ints([w, h, d])
            self.h_geom = floats(self.aabb[0].tolist() + self.invgridSize.tolist())
            return
        flat = (self.alpha_volume.reshape(-1) > 0).to(torch.int64)
        pad = (-flat.numel()) % 32
        if pad:
            flat = torch.cat([flat, flat.new_zeros(pad)])
        words = (flat.view(-1, 32) << torch.arange(32, device=flat.device)).sum(-1)
        words = torch.where(words >= 2 ** 31, words - 2 ** 32, words).to(torch.int32)
        self.bits = words.contiguous()
        self.h_dims = ints([w, h, d])
        self.h_geom = floats(self.aabb[0].tolist() + self.invgridSize.tolist())

    def sample_alpha(self, xyz_sampled):
        """1.0 where the trilinear lookup of the reference would be > 0, else 0.0."""
        xyz = xyz_sampled.reshape(-1, 3).contiguous().float()
        n = xyz.shape[0]
        # a degenerate "ray" per point: o = xyz, d = 0, one sample at depth 0 (NDC table of one entry)
        ztab = torch.zeros((1,), device=xyz.device)
        big = floats([-3e38] * 3 + [3e38] * 3 + [1.0] * 3 + [0.0, 0.0, 0.0])
        _, _, keep = ops.sample_ray_dense(xyz, torch.zeros_like(xyz), ztab, True, 1, big, self)
        return keep.view(-1).float()

    def normalize_coord(self, xyz_sampled):
        return (xyz_sampled - self.aabb[0]) * self.invgridSize - 1


# ------------------------------------------------------------------ appearance-stage capacity (memory model)
class AppCapacityTracker:
    """Host-side bound on the number of appearance samples of a training call.

    A (samples whose weight passes rayMarch_weight_thres) only exists on the device, and the appearance stage is
    where the large per-sample buffers live (staged operand tiles: 1.26 KB per sample with the MLP_Fea head). The
    tracker receives A of every training call through an asynchronous device->pinned-host copy (no
    synchronisation: the value is read when its event has completed, typically one or two calls later), keeps a
    slowly decaying maximum of A per ray, and after `warm` observations sizes the stage to
    `margin * max_per_ray * n_rays + floor` (at most N*S). jt_alpha_fwd clamps the list to that capacity and raises
    a device flag; if the flag ever comes back set, the next forward raises JtError -- the flagged call rendered
    with a truncated appearance list -- and the capacity returns to N*S until the history is rebuilt."""

    def __init__(self, margin=2.0, floor=65536, warm=8, decay=0.995):
        self.margin, self.floor, self.warm, self.decay = margin, floor, warm, decay
        self.reset()

    def reset(self):
        self.max_per_ray, self.seen, self.pending, self.overflow = 0.0, 0, [], None
        self._pool = getattr(self, "_pool", [])

    def submit(self, a_total, app_used, n_rays):
        host = self._pool.pop() if self._pool else torch.empty((3,), dtype=torch.int32).pin_memory()
        host[0:1].copy_(a_total, non_blocking=True)
        host[1:3].copy_(app_used, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self.pending.append((ev, host, int(n_rays)))

    def poll(self):
        while self.pending and self.pending[0][0].query():
            ev, host, n = self.pending.pop(0)
            a, used, ovf = (int(v) for v in host.tolist())
            if ovf:
                self.overflow = (a, used)
            self.max_per_ray = max(self.max_per_ray * self.decay, a / max(n, 1))
            self.seen += 1
            self._pool.append(host)
        if len(self.pending) > 64:                     # nobody polls fast enough: drop the oldest
            self.pending = self.pending[-64:]

    def capacity(self, n_rays, cap):
        self.poll()
        if self.overflow is not None:
            a, used = self.overflow
            self.reset()
            raise _lib.JtError(
                f"appearance capacity exceeded in an earlier training call: {a} appearance samples, buffers sized for "
                f"{used}; that call composited a truncated sample list. The capacity is back to N*S; set "
                "B200_VMSplit.app_capacity = None to keep it there (INTEGRATION.md, memory model).")
        if self.seen < self.warm:
            return None
        return min(int(cap), int(self.margin * self.max_per_ray * n_rays) + self.floor)


# ------------------------------------------------------------------ shading heads (parameter containers)
class MLPRender_Fea(torch.nn.Module):
    """Parameter layout of reference MLPRender_Fea (tensorBase.py:101-114): mlp.{0,2,4}."""

    def __init__(self, in_chanel, viewpe=6, feape=6, featureC=128):
        super().__init__()
        self.in_mlpC = 2 * viewpe * 3 + 2 * feape * in_chanel + 3 + in_chanel
        self.viewpe, self.feape = viewpe, feape
        self.mlp = torch.nn.Sequential(torch.nn.Linear(self.in_mlpC, featureC), torch.nn.ReLU(inplace=True),
                                       torch.nn.Linear(featureC, featureC), torch.nn.ReLU(inplace=True),
                                       torch.nn.Linear(featureC, 3))
        torch.nn.init.constant_(self.mlp[-1].bias, 0)

    def head_params(self):
        m = self.mlp
        return [m[0].weight, m[0].bias, m[2].weight, m[2].bias, m[4].weight, m[4].bias]


class MLPRender_Fea_WeakView(torch.nn.Module):
    """Parameter layout of reference MLPRender_Fea_WeakView (tensorBase.py:180-196)."""

    def __init__(self, in_chanel, viewpe=6, feape=6, featureC=128):
        super().__init__()
        self.in_mlpC = (2 * feape + 1) * in_chanel
        self.mid_mlpC = 2 * viewpe * 3
        self.viewpe, self.feape = viewpe, feape
        self.layer1 = torch.nn.Linear(self.in_mlpC, featureC)
        self.layer2 = torch.nn.Linear(featureC, featureC)
        self.layer3 = torch.nn.Linear(featureC + self.mid_mlpC, 3)
        torch.nn.init.constant_(self.layer3.bias, 0)

    def head_params(self):
        return [self.layer1.weight, self.layer1.bias, self.layer2.weight, self.layer2.bias,
                self.layer3.weight, self.layer3.bias]


_OPT_FLAGS = ("abs_components", "component_wise_feature2density", "plane_feature2density", "convolve_plane_only",
              "convolve_positive_only", "ignore_negative_split")


class B200_VMSplit(torch.nn.Module):
    def __init__(self, aabb, gridSize, device, density_n_comp=8, appearance_n_comp=24, app_dim=27,
                 shadingMode="MLP_PE", alphaMask=None, near_far=[2.0, 6.0], density_shift=-10,
                 alphaMask_thres=0.001, distance_scale=25, rayMarch_weight_thres=0.0001, pos_pe=6, view_pe=6,
                 fea_pe=6, featureC=128, step_ratio=2.0, fea2denseAct="softplus", dtype=torch.float32,
                 volume_init_scale=0.1, volume_init_bias=0.1):
        super().__init__()
        if dtype not in (torch.float32, torch.bfloat16):
            raise _lib.JtError("B200_VMSplit: dtype must be torch.float32 or torch.bfloat16 (bf16 factor storage)")
        self.device = device
        # bf16 factor storage (north star: "bf16/fp32 gathers", <= 2e-2 relative class): the Parameters stay fp32
        # master copies (optimizer state, checkpoints and gradients are unchanged); the gather / scatter kernels read
        # their taps from a bf16 copy refreshed when a factor changes (csrc/factor_store.cu). Selected with
        # dtype=torch.bfloat16 at construction or by setting `factor_storage = "bf16"` afterwards.
        self.factor_storage = "bf16" if dtype == torch.bfloat16 else "fp32"
        self._store_cache = ({}, {})          # bf16 copies of the density / appearance factors (no-blur calls)
        # "auto": training calls size the appearance-stage buffers from the appearance counts of earlier calls
        # (AppCapacityTracker); None: always N*S. No-grad calls read the count on the host and allocate exactly.
        self.app_capacity = "auto"
        self._app_tracker = AppCapacityTracker()
        self.dtype = torch.float32
        self.alphaMask = alphaMask
        self.matMode = [list(m) for m in MAT_MODE]
        self.vecMode = list(VEC_MODE)
        self.comp_w = [1, 1, 1]
        self.kernel_density = None
        self.kernel_color = None
        self.c2f_mode = None
        # shading-head arithmetic: "auto" = tcgen05 tensor-core head when the configuration is
        # supported, else the fp32 SIMT head; "fp32" forces the strict-parity path; "tc" insists.
        self.head_precision = "auto"
        self.tc_fwd_split = 2
        # no-grad calls (evaluation, full-frame rendering) of the tensor-core MLP_Fea head use single-term fp16
        # operand tiles (rgb within ~2e-5 of the training forward, a quarter faster); False keeps them identical
        self.tc_infer_fp16 = True
        self._reg_cache = None
        self.grad_sync = None      # parallel.OverlappedGradSync when training data-parallel
        self.reset(aabb, gridSize, density_n_comp, appearance_n_comp, app_dim, density_shift, alphaMask_thres,
                   distance_scale, rayMarch_weight_thres, fea2denseAct, near_far, step_ratio, shadingMode, pos_pe,
                   view_pe, fea_pe, featureC, volume_init_scale, volume_init_bias)

    # ---------------------------------------------------------------- construction (tensorBase.py:426-488)
    def reset(self, aabb, gridSize, density_n_comp, appearance_n_comp, app_dim, density_shift, alphaMask_thres,
              distance_scale, rayMarch_weight_thres, fea2denseAct, near_far, step_ratio, shadingMode, pos_pe,
              view_pe, fea_pe, featureC, volume_init_scale, volume_init_bias):
        def comps(c):
            return [int(c)] * 3 if isinstance(c, (int, np.integer)) else [int(v) for v in c]
        self.density_n_comp = comps(density_n_comp)
        self.app_n_comp = comps(appearance_n_comp)
        self.app_dim = app_dim
        self.aabb = torch.as_tensor(aabb, dtype=self.dtype).clone().to(self.device)
        self.density_shift = density_shift
        self.alphaMask_thres = alphaMask_thres
        self.distance_scale = distance_scale
        self.rayMarch_weight_thres = rayMarch_weight_thres
        self.fea2denseAct = fea2denseAct
        self.near_far = near_far
        self.step_ratio = step_ratio
        self.update_stepSize(gridSize)
        self.volume_init_scale = volume_init_scale
        self.volume_init_bias = volume_init_bias
        self.init_svd_volume(gridSize[0], self.device, init_scale=volume_init_scale, init_bias=volume_init_bias)
        self.shadingMode, self.pos_pe, self.view_pe, self.fea_pe, self.featureC = shadingMode, pos_pe, view_pe, fea_pe, featureC
        self.init_render_func(shadingMode, pos_pe, view_pe, fea_pe, featureC, self.device)

    def init_render_func(self, shadingMode, pos_pe, view_pe, fea_pe, featureC, device):
        if shadingMode == "MLP_Fea":
            self.renderModule = MLPRender_Fea(self.app_dim, view_pe, fea_pe, featureC).to(device)
        elif shadingMode == "MLP_Fea_WeakView":
            self.renderModule = MLPRender_Fea_WeakView(self.app_dim, view_pe, fea_pe, featureC).to(device)
        elif shadingMode == "SH":
            if self.app_dim != 27:
                raise _lib.JtError("SH shading needs app_dim == 27 (3 x 9 degree-2 coefficients)")
            self.renderModule = None
        else:
            raise Exception(f"Unrecognized / unsupported shading module {shadingMode!r} "
                            "(B200 path implements MLP_Fea, MLP_Fea_WeakView, SH)")

    def update_stepSize(self, gridSize):
        """tensorBase.py:477-488, evaluated with torch fp32 exactly as the reference
        (the resulting floats feed the bit-exact ray-march kernel)."""
        aabb = self.aabb.detach().cpu().float()
        size = aabb[1] - aabb[0]
        g = torch.LongTensor([int(v) for v in gridSize])
        units = size / (g - 1)
        step = torch.mean(units) * self.step_ratio
        diag = torch.sqrt(torch.sum(torch.square(size)))
        self.aabbSize = size.to(self.device)
        self.invaabbSize = (2.0 / size).to(self.device)
        self.gridSize = g.to(self.device)
        self.units = units.to(self.device)
        self.stepSize = step.to(self.device)
        self.aabbDiag = diag.to(self.device)
        self.nSamples = int((diag / step).item()) + 1
        # host copies (no device->host reads on the hot path)
        self._grid = [int(v) for v in g.tolist()]
        self._h_aabb = aabb
        self._h_inv = 2.0 / size
        self._h_step = step
        self._blur_scale = torch.mean(g / size)            # batBase.py:14
        self._ztab_cache = {}

    def init_svd_volume(self, res, device, init_density=True, init_app=True, init_basis=True, init_scale=0.1,
                        init_bias=0.1):
        if init_density:
            self.density_plane, self.density_line = self.init_one_svd(self.density_n_comp, self._grid, init_scale, init_bias, device)
        if init_app:
            self.app_plane, self.app_line = self.init_one_svd(self.app_n_comp, self._grid, init_scale, init_bias, device)
        if init_basis:
            self.basis_mat = torch.nn.Linear(sum(self.app_n_comp), self.app_dim, bias=False).to(device)

    def init_one_svd(self, n_component, gridSize, scale, bias, device):
        """|bias + scale*N(0,1)| factors (tensoRF.py:159-169), stored channel-last."""
        planes, lines = [], []
        for i in range(3):
            m0, m1 = MAT_MODE[i]
            p = torch.abs(bias + scale * torch.randn((1, n_component[i], gridSize[m1], gridSize[m0])))
            l = torch.abs(bias + scale * torch.randn((1, n_component[i], gridSize[VEC_MODE[i]], 1)))
            planes.append(torch.nn.Parameter(_to_cl(p.to(device))))
            lines.append(torch.nn.Parameter(_to_cl(l.to(device))))
        return torch.nn.ParameterList(planes), torch.nn.ParameterList(lines)

    # ---------------------------------------------------------------- small reference helpers
    def normalize_coord(self, xyz_sampled):
        return (xyz_sampled - self.aabb[0]) * self.invaabbSize - 1

    def feature2density(self, density_features):
        if self.fea2denseAct == "softplus":
            return F.softplus(density_features + self.density_shift)
        elif self.fea2denseAct == "relu":
            return F.relu(density_features + self.density_shift)

    def get_optparam_groups(self, lr_init_spatialxyz=0.02, lr_init_network=0.001):
        groups = [{"params": self.density_line, "lr": lr_init_spatialxyz},
                  {"params": self.density_plane, "lr": lr_init_spatialxyz},
                  {"params": self.app_line, "lr": lr_init_spatialxyz},
                  {"params": self.app_plane, "lr": lr_init_spatialxyz},
                  {"params": self.basis_mat.parameters(), "lr": lr_init_network}]
        if isinstance(self.renderModule, torch.nn.Module):
            groups += [{"params": self.renderModule.parameters(), "lr": lr_init_network}]
        return groups

    def freeze_scene(self, opt=None):
        self._set_scene_grad(False)

    def unfreeze_scene(self, opt=None):
        self._set_scene_grad(True)

    def _set_scene_grad(self, flag):
        self.basis_mat.weight.requires_grad = flag
        if isinstance(self.renderModule, torch.nn.Module):
            self.renderModule.requires_grad_(flag)
        for plist in (self.density_plane, self.density_line, self.app_plane, self.app_line):
            for p in plist:
                p.requires_grad = flag

    # ---------------------------------------------------------------- per-step regularisers (section 8f-2)
    _REG_TERMS = (1, 1, 1, 0, 0, 0, 2, 2, 2, 0, 0, 0)      # TV slot: density planes -> 1, app planes -> 2
    _REG_L1 = (1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0)         # L1 covers density planes and lines

    def _reg_factors(self):
        return [*self.density_plane, *self.density_line, *self.app_plane, *self.app_line]

    def _reg_node(self):
        """(L1, TV_density, TV_app) from ONE sweep over the factors, shared by the three methods the
        reference calls back to back (model/tensorf.py:127-130); recomputed when a factor changes."""
        fs = self._reg_factors()
        key = tuple((id(p), p._version, p.requires_grad) for p in fs) + (torch.is_grad_enabled(),)
        if self._reg_cache is None or self._reg_cache[0] != key:
            from .sweeps import FieldRegularizers
            self._reg_cache = (key, FieldRegularizers.apply(self._REG_TERMS, self._REG_L1, *fs))
        return self._reg_cache[1]

    def density_L1(self):
        """tensoRF.py:212-216."""
        return self._reg_node()[0]

    def TV_loss_density(self, reg):
        """tensoRF.py:218-222 with reg = TVLoss (tensorBase.py:16-41); only its weight is read."""
        return self._reg_node()[1] * float(getattr(reg, "TVLoss_weight", 1.0))

    def TV_loss_app(self, reg):
        """tensoRF.py:224-228."""
        return self._reg_node()[2] * float(getattr(reg, "TVLoss_weight", 1.0))

    @torch.no_grad()
    def regularize_(self, w_l1=0.0, w_tv_density=0.0, w_tv_app=0.0, values=True):
        """Fused fast path: p.grad += d/dp (w_l1*L1 + w_tv_density*TV_density + w_tv_app*TV_app) for all factors in
        one sweep, without autograd nodes; returns the [3] value tensor (or None). Terms with a zero weight are
        not swept (Blender configs: TV weights are 0, bat_blender_VM.yaml:138-139)."""
        from . import sweeps
        fs = [p for p in self._reg_factors()]
        xs = [ops.phys_cl(p.data) for p in fs]
        out = sweeps.reg_values(xs, self._REG_TERMS, self._REG_L1) if values else None
        sel = [i for i, p in enumerate(fs) if p.requires_grad]
        gs = []
        for i in sel:
            if fs[i].grad is None:
                fs[i].grad = torch.zeros_like(fs[i], memory_format=torch.preserve_format)
            gs.append(ops.phys_cl(fs[i].grad))
            assert gs[-1].data_ptr() == fs[i].grad.data_ptr(), "gradient buffers must be channel-last like the factors"
        sweeps.reg_grads_([xs[i] for i in sel], gs, [self._REG_TERMS[i] for i in sel],
                          [self._REG_L1[i] for i in sel], (w_l1, w_tv_density, w_tv_app))
        return out

    # ---------------------------------------------------------------- geometry blobs for the C ABI
    def _h_geom(self):
        near, far = self.near_far
        near32 = float(torch.tensor(float(near), dtype=torch.float32))
        far32 = float(torch.tensor(float(far), dtype=torch.float32))
        return floats(self._h_aabb[0].tolist() + self._h_aabb[1].tolist() + self._h_inv.tolist() +
                      [float(self._h_step), near32, far32])

    def _mask(self):
        return self.alphaMask if self.alphaMask is not None else None

    def _ndc_table(self, n_samples, is_train):
        """linspace(near, far, S) built with torch on the CPU (bit-identical to the
        oracle), cached; stratified jitter added on the device (tensorBase.py:556-559)."""
        near, far = float(self.near_far[0]), float(self.near_far[1])
        key = (near, far, n_samples)
        z = self._ztab_cache.get(key)
        if z is None:
            if len(self._ztab_cache) > 64:
                self._ztab_cache.clear()
            z = torch.linspace(near, far, n_samples, dtype=torch.float32).to(self.device)
            self._ztab_cache[key] = z
        if is_train:
            z = z + torch.rand_like(z) * ((far - near) / n_samples)
        return z

    # ---------------------------------------------------------------- K1 API
    def sample_ray(self, rays_o, rays_d, is_train=True, N_samples=-1, jitter=None):
        """tensorBase.py:572-612 -> (rays_pts [N,S,3], interpx [N,S], valid [N,S])."""
        n_samples = N_samples if N_samples > 0 else self.nSamples
        aux = None
        if is_train:
            aux = jitter if jitter is not None else torch.rand((rays_o.shape[0],), device=rays_o.device)
            aux = aux.reshape(-1).contiguous().float()
        return ops.sample_ray_dense(rays_o.detach().contiguous().float(), rays_d.detach().contiguous().float(), aux,
                                    False, n_samples, self._h_geom(), None)

    def sample_ray_ndc(self, rays_o, rays_d, is_train=True, N_samples=-1, simulate_euclid_sample=False,
                       simulate_euclid_depth=False, ndc_near_plane=1.0, jitter=None):
        """tensorBase.py:554-571 (simulate_euclid_* are False in every shipped config)."""
        if simulate_euclid_sample or simulate_euclid_depth:
            raise _lib.JtError("ndc_simulate_euclid_* is not supported by the B200 path (False in all reference configs)")
        n_samples = N_samples if N_samples > 0 else self.nSamples
        z = self._ndc_table(n_samples, is_train and jitter is None)
        if is_train and jitter is not None:
            near, far = float(self.near_far[0]), float(self.near_far[1])
            z = z + jitter.reshape(-1).to(z) * ((far - near) / n_samples)
        pts, zz, valid = ops.sample_ray_dense(rays_o.detach().contiguous().float(),
                                              rays_d.detach().contiguous().float(), z.contiguous(), True, n_samples,
                                              self._h_geom(), None)
        return pts, z.unsqueeze(0), valid

    # ---------------------------------------------------------------- K5 API
    def get_kernel(self, opt, c2f_mode, c2f_parameter, c2f_kernel_size=25):
        """BatBase.get_kernel (batBase.py:13-25). The taps are computed on the host and STAY there: the blur
        kernels take them through their launch parameters (constant bank), so the per-step host->device copy of
        the reference (a stream synchronisation for pageable memory) is gone and the host keeps running ahead
        of the GPU. Returns a CPU tensor carrying the tap list as `_jt_host`."""
        t = self._blur_scale * float(c2f_parameter)
        if c2f_mode == "uniform-gaussian":
            k = gaussian_taps(t, c2f_kernel_size)
        elif c2f_mode == "uniform-average":
            k = average_taps(t, c2f_kernel_size)
        else:
            raise RuntimeError(f"invalid c2f_mode {c2f_mode}")
        kd = k.to(dtype=torch.float32)
        kd._jt_host = kd.reshape(-1).tolist()
        return kd

    def convolute_line(self, kernel, line):
        return ops.BlurFactor.apply(line, kernel, line.shape[2], 1, 2)

    def convolute_plane(self, kernel, plane, H, W):
        return ops.BlurFactor.apply(plane, kernel, int(H), int(W), 3)

    def _blurred(self, planes, lines, kernel):
        """All six factors of one group, blurred (bateRF.py:64-78 / 105-118)."""
        if kernel is None:
            return list(planes), list(lines)
        bp, bl = [], []
        for i in range(3):
            m0, m1 = MAT_MODE[i]
            bp.append(self.convolute_plane(kernel, planes[i], self._grid[m0], self._grid[m1]))
            bl.append(self.convolute_line(kernel, lines[i]))
        return bp, bl

    def _blurred_all(self, kernel_density, kernel_color):
        """The 12 factors of a forward call, blurred by one autograd node / two launches per direction
        (bateRF.py:64-78 and 105-118 run 18 conv1d calls with their pads and permutes)."""
        groups = [(self.density_plane, self.density_line, kernel_density), (self.app_plane, self.app_line, kernel_color)]
        active = [(p, l, k) for p, l, k in groups if k is not None]
        if not active:
            return list(self.density_plane), list(self.density_line), list(self.app_plane), list(self.app_line)
        tapsets, metas, factors = [], [], []
        for p, l, k in active:
            ht = getattr(k, "_jt_host", None)
            tapsets.append(list(ht) if ht is not None else k.detach().reshape(-1).float().cpu().tolist())
        if len(tapsets) == 2 and len(tapsets[0]) != len(tapsets[1]):      # different tap counts: one node per group
            dp, dl = self._blurred(self.density_plane, self.density_line, kernel_density)
            ap, al = self._blurred(self.app_plane, self.app_line, kernel_color)
            return dp, dl, ap, al
        for s, (p, l, k) in enumerate(active):
            for i in range(3):
                m0, m1 = MAT_MODE[i]
                factors.append(p[i])
                metas.append((self._grid[m0], self._grid[m1], 3, s))
            for i in range(3):
                factors.append(l[i])
                metas.append((l[i].shape[2], 1, 2, s))
        outs = list(ops.BlurGroup.apply(metas, tapsets, *factors))
        res = []
        for p, l, k in groups:
            if k is None:
                res += [list(p), list(l)]
            else:
                res += [outs[:3], outs[3:6]]
                outs = outs[6:]
        return res[0], res[1], res[2], res[3]

    # ---------------------------------------------------------------- K2 API
    def compute_densityfeature(self, xyz_sampled, kernel=None, c2f_mode=None, interp_mode="bilinear"):
        """bateRF.py:41-94 / tensoRF.py:230-251: [V,3] normalised coords -> [V]."""
        self._check_interp(interp_mode)
        planes, lines = self._blurred(self.density_plane, self.density_line, kernel if c2f_mode is not None else None)
        return ops.DensityFeature.apply(xyz_sampled.reshape(-1, 3), *planes, *lines)

    def compute_appfeature(self, xyz_sampled, kernel=None, c2f_mode=None, interp_mode="bilinear"):
        """bateRF.py:97-130 / tensoRF.py:254-270: [A,3] -> [A, app_dim]."""
        self._check_interp(interp_mode)
        planes, lines = self._blurred(self.app_plane, self.app_line, kernel if c2f_mode is not None else None)
        comps = ops.AppComponents.apply(xyz_sampled.reshape(-1, 3), *planes, *lines)
        return ops.Linear.apply(comps, self.basis_mat.weight, None)

    @staticmethod
    def _check_interp(mode):
        if mode != "bilinear":
            raise _lib.JtError(f"grid_sample_interp_mode={mode!r}: only 'bilinear' is implemented (all reference configs)")

    def _density_factorset(self):
        """Density factors as the last forward saw them (blurred with the cached density kernel, batBase.py:37)."""
        planes, lines = self._blurred(self.density_plane, self.density_line,
                                      self.kernel_density if self.c2f_mode is not None else None)
        return ops.FactorSet([p.detach() for p in planes], [l.detach() for l in lines])

    def _app_factorset(self):
        """Appearance factors as the last forward saw them (blurred with the cached colour kernel, batBase.py:37)."""
        planes, lines = self._blurred(self.app_plane, self.app_line,
                                      self.kernel_color if self.c2f_mode is not None else None)
        return ops.FactorSet([p.detach() for p in planes], [l.detach() for l in lines])

    _RGB_CHUNK = 1 << 20      # points per head call: bounds the strict-fp32 head's ~2 KB per point of buffers

    @torch.no_grad()
    def compute_rgb(self, xyz_locs, viewdirs):
        """Colour of the field at world points xyz_locs [..., 3] seen along viewdirs [..., 3] (or one [3] for all
        points): rgb [..., 3], the reference's renderModule(pts, viewdirs, compute_appfeature(pts)) as a no-grad
        forward computes it. The head is the one forward picks (head_precision, tc_fwd_split, tc_infer_fp16,
        factor_storage); the appearance factors are blurred with the colour kernel the last forward cached, so
        colour and compute_alpha's geometry come from the same field state; the PE progress is 1. viewdirs reach
        the head as given (not normalised). Points outside the aabb shade zero appearance components, as
        grid_sample's zero padding gives. Rows are independent: the result does not depend on how many points are
        passed at once or in which order."""
        shape = xyz_locs.shape[:-1]
        ops._need_cuda(xyz_locs, "xyz_locs")
        xyz = xyz_locs.reshape(-1, 3).float()
        n = xyz.shape[0]
        if viewdirs.dim() == 1:
            dirs = viewdirs.reshape(1, 3).float().expand(n, 3)
        else:
            dirs = viewdirs.reshape(-1, 3).float()
            if dirs.shape[0] != n:
                raise _lib.JtError(f"compute_rgb: {dirs.shape[0]} view directions for {n} points")
        ops._need_cuda(dirs, "viewdirs")
        storage = self._checked_storage()
        rgb = torch.empty((n, 3), device=xyz.device)
        if n == 0:
            return rgb.view(*shape, 3)
        afs = self._app_factorset()
        if storage == "bf16":          # the bf16 copy is cached, like forward's, only for the unblurred Parameters
            afs = afs.with_bf16_store(self._store_cache[1] if self.c2f_mode is None else None)
        cfg = RenderCfg(**self._head_fields())
        basis_w = self.basis_mat.weight.detach().contiguous()
        head = [t.detach().contiguous() for t in self.renderModule.head_params()] if self.renderModule is not None else []
        for s in range(0, n, self._RGB_CHUNK):
            e = min(n, s + self._RGB_CHUNK)
            rgb[s:e] = shade_points(cfg, afs, self.normalize_coord(xyz[s:e]), dirs[s:e], basis_w, head)
        return rgb.view(*shape, 3)

    @torch.no_grad()
    def compute_alpha(self, xyz_locs, length=1):
        """BatBase.compute_alpha (batBase.py:27-42) as one kernel: mask test, normalisation, density gather,
        activation, 1 - exp(-sigma * length). Reuses the density kernel cached by the last forward."""
        shape = xyz_locs.shape[:-1]
        a = ops.field_alpha(self._density_factorset(), self._h_geom(), self.density_shift,
                            0 if self.fea2denseAct == "softplus" else 1, float(length), xyz=xyz_locs,
                            mask=self.alphaMask)
        return a.view(shape)

    @torch.no_grad()
    def compute_density_grad(self, xyz_locs):
        """Density and its gradient at points xyz_locs [..., 3] in the field's input coordinates (world, or NDC for an
        NDC field): (sigma [...], grad [..., 3]), grad = d sigma / d xyz, the analytic derivative of the field
        compute_alpha evaluates (jt_field_density_grad). Same field state as compute_alpha: the density factors
        blurred with the kernel the last forward cached, the fp32 factors whatever factor_storage is, and the alpha
        mask (rejected points give sigma 0, grad 0). At a cell boundary the derivative is the one-sided one of the
        cell the tap rounding selects. No autograd; rows are independent of each other."""
        shape = xyz_locs.shape[:-1]
        sigma, grad = ops.field_density_grad(self._density_factorset(), self._h_geom(), self.density_shift,
                                             0 if self.fea2denseAct == "softplus" else 1, xyz=xyz_locs,
                                             mask=self.alphaMask)
        return sigma.view(shape), grad.view(*shape, 3)

    @torch.no_grad()
    def compute_normals(self, xyz_locs):
        """Unit outward surface normals at points xyz_locs [..., 3]: -grad / |grad| of compute_density_grad's
        gradient, pointing toward decreasing density; (0, 0, 0) where the gradient is zero (masked points, empty
        space, points outside the aabb) or not finite. Coordinates as compute_density_grad."""
        shape = xyz_locs.shape[:-1]
        _, nrm = ops.field_density_grad(self._density_factorset(), self._h_geom(), self.density_shift,
                                        0 if self.fea2denseAct == "softplus" else 1, xyz=xyz_locs,
                                        mask=self.alphaMask, normals=True, want_sigma=False)
        return nrm.view(*shape, 3)

    @torch.no_grad()
    def render_normals(self, center, ray_dir, ndc_ray=False, N_samples=-1):
        """Normal map of rays: (normal_map [N,3], depth [N], opacity [N]). normal_map = sum_k w_k n_k over every
        valid sample of the ray, w_k the compositing weights (those whose sum is opacity) and n_k compute_normals at
        the sample (field coordinates: world, or NDC with ndc_ray); it is not renormalised, |normal_map| <= opacity.
        Samples, alpha mask rule (the mask only without a cached blur, batBase.py:76), blur and factor storage are
        those of forward(..., is_train=False) with the same module state, so depth and opacity equal that forward's
        bit for bit. No shading head or appearance stage runs. Each ray's result is independent of the batch."""
        rays_o = center.reshape(-1, 3).detach().contiguous().float()
        rays_d = ray_dir.reshape(-1, 3).detach().contiguous().float()
        ops._need_cuda(rays_o, "center")
        ops._need_cuda(rays_d, "ray_dir")
        n = rays_o.shape[0]
        if n == 0:
            z = torch.zeros((0,), device=rays_o.device)
            return torch.zeros((0, 3), device=rays_o.device), z, z.clone()
        n_samples = N_samples if N_samples > 0 else self.nSamples
        aux = self._ndc_table(n_samples, False).contiguous() if ndc_ray else None
        blur_active = self.c2f_mode is not None
        cfg = RenderCfg(
            n_samples=int(n_samples), ndc=bool(ndc_ray), h_geom=self._h_geom(),
            mask=(self.alphaMask if (self.alphaMask is not None and not blur_active) else None),   # batBase.py:76
            density_shift=float(self.density_shift), act=(0 if self.fea2denseAct == "softplus" else 1),
            distance_scale=float(self.distance_scale), thres=float(self.rayMarch_weight_thres),
            depth_bias=-float(self.near_far[0]) + 0.05)
        dfs = self._density_factorset()
        gather_fs = dfs
        if self._checked_storage() == "bf16":      # forward's density gather reads the bf16 copy
            gather_fs = dfs.with_bf16_store(self._store_cache[0] if not blur_active else None)
        return render_normals(cfg, gather_fs, dfs, rays_o, rays_d, aux)

    @torch.no_grad()
    def raycast(self, center, ray_dir, level=0.005, ndc_ray=False, N_samples=-1, colors=False):
        """First hit of each ray on the surface extract_mesh(level) contours, {compute_alpha(p, stepSize) >= level}
        inside the aabb (jt_raycast): (hit [N] bool, t [N], xyz [N,3], normal [N,3]), plus rgb [N,3] with colors=True.
        The candidates are the sample depths of forward(..., is_train=False) with the same ndc_ray / N_samples; the
        first inside sample is refined to the first crossing between it and the sample before it. t is the ray
        parameter of xyz = center + t * ray_dir (+inf on a miss; not forward's depth_map), xyz the fp32 point known to
        be inside (0 on a miss). normal = compute_normals(xyz) and rgb = compute_rgb(xyz, viewdir) on the hits, 0 on
        misses; viewdir is ray_dir as forward's head sees it (normalised for NDC rays, as given otherwise). Same field
        state as compute_alpha: the density factors blurred with the kernel the last forward cached, the fp32 factors
        whatever factor_storage is, and the alpha mask. Each ray's result is independent of the batch."""
        rays_o = center.reshape(-1, 3).detach().contiguous().float()
        rays_d = ray_dir.reshape(-1, 3).detach().contiguous().float()
        n_samples = N_samples if N_samples > 0 else self.nSamples
        ztab = self._ndc_table(n_samples, False).contiguous() if ndc_ray else None
        t, xyz, _ = ops.raycast(self._density_factorset(), self._h_geom(), self.density_shift,
                                0 if self.fea2denseAct == "softplus" else 1, float(self._h_step), level, rays_o,
                                rays_d, n_samples, ztab=ztab, mask=self.alphaMask)
        hit = torch.isfinite(t)
        # rows are independent in both point queries: evaluate every row (no host sync), keep the hits' rows
        normal = torch.where(hit[:, None], self.compute_normals(xyz), 0.0)
        if not colors:
            return hit, t, xyz, normal
        dirs = rays_d / torch.linalg.vector_norm(rays_d, dim=-1, keepdim=True) if ndc_ray else rays_d
        return hit, t, xyz, normal, torch.where(hit[:, None], self.compute_rgb(xyz, dirs), 0.0)

    # ---------------------------------------------------------------- forward (batBase.py:44-165)
    def forward(self, opt, center, ray_dir, white_bg=True, is_train=False, ndc_ray=False, N_samples=-1,
                c2f_parameter_density=None, c2f_parameter_color=None, c2f_mode=None, c2f_kernel_size=None,
                is_test_optim=False, view_pe_progress=1.0, fea_pe_progress=1.0, jitter=None, bg_coin=None):
        """Returns (rgb_map [N,3], depth_map [N], opacity [N]); differentiable w.r.t.
        the field parameters and `center` / `ray_dir` (joint pose optimisation).

        Extra keyword-only knobs (not in the reference, used by the parity tests):
        `jitter` replaces the stratified-sampling random numbers, `bg_coin`
        replaces the train-time background coin flip `torch.rand((1,)) < 0.5`."""
        self.opt = opt
        self._check_opt(opt)
        self._reg_cache = None        # a new step: the regulariser node of the previous one is stale
        n_samples = N_samples if N_samples > 0 else self.nSamples
        dev = center.device

        blur_active = c2f_parameter_density is not None or c2f_parameter_color is not None
        self.c2f_mode = c2f_mode
        if c2f_mode is not None:
            dmode = "uniform-gaussian" if is_test_optim else c2f_mode
            self.kernel_density = self.get_kernel(opt, dmode, c2f_parameter_density, c2f_kernel_size)
            self.kernel_color = self.get_kernel(opt, c2f_mode, c2f_parameter_color, c2f_kernel_size)
        else:
            self.kernel_density = None
            self.kernel_color = None

        if ndc_ray:
            if opt.camera.ndc_simulate_euclid_sample or opt.camera.ndc_simulate_euclid_depth:
                raise _lib.JtError("ndc_simulate_euclid_* is not supported by the B200 path")
            aux = self._ndc_table(n_samples, is_train and jitter is None)
            if is_train and jitter is not None:
                near, far = float(self.near_far[0]), float(self.near_far[1])
                aux = aux + jitter.reshape(-1).to(aux) * ((far - near) / n_samples)
            aux = aux.contiguous()
        elif is_train:
            aux = jitter if jitter is not None else torch.rand((center.shape[0],), device=dev)
            aux = aux.reshape(-1).contiguous().float()
        else:
            aux = None

        # same short-circuit as batBase.py:154, so the host RNG stream is consumed identically
        white = bool(white_bg or (is_train and (bool(torch.rand((1,)) < 0.5) if bg_coin is None else bool(bg_coin))))

        cfg = RenderCfg(
            n_samples=int(n_samples), ndc=bool(ndc_ray), white_bg=white, h_geom=self._h_geom(),
            h_inv=floats(self._h_inv.tolist()),
            mask=(self.alphaMask if (self.alphaMask is not None and not blur_active) else None),   # batBase.py:76
            density_shift=float(self.density_shift), act=(0 if self.fea2denseAct == "softplus" else 1),
            distance_scale=float(self.distance_scale), thres=float(self.rayMarch_weight_thres),
            depth_bias=-float(self.near_far[0]) + 0.05, fea_prog=float(fea_pe_progress),
            view_prog=float(view_pe_progress), **self._head_fields())

        cfg.grad_sync = self.grad_sync
        cfg.grad_enabled = torch.is_grad_enabled()
        cfg.storage = self._checked_storage()
        if self.app_capacity == "auto" and cfg.grad_enabled:
            cfg.app_cap = self._app_tracker.capacity(center.reshape(-1, 3).shape[0], center.reshape(-1, 3).shape[0] * n_samples)
            cfg.app_monitor = self._app_tracker.submit
        elif isinstance(self.app_capacity, (int, float)) and not isinstance(self.app_capacity, bool):
            cap_all = center.reshape(-1, 3).shape[0] * n_samples
            cfg.app_cap = int(self.app_capacity * cap_all) if self.app_capacity <= 1.0 else int(self.app_capacity)
        cfg.bf16_backward_taps = bool(getattr(self, "bf16_backward_taps", False))
        # the bf16 copies are cached per (storage, version) only for the module's own Parameters: blurred factors
        # are fresh buffers every call (an address + version key could alias a previous step's buffer)
        cfg.store_cache = self._store_cache if self.kernel_density is None and self.kernel_color is None else (None, None)
        dp, dl, ap, al = self._blurred_all(self.kernel_density, self.kernel_color)
        head = self.renderModule.head_params() if self.renderModule is not None else []
        return VMRender.apply(cfg, center.reshape(-1, 3), ray_dir.reshape(-1, 3), aux, *dp, *dl, *ap, *al,
                              self.basis_mat.weight, *head)

    render = forward      # north_star calls the entry point `render`; the reference engine calls forward

    def _head_fields(self):
        """The RenderCfg fields that choose and size the shading head (forward and compute_rgb)."""
        tc = self.head_precision == "tc" or (self.head_precision == "auto" and self.tc_available())
        return dict(shading=self.shadingMode, app_dim=int(self.app_dim), fea_pe=int(self.fea_pe),
                    view_pe=int(self.view_pe), hidden=int(self.featureC), tc_fwd_split=int(self.tc_fwd_split),
                    tc_infer_fp16=bool(self.tc_infer_fp16), head="tc" if tc else "fp32")

    def _checked_storage(self):
        if self.factor_storage not in ("fp32", "bf16"):
            raise _lib.JtError(f"factor_storage {self.factor_storage!r}: expected 'fp32' or 'bf16'")
        return self.factor_storage

    def tc_available(self):
        """True when the tcgen05 shading-head kernels cover this configuration (what head_precision="auto" picks):
        3 x 48 appearance components with app_dim 27 and MLP_Fea (hidden 64, pe 2) or SH shading (Blender configs), or
        3 x 20 components with app_dim 20 and MLP_Fea_WeakView (hidden 32, pe 2) (the LLFF config)."""
        return tc_head(self.shadingMode, int(self.app_dim), int(self.featureC), int(self.fea_pe), int(self.view_pe),
                       self.app_n_comp) is not None

    def _check_opt(self, opt):
        arch = opt.arch
        for f in _OPT_FLAGS:
            if getattr(arch, f, False):
                raise _lib.JtError(f"opt.arch.{f}=True is not implemented by the B200 path (False in all reference configs)")
        if getattr(getattr(opt, "nerf", None), "bbox_cycle_xy", False):
            raise _lib.JtError("opt.nerf.bbox_cycle_xy=True (tensorBase.py:581-608: wrapped x/y sampling) is not "
                               "implemented by the B200 path (absent from every reference config)")
        sh = arch.shading
        if not (sh.detach_viewdirs and sh.detach_xyz):
            raise _lib.JtError("the B200 path implements detach_viewdirs/detach_xyz = True (all reference configs)")
        if getattr(sh, "predict_density", False):
            raise _lib.JtError("shading.predict_density is not implemented by the B200 path")
        self._check_interp(arch.tensorf.grid_sample_interp_mode)
        if self.fea2denseAct not in ("softplus", "relu"):
            raise _lib.JtError(f"fea2denseAct {self.fea2denseAct!r} unsupported")

    # ---------------------------------------------------------------- maintenance (between steps)
    @torch.no_grad()
    def upsample_volume_grid(self, res_target):
        """tensoRF.py:274-295: bilinear align_corners=True resize of every factor (jt_resize_bilinear_cl)."""
        res_target = [int(v) for v in res_target]
        for planes, lines in ((self.app_plane, self.app_line), (self.density_plane, self.density_line)):
            for i in range(3):
                m0, m1 = MAT_MODE[i]
                planes[i] = torch.nn.Parameter(ops.resize_bilinear_cl(planes[i].data, res_target[m1], res_target[m0]))
                lines[i] = torch.nn.Parameter(ops.resize_bilinear_cl(lines[i].data, res_target[VEC_MODE[i]], 1))
        self.update_stepSize(res_target)
        self._reg_cache = None
        self._store_cache = ({}, {})
        self._app_tracker.reset()

    def _dense_tables(self, gridSize):
        return [torch.linspace(0, 1, int(g)).to(self.device) for g in gridSize]

    @torch.no_grad()
    def _dense_alpha_zyx(self, gridSize):
        """alpha on the dense grid in [gz,gy,gx] order, one launch (tensorBase.py:618-633 without the xyz grid)."""
        gridSize = [int(v) for v in gridSize]
        return ops.field_alpha(self._density_factorset(), self._h_geom(), self.density_shift,
                               0 if self.fea2denseAct == "softplus" else 1, float(self._h_step),
                               lin=self._dense_tables(gridSize), grid=gridSize, mask=self.alphaMask)

    @torch.no_grad()
    def getDenseAlpha(self, gridSize=None):
        """tensorBase.py:618-633 -> (alpha [gx,gy,gz], dense_xyz [gx,gy,gz,3])."""
        gridSize = self._grid if gridSize is None else [int(v) for v in gridSize]
        lin = self._dense_tables(gridSize)
        samples = torch.stack(torch.meshgrid(*lin, indexing="ij"), -1)
        dense_xyz = self.aabb[0] * (1 - samples) + self.aabb[1] * samples
        return self._dense_alpha_zyx(gridSize).permute(2, 1, 0), dense_xyz

    @torch.no_grad()
    def extract_mesh(self, level=0.005, gridSize=None, colors=False, normal_source="lattice"):
        """The field's geometry as a triangle mesh: marching cubes (ops.marching_cubes) on the dense alpha grid of
        getDenseAlpha(gridSize) at alpha `level` (0.005 is TensoRF's exporter level). Honours the alpha mask and a
        cached density blur exactly as getDenseAlpha does. Returns (verts [V,3] fp32 world coordinates, faces [F,3]
        int32) on the module's device; normals point out of the high-alpha region.
        colors=True returns (verts, faces, normals, rgb) with the same verts and faces: normals [V,3] point out of the
        high-alpha region, and rgb [V,3] = compute_rgb(verts, -normals), the colour seen looking at the surface
        head-on (a vertex with a zero normal is shaded with a zero view direction). normal_source="lattice" (default):
        the unit gradients of the alpha volume the surface was extracted from (ops.marching_cubes(normals=True));
        "field": compute_normals(verts), the field's own density gradient at each vertex. For an NDC (LLFF) field the
        vertices, normals and view directions are all in the field's NDC coordinates."""
        if normal_source not in ("lattice", "field"):
            raise _lib.JtError(f"extract_mesh: normal_source {normal_source!r}: expected 'lattice' or 'field'")
        gridSize = self._grid if gridSize is None else [int(v) for v in gridSize]
        mesh = ops.marching_cubes(self._dense_alpha_zyx(gridSize), level, self._dense_tables(gridSize), self._h_aabb,
                                  normals=colors and normal_source == "lattice")
        if not colors:
            return mesh
        if normal_source == "field":
            verts, faces = mesh
            normals = self.compute_normals(verts)
        else:
            verts, faces, normals = mesh
        return verts, faces, normals, self.compute_rgb(verts, -normals)

    def export_mesh(self, path, level=0.005, gridSize=None, colors=False, normal_source="lattice"):
        """extract_mesh written to `path` as a binary little-endian PLY (float x, y, z per vertex; `list uchar int
        vertex_indices` per face). colors=True adds `float nx, ny, nz` and `uchar red, green, blue` per vertex (the
        names MeshLab, Blender and Open3D read), colours quantised as floor(clamp(rgb, 0, 1) * 255 + 0.5) in fp32.
        normal_source: as extract_mesh. Returns (V, F)."""
        mesh = self.extract_mesh(level, gridSize, colors=colors, normal_source=normal_source)
        verts, faces = mesh[0], mesh[1]
        v = verts.cpu().numpy().astype("<f4")
        props = "property float x\nproperty float y\nproperty float z\n"
        if colors:
            rgb = np.clip(mesh[3].cpu().numpy(), np.float32(0), np.float32(1))
            vt = np.empty((v.shape[0],), dtype=[("p", "<f4", (3,)), ("n", "<f4", (3,)), ("c", "u1", (3,))])
            vt["p"] = v
            vt["n"] = mesh[2].cpu().numpy()
            vt["c"] = np.floor(rgb * np.float32(255) + np.float32(0.5))
            props += ("property float nx\nproperty float ny\nproperty float nz\n"
                      "property uchar red\nproperty uchar green\nproperty uchar blue\n")
            v = vt
        f = np.empty((faces.shape[0],), dtype=[("n", "u1"), ("i", "<i4", (3,))])
        f["n"] = 3
        f["i"] = faces.cpu().numpy()
        header = ("ply\nformat binary_little_endian 1.0\n"
                  f"element vertex {v.shape[0]}\n{props}"
                  f"element face {f.shape[0]}\nproperty list uchar int vertex_indices\nend_header\n")
        with open(path, "wb") as fh:
            fh.write(header.encode("ascii"))
            fh.write(v.tobytes())
            fh.write(f.tobytes())
        return v.shape[0], f.shape[0]

    @torch.no_grad()
    def updateAlphaMask(self, gridSize=(200, 200, 200)):
        """tensorBase.py:635-661: dense alpha -> clamp -> max_pool3d(5) -> threshold -> mask + new aabb, four
        launches and one 28-byte read-back (the reference synchronises here too: boolean indexing, prints)."""
        gridSize = [int(v) for v in gridSize]
        alpha = self._dense_alpha_zyx(gridSize)
        vol, bits, stats = ops.alpha_mask_build(alpha, self.alphaMask_thres)
        st = stats.tolist()
        if st[6] == 0:
            raise RuntimeError("updateAlphaMask: no voxel reaches alphaMask_thres (the reference fails on the empty "
                               "amin at tensorBase.py:654 as well)")
        self.alphaMask = AlphaGridMask(self.device, self.aabb, vol, packed_bits=bits)
        lin = self._dense_tables(gridSize)
        lo = torch.stack([lin[a][st[2 * a]] for a in range(3)])
        hi = torch.stack([lin[a][st[2 * a + 1]] for a in range(3)])
        # dense_xyz = aabb[0]*(1-s) + aabb[1]*s is monotone per axis: amin/amax of the kept points sit at the
        # extreme kept indices
        return torch.stack((self.aabb[0] * (1 - lo) + self.aabb[1] * lo, self.aabb[0] * (1 - hi) + self.aabb[1] * hi))

    @torch.no_grad()
    def shrink(self, new_aabb):
        """tensoRF.py:297-334: crop every factor to the voxel range covering new_aabb."""
        xyz_min, xyz_max = new_aabb
        t_l = torch.round((xyz_min - self.aabb[0]) / self.units).long()
        b_r = torch.round((xyz_max - self.aabb[0]) / self.units).long() + 1
        b_r = torch.stack([b_r, self.gridSize]).amin(0)
        tl, br = t_l.tolist(), b_r.tolist()
        for i in range(3):
            v = VEC_MODE[i]
            m0, m1 = MAT_MODE[i]
            for lines in (self.density_line, self.app_line):
                lines[i] = torch.nn.Parameter(_to_cl(lines[i].data[..., tl[v]:br[v], :]))
            for planes in (self.density_plane, self.app_plane):
                planes[i] = torch.nn.Parameter(_to_cl(planes[i].data[..., tl[m1]:br[m1], tl[m0]:br[m0]]))
        if not torch.all(self.alphaMask.gridSize == self.gridSize):
            lo, hi = t_l / (self.gridSize - 1), (b_r - 1) / (self.gridSize - 1)
            corrected = torch.zeros_like(new_aabb)
            corrected[0] = (1 - lo) * self.aabb[0] + lo * self.aabb[1]
            corrected[1] = (1 - hi) * self.aabb[0] + hi * self.aabb[1]
            new_aabb = corrected
        self.aabb = new_aabb
        self._reg_cache = None
        self._store_cache = ({}, {})
        self._app_tracker.reset()
        new_size = b_r - t_l
        self.update_stepSize((int(new_size[0]), int(new_size[1]), int(new_size[2])))

    def load_state_dict(self, *a, **kw):
        out = super().load_state_dict(*a, **kw)
        self._store_cache = ({}, {})           # new factor values: bf16 copies and the appearance-count history are stale
        self._app_tracker.reset()
        self._reg_cache = None
        return out

    # ---------------------------------------------------------------- checkpoint side-state (tensorBase.py:508-552)
    def get_reset_kwargs(self):
        return {"aabb": self.aabb, "gridSize": list(self._grid), "density_n_comp": self.density_n_comp,
                "appearance_n_comp": self.app_n_comp, "app_dim": self.app_dim, "density_shift": self.density_shift,
                "alphaMask_thres": self.alphaMask_thres, "distance_scale": self.distance_scale,
                "rayMarch_weight_thres": self.rayMarch_weight_thres, "fea2denseAct": self.fea2denseAct,
                "near_far": self.near_far, "step_ratio": self.step_ratio, "shadingMode": self.shadingMode,
                "pos_pe": self.pos_pe, "view_pe": self.view_pe, "fea_pe": self.fea_pe, "featureC": self.featureC,
                "volume_init_scale": self.volume_init_scale, "volume_init_bias": self.volume_init_bias}

    def save_param_state(self):
        ckpt = {"tensorf_reset_kwargs": self.get_reset_kwargs()}
        if self.alphaMask is not None:
            vol = self.alphaMask.alpha_volume.bool().cpu().numpy()
            ckpt.update({"alphaMask.shape": vol.shape, "alphaMask.mask": np.packbits(vol.reshape(-1)),
                         "alphaMask.aabb": self.alphaMask.aabb.cpu()})
        return ckpt

    def load_param_state(self, ckpt):
        if "alphaMask.aabb" in ckpt.keys():
            length = np.prod(ckpt["alphaMask.shape"])
            vol = torch.from_numpy(np.unpackbits(ckpt["alphaMask.mask"])[:length].reshape(ckpt["alphaMask.shape"]))
            self.alphaMask = AlphaGridMask(self.device, ckpt["alphaMask.aabb"].to(self.device), vol.float().to(self.device))
        self.reset(**ckpt["tensorf_reset_kwargs"])


def _to_cl(x):
    """Force channel-last physical layout ([H][W][C]) for a [1,C,H,W] tensor, also for
    degenerate shapes where torch's channels_last stride check is ambiguous."""
    n, c, h, w = x.shape
    buf = x.permute(0, 2, 3, 1).contiguous()
    return buf.permute(0, 3, 1, 2)
