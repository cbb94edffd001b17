#!/usr/bin/env python
"""bench.py -- rays/s forward+backward of the TensoRF-VM render hot path.

    python bench.py --gpus N --steps K --warmup W            (own arm, B200 kernels)
    python bench.py --impl reference --gpus N ...            (reference arm: CPU port)
    python bench.py ... --dump-outputs DIR                   (+ the last timed step's outputs as DIR/*.npy)

Workload (BASELINE.json configs[1], "cfg2_sh"): TensoRF-VM 300^3 grid, density 3x16 /
appearance 3x48 components, app_dim 27, SH shading, 4096-ray batch, S=1000 samples per
ray, forward + backward to all factor / basis / ray gradients. Synthetic Blender-shaped
rays and random-init factors (joint_tensorf_b200.synth). The same field with the
MLP_Fea shading head (`--workload cfg2`, the head of the BAT VM_MLP configs) is timed in
the same run and reported under "also".

A step = one training iteration without the optimizer (SURVEY.md section 8d timing
protocol): se3_refine + fixed poses -> rays of the sampled pixels (jt_pose_rays_fwd) ->
stratified jitter -> forward -> MSE -> backward to all factor / head / se3_refine
gradients (+ one NCCL all-reduce of the flat gradient bucket when N > 1).
N > 1 is weak scaling: every rank renders its own 4096 rays.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "rays/sec fwd+bwd (300^3 VM, 4096-ray batch)"
UNIT = "rays/s"
RENDER_METRIC = "ms per 800x800 frame (300^3 VM field, image-sharded full-frame inference)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2_sh",
                    help="cfg2_sh = BASELINE.json configs[1] (300^3, 3x16 / 3x48 comps, app_dim 27, SH shading); "
                         "cfg2 = same field with the MLP_Fea head; cfg1 = 128^3; cfg4 = LLFF NDC 617x687x617")
    ap.add_argument("--no-also", action="store_true",
                    help="skip the second head variant of the 300^3 field (cfg2 <-> cfg2_sh) timed after the headline")
    ap.add_argument("--rays", type=int, default=4096)
    ap.add_argument("--blur", type=float, default=0.0, help="c2f blur parameter (0 = off, cfg3 uses 0.15)")
    ap.add_argument("--cpu-rays", type=int, default=0,
                    help="rays per step of the CPU reference / cpu_baseline legs (0 = the full --rays batch)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = --rays per GPU, strong = --rays in total, sharded over the ranks (SURVEY 8e)")
    ap.add_argument("--mode", default="train", choices=["train", "render"],
                    help="render = BASELINE configs[4]: --frames full 800x800 frames, image-sharded over the ranks, ms/frame")
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--nccl-max-ctas", type=int, default=0,
                    help="N > 1: cap the CTAs NCCL may use (NCCL_MAX_CTAS) so the collectives leave SMs to the kernels "
                         "they overlap with (0 = NCCL's default)")
    ap.add_argument("--cuda-graph", action="store_true",
                    help="capture the step (pose -> rays -> forward -> loss -> backward [-> all-reduce]) into a CUDA graph "
                         "and replay it: removes the ~1.4 ms of host launch time that bounds small / strong-scaled batches")
    ap.add_argument("--sync-per-plane", action="store_true", help="N > 1: one scatter launch + all-reduce per appearance plane")
    ap.add_argument("--sync-split21", default="auto", choices=["auto", "on", "off"],
                    help="N > 1: appearance planes 0+1 | plane 2 | density, a collective after each launch (auto: 4+ ranks "
                         "and an appearance-dominated gradient bucket)")
    ap.add_argument("--sync-reserve-sms", type=int, default=0,
                    help="N > 1: SMs the density scatter leaves free for the all-reduce running next to it")
    ap.add_argument("--storage", default="fp32", choices=["fp32", "bf16"],
                    help="VM factor storage the gathers read (fp32 master parameters either way)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-breakdown", action="store_true")
    ap.add_argument("--no-render", action="store_true", help="skip the 800x800 full-frame inference timing")
    ap.add_argument("--render-chunk", type=int, default=16384, help="rays per forward call of the full-frame render")
    ap.add_argument("--head", default="auto", choices=["auto", "tc", "fp32"],
                    help="shading head: tcgen05 tensor-core kernels (auto/tc) or strict-fp32 SIMT GEMMs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed training step computed (rgb, depth, acc, "
                         "loss and every gradient, rank 0) as DIR/<name>.npy; arrays over 2^21 elements are replaced by "
                         "a fixed seeded sample of that many elements (<name>.sample.npy). Same arguments, same inputs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "b200" or a.mode != "train"):
        ap.error("--dump-outputs writes the outputs of the training step of --impl b200 --mode train")
    return a


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock + throttle reasons sampled (NVML, nvidia-smi as fallback) while the timed regions run."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], False
        self.t = threading.Thread(target=self.run, daemon=True)
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # honour CUDA_VISIBLE_DEVICES remapping via the PCI bus id of the torch device
            bus = torch.cuda.get_device_properties(index).pci_bus_id if hasattr(torch.cuda.get_device_properties(index), "pci_bus_id") else None
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            if bus is not None:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    h = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if int(pynvml.nvmlDeviceGetPciInfo(h).bus) == int(bus):
                        self.h = h
                        break
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def sample_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM)
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        flags = []
        for name, bit in (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
                          ("sw_power_cap", 0x4)):
            flags.append("Active" if (r & bit) else "Not Active")
        return [str(sm), str(mx), "0"] + flags

    def run(self):
        while not self.stop:
            try:
                if self.nvml is not None:
                    self.rows.append(self.sample_nvml())
                else:
                    out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                    self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.005 if self.nvml is not None else 0.1)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ----------------------------------------------------------------------------- CPU port (oracle) timing
def oracle_field(workload, seed=0):
    from joint_tensorf_b200 import synth
    from oracle import vm_oracle as vo
    kw, run = synth.config(workload)
    params = vo.init_params(kw["gridSize"], kw["density_n_comp"], kw["appearance_n_comp"], kw["app_dim"],
                            kw["shadingMode"], kw["featureC"], kw["view_pe"], kw["fea_pe"],
                            kw["volume_init_scale"], kw["volume_init_bias"], seed=seed)
    for v in params.values():
        v.requires_grad_(True)
    field = vo.Field(aabb=torch.tensor(kw["aabb"]), grid=kw["gridSize"], params=params, near_far=kw["near_far"],
                     step_ratio=kw["step_ratio"], density_shift=float(kw["density_shift"]),
                     distance_scale=kw["distance_scale"], weight_thres=kw["rayMarch_weight_thres"],
                     act=kw["fea2denseAct"], shading=kw["shadingMode"], view_pe=kw["view_pe"], fea_pe=kw["fea_pe"])
    return field, run


def time_cpu_port(workload, n_rays, steps, warmup, blur):
    """Reference algorithm (oracle port, same ATen CPU operators as the reference) on
    the host cores: forward + MSE + backward on a bounded sample of the workload."""
    from joint_tensorf_b200 import synth
    from oracle import vm_oracle as vo
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    field, run = oracle_field(workload)
    o, d, _ = synth.blender_rays(n_rays, max(1, min(32, n_rays // 16)), seed=1)
    target = torch.rand(n_rays, 3, generator=torch.Generator().manual_seed(2))
    kw = dict(n_samples=run["n_samples"], white_bg=run["white_bg"], ndc=run["ndc"])
    if blur > 0:
        kw.update(blur_mode="uniform-gaussian", blur_density=blur * 0.6, blur_color=blur, kernel_size=64)
    times = []
    for it in range(warmup + steps):
        oc, dc = o.clone().requires_grad_(True), d.clone().requires_grad_(True)
        jit = torch.rand(n_rays, 1)
        for p in field.params.values():
            p.grad = None
        t0 = time.perf_counter()
        rgb, _, _ = vo.render(field, oc, dc, jitter=jit, **kw)
        loss = ((rgb - target) ** 2).mean()
        loss.backward()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    sec = sum(times) / len(times)
    return n_rays / sec, sec, cores


def time_aten_gpu(workload, n_rays, steps, warmup, dev):
    """Same-box bar (SURVEY 8d): the reference ALGORITHM with stock ATen CUDA operators on this B200 -- the oracle
    port run with its tensors on the device (grid_sample / cumprod / addmm kernels, autograd backward). This is
    what the unmodified reference would execute on a GPU; reported next to the CPU baseline, never shipped."""
    from joint_tensorf_b200 import synth
    from oracle import vm_oracle as vo
    field, run = oracle_field(workload)
    field.params = {k: v.detach().to(dev).requires_grad_(True) for k, v in field.params.items()}
    field.aabb = field.aabb.to(dev)
    o, d, _ = synth.blender_rays(n_rays, 32, seed=1)
    o, d = o.to(dev), d.to(dev)
    target = torch.rand(n_rays, 3, generator=torch.Generator().manual_seed(2)).to(dev)
    kw = dict(n_samples=run["n_samples"], white_bg=run["white_bg"], ndc=run["ndc"])
    times = []
    with torch.device(dev):
        for it in range(warmup + steps):
            oc, dc = o.clone().requires_grad_(True), d.clone().requires_grad_(True)
            jit = torch.rand(n_rays, 1)
            for p in field.params.values():
                p.grad = None
            torch.cuda.synchronize()
            s_ev, e_ev = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s_ev.record()
            rgb, _, _ = vo.render(field, oc, dc, jitter=jit, **kw)
            loss = ((rgb - target) ** 2).mean()
            loss.backward()
            e_ev.record()
            torch.cuda.synchronize()
            if it >= warmup:
                times.append(s_ev.elapsed_time(e_ev) * 1e-3)
    sec = sum(times) / len(times)
    return n_rays / sec, sec


def cfg_head(model):
    """"tc" when the module will pick the tcgen05 head for its configuration, else "fp32"."""
    hp = model.head_precision
    if hp == "fp32":
        return "fp32"
    return "tc" if (hp == "tc" or model.tc_available()) else "fp32"


def synth_describe(workload, n_rays=None):
    from joint_tensorf_b200 import synth
    return synth.describe(workload, n_rays)


def time_cpu_reference(workload, n_rays, steps, warmup, blur, budget_s=240.0):
    """The reference on the host cores: the UNMODIFIED `BAT_VMSplit` when its files are present (/root/reference in
    the build container, the staged oracle/_ref on the GPU box: kind "reference"), else the oracle restatement
    (kind "port"). Returns a dict with rays/s, seconds per step, cores, steps done and the kind."""
    from oracle import reference_arm as ra
    if ra.root() is not None:
        rps, sec, cores, done, warm = ra.time_reference(workload, n_rays, steps, warmup, blur, budget_s)
        return dict(rps=rps, sec=sec, cores=cores, steps=done, warmup=warm, kind="reference",
                    what="unmodified reference BAT_VMSplit.forward + backward (model/tensorf_repr/batBase.py:44-165), "
                         f"torch CPU, {cores} threads" +
                         ("; SHRender called through a 5->3 argument wrapper (the reference's own call site "
                          "crashes, SURVEY B-1)" if workload.endswith("_sh") else ""))
    rps, sec, cores = time_cpu_port(workload, n_rays, steps, warmup, blur)
    return dict(rps=rps, sec=sec, cores=cores, steps=steps, warmup=warmup, kind="port",
                what=f"oracle/vm_oracle.py restatement (same ATen CPU operators as the reference), {cores} threads")


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.mode == "render":
        return reference_render_arm(args)
    n = args.cpu_rays or args.rays
    # every step is the full ray batch (~8 s on 16 threads at cfg2_sh): the run stops early when 4 minutes are spent
    r = time_cpu_reference(args.workload, n, max(1, args.steps), max(0, args.warmup), args.blur, budget_s=240.0)
    rps = r["rps"]
    line = {
        "impl": "reference", "metric": METRIC, "value": rps, "unit": UNIT, "n_gpus": args.gpus, "steps": r["steps"],
        "warmup": r["warmup"], "ms_per_step": r["sec"] * 1e3, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": synth_describe(args.workload) + f", {n}-ray batch, fwd+bwd", "blur": args.blur,
                   "note": "rays resident, no pose generation, optimizer step excluded; steps stop at a 240 s budget"},
        "cpu_baseline": {"value": rps, "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                         "sample": f"{n} rays per step (the full batch), {r['steps']} timed steps after {r['warmup']} "
                                   f"warm-up: {r['what']}"},
        "e2e": {"value": rps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def reference_render_arm(args):
    """configs[4] on the host cores: a bounded sample (16384 rays of one 800x800 frame, no-grad forward of the
    unmodified reference / the port), extrapolated to ms per full frame and labelled as such (SURVEY 8d)."""
    from joint_tensorf_b200 import synth
    from oracle import reference_arm as ra
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    n = 16384
    o, d = synth.frame_rays(0)
    sel = torch.randperm(o.shape[0], generator=torch.Generator().manual_seed(0))[:n]
    o, d = o[sel].contiguous(), d[sel].contiguous()
    kw, run = synth.config(args.workload)
    kind = "reference" if ra.root() is not None else "port"
    if kind == "reference":
        import contextlib
        import io
        m, opt, run = ra.build_field(args.workload)

        def fwd():
            with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
                return m.forward(opt, o, d, white_bg=run["white_bg"], is_train=False, ndc_ray=run["ndc"],
                                 N_samples=run["n_samples"])[0]
    else:
        from oracle import vm_oracle as vo
        field, run = oracle_field(args.workload)

        def fwd():
            with torch.no_grad():
                return vo.render(field, o, d, n_samples=run["n_samples"], white_bg=run["white_bg"], ndc=run["ndc"])[0]
    fwd()
    t0 = time.perf_counter()
    reps = 2
    for _ in range(reps):
        fwd()
    sec = (time.perf_counter() - t0) / reps
    ms_frame = sec * (800 * 800 / n) * 1e3
    line = {"impl": "reference", "metric": RENDER_METRIC, "value": ms_frame, "unit": "ms/frame", "n_gpus": args.gpus,
            "steps": reps, "warmup": 1, "ms_per_step": sec * 1e3, "higher_is_better": False, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": synth_describe(args.workload) + ", 800x800 full-frame inference",
                       "note": f"EXTRAPOLATED from {n} rays of one frame (a full frame is ~20 min of host time)"},
            "cpu_baseline": {"value": ms_frame, "unit": "ms/frame", "cores": cores, "kind": kind,
                             "sample": f"{n} of 640000 rays, {reps} timed no-grad forwards, extrapolated x{800 * 800 / n:.1f}"},
            "e2e": {"value": ms_frame, "unit": "ms/frame", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- own arm
def logical_bytes(name, V, A, cd, ca, ctot_a):
    """SURVEY.md section 8(d)'s LOGICAL figure: every tap counted as an HBM access (fp32 factors). Kept for
    reference only -- the factors live in L2 and cells are shared along a ray, so this is not a roofline."""
    s = 4
    dens_f = V * (18 * cd * s + 16)
    app_fused = A * (18 * ca * s + 12)
    table = {
        "vm_density_fwd": dens_f, "vm_app_fwd": A * (18 * ca * s + 12 + 4 * ctot_a),
        "app_basis_fwd_tc": app_fused + A * 128, "app_basis_sh_fwd_tc": app_fused + A * 32,
        "vm_density_bwd": V * (3 * 18 * cd * s + 4 + 16), "vm_app_bwd": A * (3 * 18 * ca * s + 4 * ctot_a + 16),
    }
    return table.get(name)


def compulsory_bytes(name, V, A, fbytes_d, fbytes_a, gbytes_d, gbytes_a, ctot_a, gin_bytes, train=True):
    """HBM bytes the IMPLEMENTATION's data flow cannot avoid, per launch (DESIGN.md section 4): the per-sample streams
    (sample records 16 B + index 4 B (+ appearance slot 4 B), upstream gradients, staged operand tiles), ONE read of
    the factor set the kernel gathers from (fbytes_*: its bytes as stored, fp32 or bf16) and ONE write-back of the
    gradient planes it reduces into (gbytes_*, fp32; the REDs resolve in L2). Everything a kernel moves beyond this
    (`traffic` from ncu) is re-reads caused by L2 overflow."""
    rec_v, rec_a = 16 + 4, 16 + 4 + 4
    table = {
        "vm_density_fwd": V * (rec_v + 4) + fbytes_d,
        "vm_density_bwd": V * (rec_v + 4) + fbytes_d + gbytes_d,
        "vm_app_fwd": A * (rec_a + 4 * ctot_a) + fbytes_a,
        "vm_app_bwd": A * (rec_a + gin_bytes * ctot_a) + fbytes_a + gbytes_a,
        # gather + basis_mat (+ SHRender): records in, rgb + view direction (SH) or the 128-byte feat/dir row out,
        # + the bf16 component tile staged for the basis_mat weight gradient when training
        "app_basis_sh_fwd_tc": A * (rec_a + 32 + (2 * ctot_a if train else 0)) + fbytes_a,
        "app_basis_fwd_tc": A * (rec_a + 128 + (2 * ctot_a if train else 0)) + fbytes_a,
        # SH backward: dpre + direction in, bf16 dcomps + the DF tile out; weight-gradient kernel reads both tiles
        "sh_bwd_tc": A * (32 + 2 * ctot_a + 64) + A * (2 * ctot_a + 64),
        "head_mlp_fwd_tc": A * (128 + 16 + (320 + 160 + 160 if train else 0)),
        # data kernel: dout + feat row + the relu-mask halves of A2 / A3 in, D2 / D1 / DF / DO tiles + dcomps out;
        # weight-gradient kernel: all eight staged tiles (1264 B per sample, head_tc.cuh) in
        "head_bwd_tc": A * (16 + 128 + 256 + 336 + gin_bytes * ctot_a + 1264),
        # LLFF head: components in (4 B x sum C), feat/dir row + rgb out, 752 B of staged tiles when training;
        # backward: dout + feat row + mask halves in, D tiles + fp32 dcomps out, weight-gradient kernel reads all tiles
        "wv_head_fwd_tc": A * (4 * ctot_a + 128 + 16 + (544 if train else 0)),
        "wv_head_bwd_tc": A * (16 + 128 + 128 + 208 + 4 * ctot_a + 752),
        "alpha_fwd": V * (4 + 4 + 16 + 8 + 8), "render_bwd": V * (4 + 4 + 8 + 4 + 16 + 16 + 4),
        "composite_fwd": A * (4 + 4 + 16),
    }
    return table.get(name)


def l1_fill_bytes(name, V, A, cd, ca, s_d, s_a):
    """The binding unit of the gather / scatter kernels is not HBM but the SM's L1 data pipe (ncu:
    l1tex__data_pipe_lsu_wavefronts 66-71 % of peak on these kernels, 128 B per clock per SM): bytes that must cross
    it per launch in the current design = every tap of every sample delivered to registers once (fp32 or bf16 as
    stored) (+ the same volume again as REDs and staging copies in the scatter, not counted here)."""
    table = {
        "vm_density_fwd": V * 18 * cd * s_d, "vm_density_bwd": V * 18 * cd * s_d,
        "vm_app_fwd": A * 18 * ca * s_a, "app_basis_fwd_tc": A * 18 * ca * s_a, "app_basis_sh_fwd_tc": A * 18 * ca * s_a,
        "vm_app_bwd": A * 18 * ca * s_a,
    }
    return table.get(name)


# timer span (ops.TIMER) -> the kernel functions launched inside it, for the ncu look-up
SPAN_KERNELS = {
    "vm_app_bwd": ["vm_scatter_walk_kernel<1"], "vm_density_bwd": ["vm_scatter_walk_kernel<0"],
    "vm_density_fwd": ["vm_fwd_kernel<0"], "vm_app_fwd": ["vm_fwd_kernel<1"],
    "app_basis_sh_fwd_tc": ["app_basis_fwd_kernel"], "app_basis_fwd_tc": ["app_basis_fwd_kernel"],
    "sh_bwd_tc": ["sh_bwd_data_kernel", "head_bwd_wgrad_kernel"], "head_mlp_fwd_tc": ["head_mlp_fwd_kernel"],
    "head_bwd_tc": ["head_bwd_data_kernel", "head_bwd_wgrad_kernel"], "alpha_fwd": ["alpha_fwd_kernel", "app_fill_kernel"],
    "wv_head_fwd_tc": ["wv::wv_head_fwd_kernel"], "wv_head_bwd_tc": ["wv::wv_head_bwd_data_kernel", "wv::wv_head_bwd_wgrad_kernel"],
    "render_bwd": ["render_bwd_kernel"], "composite_fwd": ["composite_fwd_kernel"],
}


def ncu_lookup(span, workload, storage):
    """dram bytes (read + write) and L1 data-pipe utilisation of the kernels of `span` from the committed
    `ncu --set full` capture of THIS workload (profiles/ncu_kernels.json, written by scripts/ncu_summary.py --json
    from the .ncu-rep of the same code; its `commit` field says which). None when no capture matches."""
    try:
        db = json.load(open(os.path.join(ROOT, "profiles", "ncu_kernels.json")))
    except Exception:
        return None
    cap = db.get(f"{workload}:{storage}")
    if not cap:
        return None
    tot, l1, found = 0.0, [], []
    for pat in SPAN_KERNELS.get(span, []):
        hit = [k for k in cap["kernels"] if k["name"].replace("void ", "").startswith(pat)]
        if not hit:
            return None
        k = hit[0]
        tot += k["dram_read"] + k["dram_write"]
        l1.append(k.get("l1_lsu_wavefront_pct"))
        found.append(k["name"][:60])
    return {"traffic": tot, "l1_data_pipe_pct_ncu": l1[0] if l1 else None, "kernels": found,
            "capture": cap.get("file"), "commit": cap.get("commit")}


def gemm_flops(name, A, F, ctot, in_dim, H):
    table = {
        "basis_fwd": 2 * A * F * ctot, "basis_bwd_x": 2 * A * F * ctot, "basis_bwd_w": 2 * A * F * ctot,
        "mlp_l1_fwd": 2 * A * in_dim * H, "mlp_l1_bwd_x": 2 * A * in_dim * H, "mlp_l1_bwd_w": 2 * A * in_dim * H,
        "mlp_l2_fwd": 2 * A * H * H, "mlp_l2_bwd_x": 2 * A * H * H, "mlp_l2_bwd_w": 2 * A * H * H,
        "mlp_l3_fwd": 2 * A * H * 3, "mlp_l3_bwd_x": 2 * A * H * 3, "mlp_l3_bwd_w": 2 * A * H * 3,
        # fused tensor-core head: basis + 3 layers forward; data + weight gradients backward
        "head_fwd_tc": 2 * A * (F * ctot + in_dim * H + H * H + H * 3),
        "head_bwd_tc": 4 * A * (F * ctot + in_dim * H + H * H + H * 3),
        "head_mlp_fwd_tc": 2 * A * (in_dim * H + H * H + H * 3),
        "sh_bwd_tc": 4 * A * F * ctot,
    }
    return table.get(name)


DUMP_MAX_ELEMS = 1 << 21          # per array: 8 MB of float32
DUMP_MAX_BYTES = 64 << 20         # per dump


def dump_outputs(out_dir, arrays):
    """Write every tensor of `arrays` as out_dir/<name>.npy (float64 stays float64, anything else becomes float32). A
    tensor of more than DUMP_MAX_ELEMS elements is written as <name>.sample.npy instead: its elements at
    DUMP_MAX_ELEMS flat indices drawn from a generator seeded with 0, in increasing order -- the same indices for
    every run and every build, so two dumps compare element for element."""
    import numpy as np
    arrays = {k: (v.detach() if v.dtype == torch.float64 else v.detach().float()) for k, v in arrays.items()}
    size = sum(min(v.numel(), DUMP_MAX_ELEMS) * v.element_size() for v in arrays.values())
    if size > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {size} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        if v.numel() > DUMP_MAX_ELEMS:
            idx = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMS].sort().values
            v, name = v.reshape(-1)[idx.to(v.device)], name + ".sample"
        np.save(os.path.join(out_dir, name + ".npy"), v.cpu().numpy())


def own_arm(args):
    import torch.distributed as dist

    import joint_tensorf_b200 as jt
    from joint_tensorf_b200 import ops, parallel

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if args.nccl_max_ctas > 0:
            os.environ["NCCL_MAX_CTAS"] = str(args.nccl_max_ctas)
        dist.init_process_group("nccl", device_id=dev)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    tf_peak = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "measured" if peaks else "fallback"

    kw, run = jt.synth.config(args.workload)
    kw = dict(kw)
    torch.manual_seed(0)                       # identical replicas on every rank
    model = jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), dev, **kw)
    from joint_tensorf_b200.options import default_opt
    model.head_precision = args.head
    model.factor_storage = args.storage
    opt = default_opt(model.shadingMode, run["ndc"])
    # weak scaling: --rays per GPU; strong scaling: --rays in total, a contiguous 1/world slice per rank (SURVEY 8e)
    N, S = (args.rays // world if args.scaling == "strong" else args.rays), run["n_samples"]
    # Pose side of the step (SURVEY 8d protocol): 32 hemisphere views, pose noise N(0, 0.15^2) composed into the
    # fixed pose (bat.py:34,346-348), se3_refine = 0 and trainable (bat.py:350), 128 pixels shared by all views
    # (nerf.py:657-658) -> N = 4096 rays generated by jt_pose_rays_fwd, gradients back to se3_refine.
    # LLFF (cfg4): 8 forward-facing views = small rigid motions of the identity, 1008x756, focal 0.85 W, rays
    # converted to NDC (camera.py:303-340) inside the same kernel.
    ndc = bool(run["ndc"])
    n_views = 8 if ndc else 32
    H_img, W_img = (756, 1008) if ndc else (800, 800)
    R_pix = max(1, N // n_views)
    N = n_views * R_pix
    if ndc:
        gt_pose, intr = jt.synth.llff_views(n_views, (H_img, W_img), seed=1 + rank)
        base_pose = gt_pose.to(dev)
    else:
        gt_pose, intr = jt.synth.blender_views(n_views, (H_img, W_img), seed=1 + rank)
        g_noise = torch.Generator().manual_seed(50 + rank)
        pose_noise = 0.15 * torch.randn((n_views, 6), generator=g_noise)
        base_pose = jt.camera.refined_pose(pose_noise.to(dev), gt_pose.to(dev))
    intr_inv_d = intr.inverse().to(dev)
    intr_d = intr.to(dev) if ndc else None       # convert_NDC reads the focal length / principal point
    se3_refine = torch.nn.Parameter(torch.zeros((n_views, 6), device=dev))
    cam_opt = jt.options.Namespace(H=H_img, W=W_img, camera=dict(model="perspective", ndc=ndc),
                                   arch=dict(ndc_near_plane=1.0) if ndc else dict())
    pix_h = torch.randperm(H_img * W_img, generator=torch.Generator().manual_seed(7 + rank))[:R_pix].to(torch.int32)
    tgt_h = torch.rand(N, 3, generator=torch.Generator().manual_seed(100 + rank))
    pix_h, tgt_h = pix_h.pin_memory(), tgt_h.pin_memory()
    pix_d, tgt_d = pix_h.to(dev), tgt_h.to(dev)
    loss_h = torch.empty((), pin_memory=True)
    fkw = dict(white_bg=run["white_bg"], is_train=True, ndc_ray=run["ndc"], N_samples=S)
    if args.blur > 0:
        fkw.update(c2f_mode="uniform-gaussian", c2f_parameter_density=args.blur * 0.6,
                   c2f_parameter_color=args.blur, c2f_kernel_size=64)
    params = [p for p in model.parameters()] + [se3_refine]
    # data parallel: the render node's backward reduces its flat gradient bucket across ranks itself (appearance
    # part overlapped with the density scatter); the loss carries the 1/world factor, so the sums are means
    sync = (parallel.OverlappedGradSync(per_plane=args.sync_per_plane, reserve_sms=args.sync_reserve_sms,
                                        split21={"auto": "auto", "on": True, "off": False}[args.sync_split21])
            .attach(model, [se3_refine]) if world > 1 else None)
    inv_world = 1.0 / world
    last_out = {}              # --dump-outputs: the latest step's forward outputs (static tensors under --cuda-graph)

    def make_step(model, opt, params):
        def step(pix, tgt, reduce=True):
            for p in params:
                p.grad = None
            model.grad_sync = sync if reduce else None
            center, ray = jt.camera.get_center_and_ray(cam_opt, base_pose, intr_inv_d, ray_idx=pix, intr=intr_d,
                                                       se3_refine=se3_refine)
            rgb, depth, acc = model(opt, center.view(-1, 3), ray.view(-1, 3), **fkw)
            loss = ((rgb - tgt) ** 2).mean()
            (loss * inv_world if world > 1 else loss).backward()
            if sync is not None and reduce:
                sync.finish([se3_refine])
            if args.dump_outputs:
                last_out.update(rgb=rgb.detach(), depth=depth.detach(), acc=acc.detach(), loss=loss.detach())
            return loss
        return step

    step = make_step(model, opt, params)
    eager_step = step
    launches_per_graph = None
    if args.cuda_graph:
        # the whole step as ONE graph launch: static input buffers refreshed in place, static loss / gradients
        model.app_capacity = None                    # the automatic capacity tracker polls events: not capturable
        pix_s, tgt_s = pix_d.clone(), tgt_d.clone()
        lc0 = jt._lib.launch_count()
        graphed = jt.graphs.GraphedStep(lambda: eager_step(pix_s, tgt_s), warmup=3)
        launches_per_graph = (jt._lib.launch_count() - lc0) // 4       # 3 warm-up calls + the capture

        def step(pix, tgt, reduce=True):
            if not reduce:
                return eager_step(pix, tgt, reduce=False)
            if pix is not pix_s:
                pix_s.copy_(pix, non_blocking=True)
                tgt_s.copy_(tgt, non_blocking=True)
            return graphed()

    def step_e2e():
        pix = pix_h.to(dev, non_blocking=True)
        t = tgt_h.to(dev, non_blocking=True)
        loss = step(pix, t)
        loss_h.copy_(loss.detach(), non_blocking=True)

    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)          # > 126 MB L2

    def timed(fn, k, align=False):
        """Sum of the K per-step device times (CUDA events on the launching stream). The L2
        flush between steps is on the stream but outside every event pair; the host does not
        synchronise inside the loop, so it queues launches ahead as a training loop does."""
        evs = []
        t_host = time.perf_counter()
        # The timed region starts right after a device synchronize: without queued work the GPU would execute the
        # first step's ~45 launches as fast as the host can issue them (3.2 ms instead of 2.7 ms, `step_ms_rank0` of
        # profiles/r01_bench_v15.json). A few extra untimed L2-flush writes give the host the head start it has in
        # every later step; nothing inside an event pair changes.
        for _ in range(6):
            flush.fill_(1.0)
        if world > 1 and align:      # (collective: only where every rank calls timed(), never in rank-0-only sections)
            # device-side rendezvous in front of the first timed step: the hosts reach this point a few ms apart
            # (thread start-up, GC), and without it rank 0's first gradient all-reduce waits for the last rank to
            # arrive -- 6.85 ms instead of 3.2 ms for the first of the 20 steps in SCALE_r01 at N = 8. The hosts keep
            # queueing the first step while the streams wait here, as they do in front of every later step.
            dist.all_reduce(tok)
        for _ in range(k):
            flush.fill_(1.0)                                           # evict L2 between steps (untimed)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            evs.append((s, e))
        timed.host_ms = (time.perf_counter() - t_host) * 1e3 / k      # host time to ENQUEUE a step (launch-bound check)
        torch.cuda.synchronize()
        timed.per_step = [round(s.elapsed_time(e), 3) for s, e in evs]
        return sum(s.elapsed_time(e) for s, e in evs)

    tok = torch.zeros(1, device=dev)

    def barrier():
        """Host barrier + device synchronize (the contract's bracket), then -- multi-GPU only -- a one-element
        all-reduce left on the stream: a DEVICE-side rendezvous, so that the ranks' first timed step starts together
        even though their hosts leave dist.barrier() a few ms apart (measured at N=8: the first timed step took
        7.8 ms instead of 3.65 ms because rank 0 waited for the last host inside its first gradient all-reduce)."""
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if world > 1:
            dist.all_reduce(tok)

    for _ in range(max(args.warmup, 3)):
        step(pix_d, tgt_d)
    barrier()
    for _ in range(2):
        step_e2e()
    barrier()
    l0 = jt._lib.launch_count()
    with ClockSampler(local) as clk:             # clocks are sampled across both timed regions
        ms = timed(lambda: step(pix_d, tgt_d), args.steps, align=True)
        host_ms, per_step = timed.host_ms, timed.per_step
        barrier()
        launches = jt._lib.launch_count() - l0
        if launches_per_graph is not None:
            launches = launches_per_graph * args.steps               # replayed, not re-issued: count what the graph holds
        ms_e2e = timed(step_e2e, args.steps, align=True)
        barrier()
    if args.dump_outputs and rank == 0:
        grads = {f"grad.{k}": p.grad for k, p in model.named_parameters() if p.grad is not None}
        dump_outputs(args.dump_outputs, {**last_out, **grads, "grad.se3_refine": se3_refine.grad})
    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])

    ddp_breakdown = None
    if world > 1:
        # where the data-parallel step spends its time: rank 0 records CUDA events around every C-ABI call and the
        # gradient-synchronisation waits while ALL ranks run the same reduced steps (events do not synchronise)
        ops.TIMER.enabled = rank == 0
        for _ in range(2):
            step(pix_d, tgt_d)
        if rank == 0:
            ops.TIMER.summary()
        reps = 5
        for _ in range(reps):
            flush.fill_(1.0)
            step(pix_d, tgt_d)
        if rank == 0:
            ddp_breakdown = {k: round(v[0] / reps, 4) for k, v in sorted(ops.TIMER.summary().items(), key=lambda kv: -kv[1][0])}
        ops.TIMER.enabled = False
        barrier()
    roof, breakdown = None, None
    if rank == 0 and not args.no_breakdown:
        ops.TIMER.enabled = True                 # rank-0-only section: no collectives in here
        for _ in range(3):
            step(pix_d, tgt_d, reduce=False)
        ops.TIMER.summary()
        reps = 5
        for _ in range(reps):
            flush.fill_(1.0)
            step(pix_d, tgt_d, reduce=False)
        summ = ops.TIMER.summary()
        ops.TIMER.enabled = False
        V, A = (int(t.item()) for t in jt.VMRender.last_counts)      # measured on the last step's batch
        breakdown = {k: round(v[0] / reps, 4) for k, v in sorted(summ.items(), key=lambda kv: -kv[1][0])}
        cd, ca = model.density_n_comp[0], model.app_n_comp[0]
        ctot_a = sum(model.app_n_comp)
        F_, H_ = model.app_dim, model.featureC
        in_dim = F_ + 3 + 2 * model.fea_pe * F_ + 6 * model.view_pe
        s_el = 2 if args.storage == "bf16" else 4
        n_d = sum(p.numel() for p in [*model.density_plane, *model.density_line])
        n_a = sum(p.numel() for p in [*model.app_plane, *model.app_line])
        gin_b = 2 if cfg_head(model) == "tc" else 4
        sm_clock = 1.965e9
        l1_peak = 148 * 128 * sm_clock / 1e9          # GB/s: one 128-byte L1 data-pipe wavefront per clock per SM

        def roof_of(name):
            per_ms = summ[name][0] / summ[name][1]
            cb = compulsory_bytes(name, V, A, n_d * s_el, n_a * s_el, n_d * 4, n_a * 4, ctot_a, gin_b)
            fl = gemm_flops(name, A, F_, ctot_a, in_dim, H_)
            ncu = ncu_lookup(name, args.workload, args.storage)
            if cb is None:
                return None
            ach = cb / (per_ms * 1e-3) / 1e9
            r = {"kernel": name, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                 "traffic": ncu["traffic"] if ncu else None, "peak_source": peak_src, "ms_per_launch": per_ms,
                 "algorithmic_bytes": cb,
                 "algorithmic_bytes_what": "compulsory HBM bytes of the data flow: per-sample streams + one read of the "
                                           "factors + one write-back of the gradient planes (bench.py compulsory_bytes)",
                 "logical_bytes_survey_8d": logical_bytes(name, V, A, cd, ca, ctot_a)}
            if ncu:
                r["traffic_over_algorithmic"] = ncu["traffic"] / cb
                r["ncu"] = {k: ncu[k] for k in ("kernels", "capture", "commit")}
            lb = l1_fill_bytes(name, V, A, cd, ca, s_el, s_el)
            if lb is not None:
                r["binding_unit"] = {"unit": "L1 data pipe (LSU wavefronts, 128 B/clk/SM x 148 SMs at 1965 MHz)",
                                     "bytes": lb, "achieved": lb / (per_ms * 1e-3) / 1e9, "peak": l1_peak,
                                     "frac": lb / (per_ms * 1e-3) / 1e9 / l1_peak,
                                     "ncu_l1_data_pipe_pct": ncu["l1_data_pipe_pct_ncu"] if ncu else None,
                                     "what": "tap bytes delivered to registers once per sample (fp32 or bf16 as stored)"}
            if fl is not None:
                r["tensor"] = {"achieved": fl / (per_ms * 1e-3) / 1e12, "peak": tf_peak, "unit": "TFLOP/s",
                               "frac": fl / (per_ms * 1e-3) / 1e12 / tf_peak}
            return r

        top = next((k for k in breakdown if compulsory_bytes(k, V, A, 1, 1, 1, 1, ctot_a, gin_b) is not None), None)
        roof = roof_of(top) if top else None
        if roof is not None:
            roof["V"], roof["A"] = V, A
            # the north star's named targets: gather, composite (and blur when active) kernels against HBM
            fam = {}
            for k in breakdown:
                if k != top and compulsory_bytes(k, V, A, 1, 1, 1, 1, ctot_a, gin_b) is not None:
                    rk = roof_of(k)
                    fam[k] = {"ms": rk["ms_per_launch"], "hbm_frac": round(rk["frac"], 4),
                              "traffic": rk["traffic"], "algorithmic_bytes": rk["algorithmic_bytes"],
                              "l1_frac": round(rk["binding_unit"]["frac"], 4) if "binding_unit" in rk else None}
            roof["other_kernels"] = fam
            step_bytes = sum(compulsory_bytes(k, V, A, n_d * s_el, n_a * s_el, n_d * 4, n_a * 4, ctot_a, gin_b) or 0
                             for k in breakdown)
            roof["step"] = {"compulsory_bytes": step_bytes, "ms_at_hbm_peak": step_bytes / hbm_peak / 1e6,
                            "ms_measured": ms / args.steps,
                            "hbm_frac": step_bytes / (ms / args.steps * 1e-3) / 1e9 / hbm_peak}

    # second half of BASELINE.json's metric: one 800x800 frame (640 000 rays, cfg2 field, is_train=False, no
    # blur) rendered like the reference's render_by_slices (model/nerf.py:728-740), rays resident on the device
    def time_render(mdl, mopt):
        n_pix = H_img * W_img
        f_pose, f_kinv = gt_pose[:1].to(dev), intr_inv_d[:1]
        rkw = dict(white_bg=run["white_bg"], is_train=False, ndc_ray=run["ndc"], N_samples=S)
        chunk = args.render_chunk

        def render_frame():
            """render_by_slices (nerf.py:728-740): per slice, rays of that slice only (jt_pose_rays_fwd) -> forward."""
            outs = []
            with torch.no_grad():
                for c in range(0, n_pix, chunk):
                    ce, ra = jt.camera.get_center_and_ray(cam_opt, f_pose, f_kinv, pix_base=c, n_rays=min(chunk, n_pix - c),
                                                          intr=intr_d[:1] if ndc else None)
                    outs.append(mdl(mopt, ce.view(-1, 3), ra.view(-1, 3), **rkw)[0])
            return torch.cat(outs)

        render_frame()
        torch.cuda.synchronize()
        frames = 3
        s_ev, e_ev = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        flush.fill_(1.0)
        s_ev.record()
        for _ in range(frames):
            img = render_frame()
        e_ev.record()
        torch.cuda.synchronize()
        fms = s_ev.elapsed_time(e_ev) / frames
        return {"ms_per_frame": fms, "rays_per_s": n_pix / (fms * 1e-3), "frame": f"{W_img}x{H_img}",
                "frames_timed": frames, "rays_per_call": chunk, "finite": bool(torch.isfinite(img).all())}

    render = time_render(model, opt) if rank == 0 and not args.no_render else None

    # the other shading head on the same 300^3 field (cfg2_sh <-> cfg2): same rays, same protocol, timed after the
    # headline so that it cannot disturb it. Single-GPU runs only.
    also = None
    other = {"cfg2_sh": "cfg2", "cfg2": "cfg2_sh"}.get(args.workload)
    if rank == 0 and world == 1 and other and not args.no_also and args.blur == 0:
        kw_o, _ = jt.synth.config(other)
        kw_o = dict(kw_o)
        torch.manual_seed(0)
        model_o = jt.B200_VMSplit(torch.tensor(kw_o.pop("aabb")), kw_o.pop("gridSize"), dev, **kw_o)
        model_o.head_precision = args.head
        model_o.factor_storage = args.storage
        opt_o = default_opt(model_o.shadingMode, run["ndc"])
        step_o = make_step(model_o, opt_o, [p for p in model_o.parameters()] + [se3_refine])
        for _ in range(max(args.warmup, 3)):
            step_o(pix_d, tgt_d, reduce=False)
        torch.cuda.synchronize()
        ms_o = timed(lambda: step_o(pix_d, tgt_d, reduce=False), args.steps)
        also = {"workload": jt.synth.describe(other, N), "value": N * args.steps / (ms_o * 1e-3), "unit": UNIT,
                "ms_per_step": ms_o / args.steps, "steps": args.steps}
        if not args.no_render:
            also["render_800x800"] = time_render(model_o, opt_o)
        del model_o, step_o
        torch.cuda.empty_cache()

    # the strict-fp32 row: the headline workload with head_precision="fp32" (SIMT fp32 GEMMs, gradients within 1e-4 of
    # the reference instead of the 2e-2 class of the bf16-operand backward GEMMs), same protocol
    strict = None
    if rank == 0 and world == 1 and args.head != "fp32" and not args.no_also and args.blur == 0:
        model.head_precision = "fp32"
        for _ in range(3):
            step(pix_d, tgt_d, reduce=False)
        torch.cuda.synchronize()
        ms_s = timed(lambda: step(pix_d, tgt_d, reduce=False), args.steps)
        strict = {"workload": jt.synth.describe(args.workload, N) + ", head_precision=fp32 (strict parity path)",
                  "value": N * args.steps / (ms_s * 1e-3), "unit": UNIT, "ms_per_step": ms_s / args.steps,
                  "steps": args.steps, "dtype": "f32"}
        model.head_precision = args.head
        torch.cuda.empty_cache()

    # the same step replayed from a CUDA graph (joint_tensorf_b200.graphs.GraphedStep): what the ~45 ctypes launches per
    # step cost on the host, and what a launch-bound batch gains (512 rays = the per-GPU share of a strong-scaled
    # 4096-ray step on 8 GPUs)
    graph_row = None
    if rank == 0 and world == 1 and not args.cuda_graph and not args.no_also and args.blur == 0:
        try:
            model.app_capacity = None
            pix_g, tgt_g = pix_d.clone(), tgt_d.clone()
            gs = jt.graphs.GraphedStep(lambda: eager_step(pix_g, tgt_g, reduce=False), warmup=3)
            ms_g = timed(gs, args.steps)
            graph_row = {"ms_per_step": ms_g / args.steps, "value": N * args.steps / (ms_g * 1e-3), "unit": UNIT,
                         "host_enqueue_ms_per_step": round(timed.host_ms, 3),
                         "what": "the headline step captured once and replayed (one graph launch per step)"}
            del gs
        except Exception as ex:          # an optional row must never take the bench line down
            graph_row = {"error": f"{type(ex).__name__}: {ex}"[:300]}
        torch.cuda.empty_cache()

    # next rows of SURVEY 8f, timed after everything above because the optimiser changes the parameters:
    # 8f-2 a full training iteration = the step above + density_L1 regulariser (Blender weight 8e-5, TV weights 0,
    # bat_blender_VM.yaml:134-139) + Adam update of every parameter; 8f-3 the between-step maintenance ops.
    extras = None
    if rank == 0 and not args.no_breakdown:
        from joint_tensorf_b200.sweeps import FusedAdam
        fused = FusedAdam(model.get_optparam_groups(0.02, 1e-3) + [{"params": [se3_refine], "lr": 1e-3}],
                          betas=(0.9, 0.99))
        decay = 0.1 ** (1 / 30000)

        def train_step():
            step(pix_d, tgt_d, reduce=False)
            model.regularize_(8e-5, 0.0, 0.0)
            fused.step()
            for grp in fused.param_groups:
                grp["lr"] *= decay

        for _ in range(3):
            train_step()
        torch.cuda.synchronize()
        ms_train = timed(train_step, 5) / 5
        ops.TIMER.enabled = True
        model.regularize_(8e-5, 1.0, 1.0)
        fused.step()
        ops.TIMER.summary()
        for _ in range(5):
            flush.fill_(1.0)
            model.regularize_(8e-5, 1.0, 1.0)            # all three terms: the LLFF configuration (weights 10.0)
            fused.step()
        sw = {k: round(v[0] / 5, 4) for k, v in ops.TIMER.summary().items()}
        n_par = sum(p.numel() for grp in fused.param_groups for p in grp["params"])
        # arrays the three-term sweep touches: density planes + lines (L1, TV) and appearance planes (TV)
        n_sw = sum(p.numel() for p in [*model.density_plane, *model.density_line, *model.app_plane])
        # algorithmic bytes: Adam reads p, g, m, v and writes p, m, v; the value sweep reads x once; the gradient
        # sweep reads x and read-modify-writes g
        sweep_bytes = {"adam": 28 * n_par, "reg_values": 4 * n_sw, "reg_grads": 12 * n_sw}
        extras = {"train_step_ms": round(ms_train, 4),
                  "train_step_what": "step + density_L1 (value + gradient sweep) + fused Adam over all parameters",
                  "sweep_ms": sw,
                  "sweep_gbs": {k: round(sweep_bytes[k] / (sw[k] * 1e-3) / 1e9, 1) for k in sweep_bytes if sw.get(k)},
                  "sweep_bytes": sweep_bytes, "hbm_peak_gbs": hbm_peak}
        # maintenance: dense alpha on 200^3 (tensorf.py update_alphamask), mask build, 150^3 -> 300^3 upsample
        model.kernel_density, model.c2f_mode = None, None
        kw2, _ = jt.synth.config(args.workload)
        kw2 = dict(kw2)
        kw2.pop("gridSize")
        aabb2 = torch.tensor(kw2.pop("aabb"))
        mt = None
        for rep in range(2):                          # rep 0 warms up, rep 1 is measured
            ops.TIMER.summary()
            a_zyx = model._dense_alpha_zyx([200, 200, 200])
            ops.alpha_mask_build(a_zyx, model.alphaMask_thres)
            small = jt.B200_VMSplit(aabb2, [150, 150, 150], dev, **kw2)
            small.upsample_volume_grid([300, 300, 300])
            del small
            mt = ops.TIMER.summary()
        ops.TIMER.enabled = False
        extras["maintenance_ms"] = {"dense_alpha_200^3": round(mt["field_alpha"][0], 4),
                                    "maxpool5_threshold_pack_200^3": round(mt["alpha_mask_build"][0], 4),
                                    "upsample_150^3_to_300^3_all_factors": round(mt["resize_bilinear"][0], 4)}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n_cpu = args.cpu_rays or N
        r = time_cpu_reference(args.workload, n_cpu, 2, 1, args.blur, budget_s=60.0)
        cpu = {"value": r["rps"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
               "sample": f"{n_cpu} of {N} rays per step, {r['steps']} timed fwd+bwd steps after {r['warmup']} warm-up: "
                         f"{r['what']}"}

    aten = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            rps, sec = time_aten_gpu(args.workload, N, 3, 1, dev)
            aten = {"value": rps, "unit": UNIT, "ms_per_step": sec * 1e3,
                    "what": f"reference algorithm (oracle port) with stock ATen CUDA kernels on this GPU, {N} rays, "
                            "fwd+bwd, 3 timed iterations; rays resident, no pose generation"}
        except Exception as ex:      # a baseline leg must never take the bench line down
            aten = {"error": f"{type(ex).__name__}: {ex}"[:300]}
        torch.cuda.empty_cache()

    if rank == 0:
        rays_total = N * world
        h2d = pix_h.numel() * 4 + tgt_h.numel() * 4
        line = {
            "metric": METRIC, "value": rays_total * args.steps / (ms * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "warmup_requested": args.warmup,
            "dtype": ("f32" if args.head == "fp32" else "f32 (basis/shading GEMMs on tcgen05: bf16 operands, f32 accumulate)") +
                     ("; VM factors gathered from a bf16 copy (fp32 master parameters and gradients)" if args.storage == "bf16" else ""),
            "data": "synthetic",
            "config": {"workload": jt.synth.describe(args.workload, N) +
                                   f" ({n_views} views x {R_pix} pixels, rays generated from se3_refine + pose inside the step), "
                                   "fwd+bwd to factor/basis/head/se3 gradients, optimizer step excluded",
                       "head": args.head, "factor_storage": args.storage, "rays_per_gpu": N,
                       "cuda_graph": bool(args.cuda_graph),
                       "head_arith": "forward: hi+lo split bf16 operands (3 MMAs per product, fp32-class, rgb within 1e-4); "
                                     "backward: bf16 operands, f32 accumulate (gradients within 2e-2 rel)",
                       "blur": args.blur, "l2": "256 MB write between timed steps (L2 flushed)",
                       "parallelism": f"ray-sharded x{world}, NCCL all-reduce of the flat fp32 gradient bucket inside the backward "
                                      "(appearance part overlapped with the density scatter)"},
            "e2e": {"value": rays_total * args.steps / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches), "host_enqueue_ms_per_step": round(host_ms, 3),
            "step_ms_rank0": per_step,
            "clocks": clk.summary(),
        }
        if roof is not None:
            line["roofline"] = roof
        if breakdown is not None:
            line["kernel_ms_per_step"] = breakdown
        if ddp_breakdown is not None:
            line["kernel_ms_per_step_data_parallel_rank0"] = ddp_breakdown
        if render is not None:
            line["render_800x800"] = render
        if also is not None:
            line["also"] = also
        if strict is not None:
            line["strict_fp32"] = strict
        if graph_row is not None:
            line["cuda_graph_replay"] = graph_row
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if aten is not None:
            line["aten_gpu_baseline"] = aten
        if extras is not None:
            line["next_rows"] = extras
        print(json.dumps(line), flush=True)
    if world > 1 and args.cuda_graph:
        # a process group whose collectives were captured into a live CUDA graph does not tear down cleanly
        # (destroy_process_group hung at N = 2): synchronise, meet the other ranks, leave without the teardown
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        os._exit(0)
    if world > 1:
        dist.destroy_process_group()


def render_arm(args):
    """BASELINE configs[4]: --frames full 800x800 views of the 300^3 field, image-sharded over the ranks (rank r
    renders frames r, r + W, ...: parallel.frames_of_rank, the slicing of nerf.py:728-740 per frame), no
    collective on the data path. value = ms per frame = (max over ranks of the device time for its frames) / frames.
    e2e: every frame's pose comes from pinned host memory and its rgb image goes back to the host."""
    import torch.distributed as dist

    import joint_tensorf_b200 as jt
    from joint_tensorf_b200 import parallel
    from joint_tensorf_b200.options import default_opt

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    wl = args.workload if args.workload in ("cfg2", "cfg2_sh") else "cfg2"
    kw, run = jt.synth.config(wl)
    kw = dict(kw)
    torch.manual_seed(0)
    model = jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), dev, **kw)
    model.head_precision = args.head
    model.factor_storage = args.storage
    opt = default_opt(model.shadingMode, False)
    H_img = W_img = 800
    n_pix = H_img * W_img
    poses_h, intr = jt.synth.blender_views(args.frames, (H_img, W_img), seed=11)
    poses_h = poses_h.pin_memory()
    kinv = intr[:1].inverse().to(dev)
    cam_opt = jt.options.Namespace(H=H_img, W=W_img, camera=dict(model="perspective", ndc=False), arch=dict())
    rkw = dict(white_bg=True, is_train=False, ndc_ray=False, N_samples=run["n_samples"])
    chunk = args.render_chunk
    mine = parallel.frames_of_rank(args.frames, rank, world)
    img_h = torch.empty((n_pix, 3), pin_memory=True)

    def render_frame(pose_d):
        outs = []
        with torch.no_grad():
            for c in range(0, n_pix, chunk):
                ce, ra = jt.camera.get_center_and_ray(cam_opt, pose_d, kinv, pix_base=c, n_rays=min(chunk, n_pix - c))
                outs.append(model(opt, ce.view(-1, 3), ra.view(-1, 3), **rkw)[0])
        return torch.cat(outs)

    def run_all(e2e):
        finite = True
        s_ev, e_ev = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        poses_d = poses_h.to(dev)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        s_ev.record()
        for f in mine:
            pose = poses_h[f:f + 1].to(dev, non_blocking=True) if e2e else poses_d[f:f + 1]
            img = render_frame(pose)
            if e2e:
                img_h.copy_(img, non_blocking=True)
        e_ev.record()
        torch.cuda.synchronize()
        finite = bool(torch.isfinite(img).all()) if mine else True
        t = torch.tensor([s_ev.elapsed_time(e_ev)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), finite

    for f in mine[:max(1, min(args.warmup, 3))]:
        render_frame(poses_h[f:f + 1].to(dev))
    l0 = jt._lib.launch_count()
    with ClockSampler(local) as clk:
        ms, finite = run_all(False)
        launches = jt._lib.launch_count() - l0
        if launches_per_graph is not None:
            launches = launches_per_graph * args.steps               # replayed, not re-issued: count what the graph holds
        ms_e2e, _ = run_all(True)
    if rank == 0:
        line = {"metric": RENDER_METRIC, "value": ms / args.frames, "unit": "ms/frame", "n_gpus": world,
                "steps": args.frames, "warmup": max(1, min(args.warmup, 3)), "ms_per_step": ms / args.frames,
                "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32 (MLP_Fea inference GEMMs: fp16 operands on tcgen05, f32 accumulate)" if wl == "cfg2" else
                         "f32 (basis GEMM: hi+lo bf16 operands on tcgen05)",
                "data": "synthetic",
                "config": {"workload": jt.synth.describe(wl) + f", {args.frames} hemisphere views at 800x800, is_train=False, "
                                       f"{chunk} rays per forward call, frames dealt round-robin to the ranks",
                           "frames_per_rank": len(mine), "head": args.head, "factor_storage": args.storage,
                           "parallelism": f"image-sharded x{world}, no collective on the data path",
                           "l2": "each frame streams 640 000 rays x ~650 samples: working set >> L2"},
                "e2e": {"value": ms_e2e / args.frames, "unit": "ms/frame", "h2d_bytes_per_step": 48,
                        "d2h_bytes_per_step": n_pix * 12, "ms_per_step": ms_e2e / args.frames},
                "rays_per_s": args.frames * n_pix / (ms * 1e-3), "single_gpu_ms_per_frame_rank0": ms * world / args.frames
                if world > 1 else ms / args.frames, "finite": finite, "gpu_launches": int(launches),
                "clocks": clk.summary()}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        reference_arm(a)
    elif a.mode == "render":
        render_arm(a)
    else:
        own_arm(a)
