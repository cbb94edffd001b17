"""Time the field geometry queries on the benchmark's random-init fields: compute_density_grad (jt_field_density_grad
at explicit points) on cfg2_sh (300^3, 3 x 16 density channels) and cfg4 (617x687x617), and render_normals on full
800x800 frames (synth.frame_rays, 4096-ray slices) of cfg2_sh, next to the no-grad forward of the same frames.

Point queries: 2^22 uniform points in the aabb, CUDA events around each call, median of --reps calls after warm-up,
a 256 MB write before each call evicts the L2 (outside the timed region). Frames: the whole frame's slices between
two events, L2 flushed before each frame. The per-kernel times (`spans`) come from a separate pass with ops.TIMER's
events around every launch: the density gather of forward (vm_density_fwd) and the gradient gather of render_normals
(field_density_grad) summed over the frame, and per valid sample.

    python scripts/normals_bench.py [--warmup 2] [--reps 10] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

import joint_tensorf_b200 as jt  # noqa: E402
from joint_tensorf_b200 import ops  # noqa: E402
from joint_tensorf_b200.options import default_opt  # noqa: E402

DEV = "cuda:0"
SLICE = 4096


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        name, power, clock = torch.cuda.get_device_name(0), "unknown", "unknown"
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def _stats(times):
    times = sorted(times)
    return dict(median=round(times[len(times) // 2], 4), min=round(times[0], 4))


def timed(fn, warmup, reps, flush):
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(reps):
        flush.fill_(1.0)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        times.append(s.elapsed_time(e))
    return _stats(times)


def _module(workload):
    kw, run = jt.synth.config(workload)
    kw = dict(kw)
    torch.manual_seed(0)
    return jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), DEV, **kw), run


def bench_points(workload, n, warmup, reps, flush):
    m, _ = _module(workload)
    g = torch.Generator().manual_seed(1)
    lo, hi = m.aabb[0].cpu(), m.aabb[1].cpu()
    xyz = (lo + (hi - lo) * torch.rand(n, 3, generator=g)).to(DEV)
    ms = timed(lambda: m.compute_density_grad(xyz), warmup, reps, flush)
    alpha_ms = timed(lambda: m.compute_alpha(xyz), warmup, reps, flush)
    res = dict(workload=workload, grid_xyz=list(m._grid), points=n, density_grad_ms=ms,
               density_grad_Gpoints_per_s=round(n / (ms["median"] * 1e-3) / 1e9, 3), compute_alpha_ms=alpha_ms)
    del m, xyz
    torch.cuda.empty_cache()
    return res


def bench_frame(workload, warmup, reps, flush):
    m, run = _module(workload)
    S = run["n_samples"]
    o, d = jt.synth.frame_rays()
    o, d = o.to(DEV), d.to(DEV)
    opt = default_opt(m.shadingMode, False)
    slices = [(i, min(i + SLICE, o.shape[0])) for i in range(0, o.shape[0], SLICE)]

    def fwd():
        with torch.no_grad():
            for a, b in slices:
                m.forward(opt, o[a:b], d[a:b], white_bg=True, is_train=False, N_samples=S)

    def nrm():
        for a, b in slices:
            m.render_normals(o[a:b], d[a:b], N_samples=S)

    fwd_ms = timed(fwd, warmup, reps, flush)
    nrm_ms = timed(nrm, warmup, reps, flush)
    # kernel spans and the frame's valid-sample count, in a pass of their own
    samples = 0
    ops.TIMER.enabled = True
    with torch.no_grad():
        for a, b in slices:
            m.forward(opt, o[a:b], d[a:b], white_bg=True, is_train=False, N_samples=S)
            samples += int(jt.VMRender.last_counts[0].item())
    spans_f = ops.TIMER.summary()
    nrm()
    spans_n = ops.TIMER.summary()
    ops.TIMER.enabled = False
    dens = spans_f["vm_density_fwd"][0]
    grad = spans_n["field_density_grad"][0]
    ncomp = spans_n["normal_composite"][0]
    res = dict(workload=workload, frame="800x800", slice_rays=SLICE, n_samples=S, valid_samples=samples,
               forward_nograd_ms=fwd_ms, render_normals_ms=nrm_ms,
               spans=dict(forward_vm_density_fwd_ms=round(dens, 4), render_normals_field_density_grad_ms=round(grad, 4),
                          render_normals_normal_composite_ms=round(ncomp, 4),
                          vm_density_fwd_ns_per_sample=round(dens * 1e6 / max(samples, 1), 4),
                          field_density_grad_ns_per_sample=round(grad * 1e6 / max(samples, 1), 4)))
    del m
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--points", type=int, default=1 << 22)
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("normals_bench.py needs a CUDA device")
    flush = torch.empty((64 << 20,), device=DEV)           # 256 MB > the 126 MB L2
    doc = dict(what="compute_density_grad (jt_field_density_grad) points/s, render_normals and no-grad forward per "
                    "800x800 frame in 4096-ray slices; L2 flushed before each timed call",
               **gpu_info(), torch=torch.__version__,
               points=[bench_points(w, args.points, args.warmup, args.reps, flush) for w in ("cfg2_sh", "cfg4")],
               frames=[bench_frame("cfg2_sh", args.warmup, args.reps, flush)])
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
