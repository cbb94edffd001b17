"""Time the ray caster (B200_VMSplit.raycast's jt_raycast) on full 800x800 frames in 4096-ray slices of the benchmark's
random-init fields: cfg2_sh (300^3, Blender-shaped rays of synth.frame_rays) and cfg4 (617x687x617, 640000 LLFF NDC
rays of synth.llff_ndc_rays), at the dense alpha's median and 0.99 quantile levels (mesh_bench's choice), next to
render_normals and the no-grad forward of the same frames.

Each frame's slices run between two CUDA events, L2 flushed (a 256 MB write) before each frame; median of --reps
frames after --warmup. The kernel is timed with rays handed out by its atomic counter (the default) and by a static
grid stride. Samples gathered per ray: the sample phase gathers whole iterations of 16 (2 lanes per sample) or 8
samples up to the hit (or to the end of the ray's run through the box), plus 15 or 7 sub-points per refinement round;
the script counts the in-box samples up to the hit from k and the marcher's valid mask, and the rounds from the kernel.

    python scripts/raycast_bench.py [--warmup 2] [--reps 5] [--out FILE]
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
FRAME = 800 * 800


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        name, power, clock = torch.cuda.get_device_name(0), "unknown", "unknown"
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


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
    times = sorted(times)
    return dict(median=round(times[len(times) // 2], 3), min=round(times[0], 3))


def bench(workload, warmup, reps, flush):
    kw, run = jt.synth.config(workload)
    kw = dict(kw)
    torch.manual_seed(0)
    m = jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), DEV, **kw)
    S, ndc = run["n_samples"], run["ndc"]
    if ndc:
        o, d, _ = jt.synth.llff_ndc_rays(n_rays=FRAME)
    else:
        o, d = jt.synth.frame_rays()
    o, d = o.to(DEV), d.to(DEV)
    slices = [(i, min(i + SLICE, o.shape[0])) for i in range(0, o.shape[0], SLICE)]
    opt = default_opt(m.shadingMode, ndc)
    a = m._dense_alpha_zyx(m._grid).reshape(-1).sort().values
    levels = {name: float(a[int(q * (a.numel() - 1))]) for name, q in (("median", 0.5), ("q0.99", 0.99))}
    del a
    torch.cuda.empty_cache()
    lanes = 15 if all(c == 16 for c in m.density_n_comp) else 7
    fs, geom, act = m._density_factorset(), m._h_geom(), 0 if m.fea2denseAct == "softplus" else 1
    ztab = m._ndc_table(S, False).contiguous() if ndc else None

    def cast(level, counter=True):
        for i, j in slices:
            ops.raycast(fs, geom, m.density_shift, act, float(m._h_step), level, o[i:j], d[i:j], S, ztab=ztab,
                        mask=m.alphaMask, counter=counter)

    def fwd():
        with torch.no_grad():
            for i, j in slices:
                m.forward(opt, o[i:j], d[i:j], white_bg=run["white_bg"], is_train=False, ndc_ray=ndc, N_samples=S)

    def nrm():
        for i, j in slices:
            m.render_normals(o[i:j], d[i:j], ndc_ray=ndc, N_samples=S)

    rows = []
    for name, level in levels.items():
        ms = timed(lambda: cast(level), warmup, reps, flush)
        ms_static = timed(lambda: cast(level, counter=False), warmup, reps, flush)
        ms_method = timed(lambda: [m.raycast(o[i:j], d[i:j], level=level, ndc_ray=ndc, N_samples=S)
                                   for i, j in slices], warmup, reps, flush)
        # samples gathered per ray: in-box samples up to the hit (the whole box run on a miss) + refinement sub-points
        hits, gathered, marched, rounds_sum = 0, 0, 0, 0
        for i, j in slices:
            t, _, k, rnd = ops.raycast(fs, geom, m.density_shift, act, float(m._h_step), level, o[i:j], d[i:j], S,
                                       ztab=ztab, mask=m.alphaMask, rounds=True)
            if ndc:
                _, _, valid = m.sample_ray_ndc(o[i:j], d[i:j], is_train=False, N_samples=S)
            else:
                _, _, valid = m.sample_ray(o[i:j], d[i:j], is_train=False, N_samples=S)
            valid = valid.bool()
            upto = torch.where(k >= 0, k, torch.full_like(k, S - 1)).long()
            in_run = valid & (torch.arange(S, device=DEV)[None, :] <= upto[:, None])
            gathered += int(in_run.sum()) + lanes * int(rnd.sum())
            marched += int(valid.sum())
            rounds_sum += int(rnd.sum())
            hits += int((k >= 0).sum())
        n = o.shape[0]
        rows.append(dict(level_name=name, level=level, hit_fraction=round(hits / n, 4), raycast_ms=ms,
                         raycast_static_stride_ms=ms_static, method_with_normals_ms=ms_method,
                         rays_per_s=round(n / (ms["median"] * 1e-3), 0),
                         samples_gathered_per_ray=round(gathered / n, 2),
                         refinement_rounds_per_hit=round(rounds_sum / max(hits, 1), 3),
                         valid_samples_per_ray=round(marched / n, 2)))
    res = dict(workload=workload, grid_xyz=list(m._grid), rays=o.shape[0], slice_rays=SLICE, n_samples=S, ndc=ndc,
               refine_points_per_round=lanes, levels=rows,
               forward_nograd_ms=timed(fwd, warmup, reps, flush), render_normals_ms=timed(nrm, warmup, reps, flush))
    del m
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", default="cfg2_sh,cfg4")
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("raycast_bench.py needs a CUDA device")
    flush = torch.empty((64 << 20,), device=DEV)           # 256 MB > the 126 MB L2
    doc = dict(what="raycast (jt_raycast) per full frame in 4096-ray slices, next to render_normals and the no-grad "
                    "forward of the same frames; L2 flushed before each frame",
               **gpu_info(), torch=torch.__version__,
               frames=[bench(w, args.warmup, args.reps, flush) for w in args.workloads.split(",")])
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
