"""Time mesh extraction on the benchmark's fields: the dense alpha grid (jt_field_alpha), marching cubes on it
(ops.marching_cubes: count, 16-byte read-back, emit), the vertex normals (jt_mc_normals) and the vertex colours
(B200_VMSplit.compute_rgb(verts, -normals), the colour pass of extract_mesh(colors=True)) separately.

Fields: the random-init cfg2_sh (300^3, SH head), cfg2 (300^3, MLP_Fea head) and cfg4 (617x687x617, WeakView head)
fields, seeded as bench.py seeds them; each runs the head head_precision="auto" picks (the tensor-core heads). Levels: the
0.99 quantile of alpha (a sparse surface) and its median (about the worst case: half the lattice edges can cross).
Quantiles rather than TensoRF's 0.005 because a random-init field need not reach 0.005 anywhere. Times: CUDA events
after warm-up, median of --reps calls, a 256 MB write between calls evicts the L2 (outside the timed region).
`vol_GBps` is the volume's bytes (4 per lattice point, read once by the classify pass) over the marching-cubes time,
reported next to the data-sheet HBM bandwidth; the emit pass reads the volume again near crossings and writes the
mesh, so this is a rate of the whole op, not a bandwidth of one kernel.
`normals_ms` is the jt_mc_normals launch alone, timed by CUDA events around it inside ops.marching_cubes(normals=True)
calls (the L2 is flushed before each call, so the normals pass finds in L2 what count and emit left there, as it does
in use); `mc_normals_op_ms` is that whole call. `rgb_ms` is compute_rgb on all vertices, L2 flushed before each call.

    python scripts/mesh_bench.py [--workloads cfg2_sh,cfg2,cfg4] [--warmup 3] [--reps 10] [--out FILE]
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

DEV = "cuda:0"
HBM_GBPS = 7700.0      # NVIDIA HGX B200 data sheet, per GPU, at up to 1000 W


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


def timed(fn, warmup, reps, flush, span=None):
    """fn's time over `reps` calls after `warmup`; with `span`, also the time of the ops.TIMER span of that name
    inside each call (returned as the "span" entry)."""
    for _ in range(warmup):
        out = fn()
    times, spans = [], []
    for _ in range(reps):
        flush.fill_(1.0)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ops.TIMER.enabled = span is not None
        s.record()
        out = fn()
        e.record()
        ops.TIMER.enabled = False
        torch.cuda.synchronize()
        times.append(s.elapsed_time(e))
        if span is not None:
            spans.append(ops.TIMER.summary()[span][0])
    res = _stats(times)
    if span is not None:
        res["span"] = _stats(spans)
    return out, res


def bench(workload, warmup, reps, flush):
    kw, _ = jt.synth.config(workload)
    kw = dict(kw)
    torch.manual_seed(0)
    m = jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), DEV, **kw)
    grid = m._grid
    alpha, alpha_ms = timed(lambda: m._dense_alpha_zyx(grid), warmup, reps, flush)
    flat = alpha.reshape(-1).sort().values
    n = flat.numel()
    rows = []
    for name, q in (("q0.99", 0.99), ("median", 0.5)):
        level = float(flat[int(q * (n - 1))])
        lin = m._dense_tables(grid)
        (verts, faces), mc_ms = timed(lambda: ops.marching_cubes(alpha, level, lin, m._h_aabb), warmup, reps, flush)
        rows.append(dict(level_name=name, level=level, V=int(verts.shape[0]), F=int(faces.shape[0]), mc_ms=mc_ms,
                         vol_GBps=round(4.0 * n / (mc_ms["median"] * 1e-3) / 1e9, 1),
                         vol_share_of_hbm=round(4.0 * n / (mc_ms["median"] * 1e-3) / 1e9 / HBM_GBPS, 3)))
        del verts, faces
        (verts, faces, nrm), op_ms = timed(lambda: ops.marching_cubes(alpha, level, lin, m._h_aabb, normals=True),
                                           warmup, reps, flush, span="mc_normals")
        normals_ms = op_ms.pop("span")
        with torch.no_grad():
            dirs = -nrm
            _, rgb_ms = timed(lambda: m.compute_rgb(verts, dirs), warmup, reps, flush)
        nv = int(verts.shape[0])
        rows[-1].update(normals_ms=normals_ms, mc_normals_op_ms=op_ms, normals_Mverts_per_s=round(
            nv / (normals_ms["median"] * 1e-3) / 1e6, 1), rgb_ms=rgb_ms,
            rgb_Mverts_per_s=round(nv / (rgb_ms["median"] * 1e-3) / 1e6, 1))
        del verts, faces, nrm, dirs
        if name == "median":                          # peak device memory of one call beyond the volume it reads
            torch.cuda.synchronize()
            before = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            out = ops.marching_cubes(alpha, level, lin, m._h_aabb)
            torch.cuda.synchronize()
            rows[-1]["peak_extra_bytes"] = torch.cuda.max_memory_allocated() - before
            del out
    scratch = int(jt._lib.lib().jt_mc_scratch_bytes(*grid))
    res = dict(workload=workload, grid_xyz=grid, points=n, volume_bytes=4 * n, scratch_bytes=scratch,
               dense_alpha_ms=alpha_ms, runs=rows)
    del m, alpha, flat
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--workloads", default="cfg2_sh,cfg2,cfg4")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("mesh_bench.py needs a CUDA device")
    flush = torch.empty(256 * 1024 * 1024 // 4, device=DEV)         # > 126 MB L2
    doc = dict(what="dense alpha (jt_field_alpha), marching cubes (ops.marching_cubes), vertex normals (jt_mc_normals) "
                    "and vertex colours (compute_rgb) on random-init fields",
               l2="256 MB write between timed calls (L2 flushed)", warmup=args.warmup, reps=args.reps,
               hbm_GBps_datasheet=HBM_GBPS, **gpu_info(),
               results=[bench(w, args.warmup, args.reps, flush) for w in args.workloads.split(",")])
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
