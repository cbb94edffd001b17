"""Time mesh extraction on the benchmark's fields: the dense alpha grid (jt_field_alpha) and marching cubes on it
(ops.marching_cubes: count, 16-byte read-back, emit) separately.

Fields: the random-init cfg2 field (300^3) and cfg4 field (617x687x617), seeded as bench.py seeds them. Levels: the
0.99 quantile of alpha (a sparse surface) and its median (about the worst case: half the lattice edges can cross).
Quantiles rather than TensoRF's 0.005 because a random-init field need not reach 0.005 anywhere. Times: CUDA events
after warm-up, median of --reps calls, a 256 MB write between calls evicts the L2 (outside the timed region).
`vol_GBps` is the volume's bytes (4 per lattice point, read once by the classify pass) over the marching-cubes time,
reported next to the data-sheet HBM bandwidth; the emit pass reads the volume again near crossings and writes the
mesh, so this is a rate of the whole op, not a bandwidth of one kernel.

    python scripts/mesh_bench.py [--workloads cfg2,cfg4] [--warmup 3] [--reps 10] [--out FILE]
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


def timed(fn, warmup, reps, flush):
    for _ in range(warmup):
        out = fn()
    times = []
    for _ in range(reps):
        flush.fill_(1.0)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = fn()
        e.record()
        torch.cuda.synchronize()
        times.append(s.elapsed_time(e))
    times.sort()
    return out, dict(median=round(times[len(times) // 2], 4), min=round(times[0], 4))


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
    ap.add_argument("--workloads", default="cfg2,cfg4")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("mesh_bench.py needs a CUDA device")
    flush = torch.empty(256 * 1024 * 1024 // 4, device=DEV)         # > 126 MB L2
    doc = dict(what="dense alpha (jt_field_alpha) and marching cubes (ops.marching_cubes) on random-init fields",
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
