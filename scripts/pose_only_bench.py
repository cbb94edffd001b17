"""Time the test-time pose-optimisation step with a frozen and with a trainable scene.

One step: se3 [1,6] -> camera.get_center_and_ray for 4096 pixels of one view -> render -> MSE -> backward -> d se3
(model/bat.py's per-image test-time optimisation). The frozen scene (freeze_scene()) and the trainable one run
alternately in one process on the same seeded field, pose and pixels. Step times: CUDA events around each step, a
256 MB write between steps evicts the L2 (outside the timed region). Kernel times of the backward: torch.profiler
in a separate pass. Prints one JSON document (and writes it to --out).

    python scripts/pose_only_bench.py [--workloads cfg2_sh,cfg2,cfg4] [--warmup 5] [--steps 50] [--out FILE]
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
from joint_tensorf_b200.options import default_opt  # noqa: E402

DEV = "cuda:0"
N_RAYS = 4096


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        name, power = torch.cuda.get_device_name(0), "unknown"
    return dict(gpu=name, power_limit=power)


def setup(workload, head):
    kw, run = jt.synth.config(workload)
    kw = dict(kw)
    ndc = bool(run["ndc"])
    if ndc:
        kw["near_far"] = [-1.0, 1.0]               # LLFF at the end of tensorf_near_plane_schedule
    torch.manual_seed(0)
    m = jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), DEV, **kw)
    m.head_precision = head
    if ndc:
        H, W = 756, 1008
        pose, intr = jt.synth.llff_views(1, (H, W), seed=1)
    else:
        H, W = 800, 800
        pose, intr = jt.synth.blender_views(1, (H, W), seed=1)
    pose, kinv = pose.to(DEV), intr.inverse().to(DEV)
    intr_d = intr.to(DEV) if ndc else None
    cam = jt.options.Namespace(H=H, W=W, camera=dict(model="perspective", ndc=ndc),
                               arch=dict(ndc_near_plane=1.0) if ndc else dict())
    pix = torch.randperm(H * W, generator=torch.Generator().manual_seed(7))[:N_RAYS].to(torch.int32).to(DEV)
    tgt = torch.rand((N_RAYS, 3), generator=torch.Generator().manual_seed(100)).to(DEV)
    se3 = torch.nn.Parameter(torch.zeros((1, 6), device=DEV))
    opt = default_opt(m.shadingMode, ndc)
    fkw = dict(white_bg=run["white_bg"], is_train=False, ndc_ray=ndc, N_samples=run["n_samples"])

    def forward():
        c, r = jt.camera.get_center_and_ray(cam, pose, kinv, ray_idx=pix, intr=intr_d, se3_refine=se3)
        rgb = m(opt, c.view(-1, 3), r.view(-1, 3), **fkw)[0]
        return ((rgb - tgt) ** 2).mean()

    def step(frozen):
        (m.freeze_scene if frozen else m.unfreeze_scene)()
        se3.grad = None
        for p in m.parameters():
            p.grad = None
        forward().backward()
        return se3.grad

    return m, forward, step, run


def kernel_times(m, forward, frozen, n=10):
    """Mean device time per backward of every kernel the backward launches (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    (m.freeze_scene if frozen else m.unfreeze_scene)()
    acc = {}
    for _ in range(n):
        for p in m.parameters():
            p.grad = None
        loss = forward()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            loss.backward()
            torch.cuda.synchronize()
        for e in prof.key_averages():
            t = getattr(e, "self_device_time_total", None)
            if t is None:
                t = getattr(e, "self_cuda_time_total", 0.0)
            if t > 0:
                acc[e.key] = acc.get(e.key, 0.0) + t
    kt = {k: round(v / n / 1e3, 4) for k, v in sorted(acc.items(), key=lambda kv: -kv[1])}
    return dict(total_ms=round(sum(kt.values()), 4), kernels_ms=kt)


def bench(workload, head, warmup, steps):
    m, forward, step, run = setup(workload, head)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=DEV)         # > 126 MB L2
    for _ in range(warmup):
        for frozen in (False, True):
            step(frozen)
    g_full, g_frozen = step(False).clone(), step(True).clone()
    times = {False: [], True: []}
    torch.cuda.synchronize()
    for _ in range(steps):                                             # alternating: frozen / trainable
        for frozen in (False, True):
            flush.fill_(1.0)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            step(frozen)
            e.record()
            times[frozen].append((s, e))
    torch.cuda.synchronize()
    ms = {k: sorted(s.elapsed_time(e) for s, e in v) for k, v in times.items()}

    def summary(v):
        return dict(mean=round(sum(v) / len(v), 4), median=round(v[len(v) // 2], 4), min=round(v[0], 4))

    res = dict(workload=workload, head=head, n_rays=N_RAYS, n_samples=run["n_samples"],
               step_ms_trainable=summary(ms[False]), step_ms_frozen=summary(ms[True]),
               d_se3_rel_diff=float((g_frozen - g_full).abs().max() / g_full.abs().max().clamp_min(1e-30)),
               bwd_kernels_trainable=kernel_times(m, forward, False), bwd_kernels_frozen=kernel_times(m, forward, True))
    res["speedup_median"] = round(res["step_ms_trainable"]["median"] / res["step_ms_frozen"]["median"], 3)
    del m, flush
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--workloads", default="cfg2_sh,cfg2,cfg4")
    ap.add_argument("--head", default="tc", choices=["tc", "fp32"])
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    args = ap.parse_args()
    if args.warmup < 5 or args.steps < 50:
        ap.error("at least 5 warm-up and 50 timed steps per mode")
    if not torch.cuda.is_available():
        sys.exit("pose_only_bench.py needs a CUDA device")
    doc = dict(what="test-time pose optimisation step (se3 -> rays -> render -> MSE -> backward), frozen vs "
                    "trainable scene, alternating in one process",
               l2="256 MB write between timed steps (L2 flushed)", warmup=args.warmup, steps=args.steps,
               **gpu_info(), results=[bench(w, args.head, args.warmup, args.steps) for w in args.workloads.split(",")])
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
