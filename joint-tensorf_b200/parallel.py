"""Ray-sharded data parallelism (SURVEY.md section 8e).

One process per GPU; every rank holds a replica of the VM factors, basis_mat, the
shading head and the per-image pose table, renders its own contiguous slice of
the step's ray list, and the gradients are summed with ONE collective over a
flat fp32 bucket (NCCL over NVLink/NVSwitch on the GPU box; gloo in the CPU
tests). The reference has no multi-GPU path (options.py:126); this is the
B200-native addition named by the north star.
"""
import torch
import torch.distributed as dist


def shard_bounds(n_items, rank, world):
    """Contiguous slice [lo, hi) of rank `rank`; sizes differ by at most one."""
    base, rem = divmod(n_items, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_rays(rays_o, rays_d, rank, world, *extra):
    lo, hi = shard_bounds(rays_o.shape[0], rank, world)
    return (rays_o[lo:hi], rays_d[lo:hi], *[e[lo:hi] for e in extra])


def frames_of_rank(n_frames, rank, world):
    """Image-sharded full-frame rendering: rank r renders frames r, r+W, ..."""
    return list(range(rank, n_frames, world))


class GradBucket:
    """Flat fp32 bucket over the gradients of `params`.

    `attach()` points every p.grad at a view of one contiguous buffer (keeping each
    parameter's strides, so channel-last factors stay channel-last) -- autograd
    then accumulates straight into the bucket and `all_reduce()` is a single
    collective with no flatten/unflatten copies."""

    def __init__(self, params):
        self.params = [p for p in params if p.requires_grad]
        self.sizes = [p.numel() for p in self.params]
        dev = self.params[0].device
        self.flat = torch.zeros((sum(self.sizes),), device=dev, dtype=torch.float32)
        self.views = []
        o = 0
        for p, n in zip(self.params, self.sizes):
            self.views.append(torch.as_strided(self.flat, p.shape, p.stride(), o))
            o += n

    def attach(self):
        for p, v in zip(self.params, self.views):
            p.grad = v

    def zero(self):
        self.flat.zero_()

    def all_reduce(self, group=None, average=True, async_op=False):
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return None
        work = dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=group, async_op=async_op)
        if average and not async_op:
            self.flat.div_(dist.get_world_size(group))
        return work


class OverlappedGradSync:
    """Sum the gradients of a step across ranks while its backward is still running.

    `sync.attach(model)` (or `model.grad_sync = sync`) makes the render node's backward hand over its flat gradient
    bucket in two parts: the appearance-factor gradients (3/4 of the bytes, complete after the appearance scatter)
    are all-reduced on NCCL's stream while the density scatter runs; the rest (density factors, basis_mat, head)
    follows and the backward's stream waits for both before the node returns, so whatever consumes the gradients
    next (p.grad, the adjoint blur -- linear, so reducing before it is the same sum) sees cross-rank sums.
    `finish(extra)` reduces the few gradients produced by later autograd nodes (se3_refine) in place.

    Semantics (read this before writing a training loop):
      * SUMS only. Scale the RENDER loss by 1/world_size for a mean: `(render_loss / world + regularisers).backward()`.
        Gradients that reach the factors from other autograd nodes (density_L1 / TV_loss_* through FieldRegularizers)
        or through `regularize_()` are NOT reduced -- they are identical on every rank (replicated parameters), so
        they must carry their full single-GPU weight, not 1/world.
      * every backward through the render node issues collectives while a synchroniser is attached: a backward that
        only some ranks run (validation on rank 0, test-time pose optimisation) must run under `with sync.paused():`
        or it hangs waiting for the other ranks.
      * `attach()` broadcasts the parameters from rank 0, so the replicas start identical even if the ranks were
        seeded differently.
    World size 1: every call is a no-op."""

    def __init__(self, group=None, per_plane=False, reserve_sms=0, split21="auto"):
        self.group = group
        self.works = []
        self.bytes = 0
        self.enabled = True
        # planes 0+1 | plane 2 | density with a collective after each launch (scatter_schedule). "auto": when it pays --
        # 4 or more ranks and an appearance part that dominates the bucket (measured: N=8 cfg2_sh 3.21 -> 3.12 ms,
        # N=2 3.04 -> 3.04, N=2 cfg4 2.15 -> 2.29)
        self.split21 = split21
        self.per_plane = per_plane        # one scatter launch + all-reduce per appearance plane (scatter_schedule)
        self.reserve_sms = reserve_sms    # SMs the density scatter leaves to the collective running next to it

    def use_split21(self, n_app, n_total):
        if self.split21 == "auto":
            return dist.get_world_size(self.group) >= 4 and n_app >= 2 * (n_total - n_app)
        return bool(self.split21)

    def _active(self):
        return self.enabled and dist.is_available() and dist.is_initialized() and dist.get_world_size(self.group) > 1

    def attach(self, model, extra_params=()):
        """Make `model` (B200_VMSplit) reduce its gradients through this object; broadcast its parameters (and
        `extra_params`, e.g. se3_refine) from rank 0."""
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(self.group) > 1:
            with torch.no_grad():
                for p in list(model.parameters()) + list(extra_params):
                    # channel-last factors: broadcast the underlying storage order, not a contiguous copy
                    buf = p.data.permute(0, 2, 3, 1) if (p.dim() == 4 and not p.data.is_contiguous()) else p.data
                    if not buf.is_contiguous():
                        tmp = buf.contiguous()
                        dist.broadcast(tmp, 0, group=self.group)
                        buf.copy_(tmp)
                    else:
                        dist.broadcast(buf, 0, group=self.group)
                    if hasattr(torch.autograd.graph, "increment_version"):
                        torch.autograd.graph.increment_version(p)      # refresh cached bf16 copies
        model.grad_sync = self
        return self

    def paused(self):
        """Context manager: backward passes inside it issue no collectives (rank-local work)."""
        import contextlib

        @contextlib.contextmanager
        def cm():
            prev, self.enabled = self.enabled, False
            try:
                yield self
            finally:
                self.enabled = prev
        return cm()

    def _reduce(self, t):
        if self._active() and t.numel() > 0:
            self.works.append(dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group, async_op=True))
            self.bytes += t.numel() * t.element_size()

    def on_app_grads(self, region):
        self._reduce(region)

    def on_rest(self, region):
        self._reduce(region)
        self.wait()

    def wait(self):
        if self.works:
            from .ops import TIMER
            with TIMER.span("grad_sync_wait"):     # device time the compute stream spends waiting for the collectives
                for w in self.works:
                    w.wait()
        self.works = []

    def finish(self, extra=()):
        """extra: parameters whose .grad was produced outside the render node (e.g. se3_refine): reduced in place,
        one small collective each (no concatenation / copy-back kernels)."""
        if self._active():
            for p in extra:
                if p.grad is not None:
                    g = p.grad if p.grad.is_contiguous() else None
                    if g is None:
                        p.grad = p.grad.contiguous()
                        g = p.grad
                    self._reduce(g)
        self.wait()


def scatter_schedule(sync, need_app, need_dens, need_rays, sizes, n_app, dens_resident):
    """The render op's factor-gradient scatter launches, in order: (app, max_ctas, plane_mask, cut) each -- app 1 walks
    the appearance factors, 0 the density factors; max_ctas and plane_mask are jt_vm_scatter_rays's launch form; after
    the launch the flat gradient bucket is complete up to offset `cut`, handed to `sync.on_app_grads` (None: no cut).
    sizes: numel of the bucket's tensors, appearance first; n_app: the appearance part; dens_resident: density-scatter
    CTAs per SM. Without a synchroniser a frozen factor group is walked coordinate-only if the rays need a gradient."""
    if sync is None:
        return [(app, 0, 7, None) for app, need in ((1, need_app), (0, need_dens)) if need or need_rays]
    if sync.per_plane:
        # variant (OverlappedGradSync(per_plane=True)): the appearance planes are walked one launch per plane and
        # each plane's gradients are all-reduced while the next launches run -- [plane 0] [plane 1] [plane 2 + the
        # three lines] [density + basis_mat + head]. Measured at N = 2 (profiles/r02e): the exposed wait halves
        # (0.21 -> 0.12 ms) but the non-persistent per-plane launches cost 0.11 ms more than they save.
        return [(1, -80, 1, sizes[0]), (1, -80, 2, sizes[0] + sizes[1]), (1, -80, 4, n_app), (0, -80, 7, None)]
    if sync.use_split21(n_app, sum(sizes)):
        # data parallel, 4+ ranks with an appearance-dominated bucket: [appearance planes 0+1: one persistent
        # launch] -> all-reduce of their 2/4 of the bucket starts -> [appearance plane 2] -> all-reduce of plane 2
        # + the three lines -> [density scatter] -> all-reduce of the rest. The collectives get a 0.7 ms window
        # (plane 2 + density) instead of the 0.4 ms of the density scatter alone, which at N = 8 is shorter than
        # the 69 MB all-reduce itself; the two launches that run next to a collective use fixed 80-sample segments
        # on a non-persistent grid, because NCCL's CTAs can only get onto an SM when scatter CTAs retire (a
        # persistent wave holds every SM until its kernel ends). Measured (profiles/r02l_*, r02n8c_*): N = 8:
        # exposed wait 0.36 -> 0.16 ms, the two scatters that share the SMs with a collective lose 0.10 ms, step
        # 3.21 -> 3.12 ms; N = 2: 3.04 vs 3.04 ms; cfg4 at N = 2 gets slower (2.15 -> 2.29: its bucket is half
        # density) -- hence use_split21.
        return [(1, 0, 3, sizes[0] + sizes[1]), (1, -80, 4, n_app), (0, -80, 7, None)]
    # 2 ranks / density-heavy buckets: the appearance part of the bucket is all-reduced while the density scatter
    # runs (non-persistent grid, or a persistent wave on the 148 SMs but sync.reserve_sms left to the collective)
    reserve = int(sync.reserve_sms)
    return [(1, 0, 7, n_app), (0, (148 - reserve) * dens_resident if reserve > 0 else -80, 7, None)]


def seed_all_ranks(seed):
    """Host RNG draws the reference makes per step (np.random.choice blur scale
    tensorf.py:198, torch.rand bg flip batBase.py:154, randperm ray_idx) must be
    identical on all ranks: seed them identically."""
    import random

    import numpy as np
    random.seed(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)
