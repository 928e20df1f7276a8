"""Batched multi-start fits sharded over GPUs (BASELINE config 4; SURVEY.md 8e).

``B`` independent ``JaxTrainer.fit`` loops (reference ``src/trainer.py:162-228``) that share the design X and differ in
their start point and, optionally, in their observations and measurement variances.  Restart b lives on rank
``b * world // B`` (contiguous shards); no data-path collective is needed because the restarts are independent.  The
ranks share only the best objective so far: either one 8-byte MIN all-reduce of a device word per optimiser chunk, on a
side stream that the fit launches never wait for, or (``trace=True``) the kernels' per-step record of it, which rides in
the one all-gather that also moves every rank's winner at the end of the fit.  The collectives run through the library's
own NCCL communicator (``comm.LfmComm``) or ``torch.distributed`` (NCCL, or gloo, whose final gather goes through
the host).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Tuple

import numpy as np


def make_restarts(theta_init: np.ndarray, B: int, scale: float = 0.5, seed: int = 42,
                  unconstrain=None, constrain=None) -> np.ndarray:
    """Start points: restart 0 is `theta_init`, restart b > 0 perturbs the UNCONSTRAINED leaves by
    scale * N(0, 1) drawn from default_rng(seed + b) (SURVEY.md 8d)."""
    from .model import L_HIGH, L_LOW, _softplus, _softplus_inv

    theta_init = np.asarray(theta_init, dtype=np.float64)
    P = theta_init.shape[0]
    G = (P - 2) // 3
    u0 = _softplus_inv(theta_init)
    r = (theta_init[3 * G] - L_LOW) / (L_HIGH - L_LOW)
    u0[3 * G] = np.log(r) - np.log1p(-r)
    U = np.empty((B, P))
    for b in range(B):
        U[b] = u0 if b == 0 else u0 + scale * np.random.default_rng(seed + b).standard_normal(P)
    TH = _softplus(U)
    TH[:, 3 * G] = L_LOW + (L_HIGH - L_LOW) * 0.5 * (1.0 + np.tanh(0.5 * U[:, 3 * G]))
    return TH


LAST_TIMING = None   # with LFM_MSF_TIMING=1: host milliseconds of the last fit's phases [setup, loop, tail]
_SIDE = {}


def _side_stream(device):
    """One side stream per device for the best-objective all-reduces (created once, not per fit)."""
    import torch

    key = device.index if device.index is not None else torch.cuda.current_device()
    if key not in _SIDE:
        _SIDE[key] = torch.cuda.Stream(device=device)
    return _SIDE[key]


def shard_bounds(B: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous restart range [lo, hi) of `rank`; sizes differ by at most one."""
    base, rem = divmod(B, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def reduce_best_gathered(allp: np.ndarray) -> np.ndarray:
    """Rows [loss, id, ...] gathered from every rank -> [best_loss, id_of_best]: MIN on the loss, then the smallest id
    among the rows that hold it; NaN / inf never win, and no finite loss gives [inf, -1]."""
    loss = np.where(np.isfinite(allp[:, 0]), allp[:, 0], np.inf)
    best = float(loss.min()) if loss.size else float("inf")
    if not np.isfinite(best):
        return np.array([np.inf, -1.0])
    return np.array([best, float(allp[loss == best, 1].min())])


@dataclass
class MultiStartResult:
    theta: np.ndarray        # (B_local, P) constrained results of this rank's shard
    history: np.ndarray      # (B_local, steps)
    info: np.ndarray         # (B_local,)
    lo: int
    hi: int
    best_loss: float         # global
    best_id: int             # global restart id
    best_theta: Optional[np.ndarray]  # global winner, broadcast to every rank
    best_trace: np.ndarray   # global best objective after every chunk
    device_ms: float = float("nan")   # CUDA-event time on this rank from the first enqueued operation (the input copy)
                                      # to the last (the read-back of the results): the fit as the device saw it


_PLANS = {}


class _Plan:
    """Everything of one rank's share of a multi-start fit that does not change between fits of the same shape, built once
    and reused: the pinned staging buffer and its device twin ([X | y | variances | start points], one host->device copy),
    the fit state with the result rows behind it (one allocation, one read-back), the key views and the events.  What is
    left per fit on the host is a few numpy copies into the staging buffer and a handful of stream-ordered calls -- the
    fit kernel is in flight ~30 us after `multi_start_fit` is entered instead of ~200 us (`tools/msf_timeline.py`)."""

    def __init__(self, device, N, G, Bl, per_lfm_y, num_iters, chunk, trace, world, var_rows):
        """`var_rows`: 0 without measurement variances, 1 with one vector shared by the shard, Bl with one row per LFM."""
        import torch

        from . import ops

        P = 3 * G + 2
        ev = lambda n: (int(n) + 1) & ~1
        self.N, self.ny, self.nv = N, (Bl if per_lfm_y else 1) * N, var_rows * N
        self.oy = ev(3 * N)
        self.ov = self.oy + ev(self.ny)
        self.oth = self.ov + ev(self.nv)
        total = self.oth + ev(Bl * P)
        self.pin_in = torch.empty(total, dtype=torch.float64, pin_memory=True)
        self.h_in = self.pin_in.numpy()
        self.d_in = torch.empty(total, dtype=torch.float64, device=device)
        self.Xd = self.d_in[:3 * N].view(N, 3)
        self.yd = self.d_in[self.oy:self.oy + self.ny]
        self.vd = self.d_in[self.ov:self.ov + self.nv] if self.nv else None
        self.th0 = self.d_in[self.oth:self.oth + Bl * P].view(Bl, P)
        self.y_stride = N if per_lfm_y else 0
        self.var_stride = N if var_rows > 1 else 0
        self.nchunks = max((num_iters + chunk - 1) // chunk, 1)
        self.nkeys = max(num_iters, 1) if trace else self.nchunks
        # behind the state of the shard, in the same allocation: what this rank contributes to the final all-gather --
        # [loss, id, theta] of the shard's winner (P + 2) and, with trace, the best objective of every step -- then the
        # per-chunk best-objective words (without trace) and the gathered rows of every rank: read back in ONE copy
        self.row = P + 2 + (self.nkeys if trace else 0)
        self.n_extra = self.row + (0 if trace else self.nkeys) + world * self.row
        self.st = ops.BatchedFitState(None, G, num_iters, extra_doubles=self.n_extra, n_keys=self.nkeys,
                                      keys_offset=(P + 2) if trace else self.row, B=Bl, device=device)
        extra = self.st.extra
        self.mine = extra[:self.row]
        self.packed = self.mine[:P + 2]
        self.keys = (self.mine[P + 2:] if trace else extra[self.row:self.row + self.nkeys]).view(torch.int64)
        self.key_views = None if trace else [self.keys[c:c + 1] for c in range(self.nchunks)]
        self.allp = extra[self.n_extra - world * self.row:].view(world, self.row)
        self.ev0, self.ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.chunk_events = [torch.cuda.Event() for _ in range(self.nchunks)] if world > 1 and not trace else None
        self.X_bytes = None

    def stage_X(self, X, Xh: np.ndarray) -> None:
        """X (host copy `Xh`) into the staging buffer, with the work that depends on its contents -- the training-flag
        check of a host X, the unique-row hint, the distinct-time bound and the structure cache -- once per distinct X."""
        from . import ops

        b = Xh.tobytes()
        if b == self.X_bytes:
            return
        ops._check_training_flags(X)   # returns early for a device-resident X (the caller's responsibility)
        st = self.st
        st.unique_hint, st.time_grid = ops.unique_rows(Xh), int(ops.distinct_times(Xh))
        ops._structure_cache(st, self.N, self.d_in.device)
        self.h_in[:3 * self.N] = Xh.reshape(-1)
        self.X_bytes = b


def multi_start_fit(X, y, theta0_all, jitter: float, *, num_iters: int = 150, lr: float = 0.01,
                    fix_params: bool = True, num_steps_per_epoch: int = 1000, chunk: Optional[int] = 1,
                    b1: float = 0.9, b2: float = 0.999, eps: float = 1e-8, trace: bool = False,
                    comm=None, queue_chunk: int = 10, variances=None) -> MultiStartResult:
    """Fit all restarts of this rank's shard on the current CUDA device.

    `theta0_all` is the (B, P) array of constrained start points of the WHOLE job (every rank passes
    the same array); the function slices its own shard.  `y` is (N,) -- B restarts of one data set -- or
    (B, N): LFM b fits y[b] on the shared design X (replicas, gene subsets of equal size, candidate transcription
    factors); the "winner" is then the LFM with the smallest final NLML over all data sets.  X, y and `variances` may be
    host arrays or CUDA tensors; a shape that fits none of these raises ValueError before any device work.

    Best-objective reduction across ranks (north_star: "one NCCL allreduce of best-objective ... state per step"):
      * ``trace=False``: `chunk` optimiser steps run per kernel launch; after every launch ONE device word (the
        atomicMin of the order-preserving image of every loss) is MIN-all-reduced on a side stream while the next
        launch is already running.  ``chunk=1`` is the literal per-step all-reduce; ``best_trace`` has one entry
        per chunk.
      * ``trace=True``: the kernels record the best objective of EVERY step in a device vector (`step_keys`,
        include/lfm_b200.h), the launches run `chunk` steps each (None: the whole fit in one launch), and the
        per-step reduction over ranks rides in the ONE all-gather that also moves the winners: ``best_trace``
        has one entry per step at the cost of a single collective per fit.
    `queue_chunk`: when the whole fit is one launch (``trace=True, chunk=None``) the kernels may run as persistent workers
    over a device-side queue of `queue_chunk`-step tasks (the queue mode of ``lfm_batched_fit_het``): used by the library
    where a static one-CTA-per-LFM assignment would leave SMs unevenly loaded (e.g. 512 LFMs per GPU), ignored
    elsewhere; 0 = never.
    `comm`: a ``dis_project_b200.comm.LfmComm`` -- the collectives then run through the C-ABI's own NCCL communicator
    (``lfm_comm_*``) and rank / world come from it; default: ``torch.distributed``.
    `variances`: None, or the measurement variances of the heteroscedastic objective, Sigma = K + diag(variances) +
    (jitter + sigma^2) I (the third output of ``dataset_3d``): (N,) / (N, 1) shared by every LFM, or (B, N) with one row
    per LFM, sliced per shard like `y` (``lfm_batched_fit_het``, include/lfm_b200.h).
    """
    import os
    import time

    import torch
    import torch.distributed as dist

    from . import ops

    theta0_all = np.asarray(theta0_all, dtype=np.float64)
    if theta0_all.ndim != 2 or theta0_all.shape[1] < 5 or (theta0_all.shape[1] - 2) % 3:
        raise ValueError(f"theta0_all must be (B, 3G+2) constrained start points, got {theta0_all.shape}")
    B, P = theta0_all.shape
    G = (P - 2) // 3
    if len(np.shape(X)) != 2 or np.shape(X)[1] != 3:
        raise ValueError(f"x must have shape (n, 3) = [time, gene_index, flag] (dataset.py:391), got {tuple(np.shape(X))}")
    N = int(np.shape(X)[0])
    per_lfm_y = ops._y_layout(np.shape(y), B, N) and B != 1
    per_lfm_var = variances is not None and ops._variance_layout(np.shape(variances), B, N)

    distributed = comm is not None or (dist.is_available() and dist.is_initialized())
    if comm is not None:
        rank, world = comm.rank, comm.world
    else:
        rank = dist.get_rank() if distributed else 0
        world = dist.get_world_size() if distributed else 1
    lo, hi = shard_bounds(B, rank, world)
    Bl = hi - lo
    if chunk is None or chunk <= 0:
        chunk = max(num_iters, 1)
    ops._lib.require_device()
    on_device = lambda a: isinstance(a, torch.Tensor) and a.is_cuda
    host = lambda a: np.asarray(a.detach().cpu() if isinstance(a, torch.Tensor) else a, dtype=np.float64)
    device = X.device if on_device(X) else torch.device("cuda", torch.cuda.current_device())
    timing = os.environ.get("LFM_MSF_TIMING") == "1"   # debug: synchronising phase timers (tools/batched_scale.py)
    tmarks = [time.perf_counter()]

    def mark():
        if timing:
            torch.cuda.synchronize()
            tmarks.append(time.perf_counter())

    key = (device.index if device.index is not None else torch.cuda.current_device(), N, G, Bl, per_lfm_y, num_iters, chunk,
           trace, world, variances is not None, per_lfm_var)
    plan = _PLANS.get(key)
    if plan is None:
        if len(_PLANS) > 8:
            _PLANS.clear()
        var_rows = 0 if variances is None else (Bl if per_lfm_var else 1)
        plan = _PLANS[key] = _Plan(device, N, G, Bl, per_lfm_y, num_iters, chunk, trace, world, var_rows)
    st = plan.st

    # host inputs are copied into the pinned staging buffer and cross PCIe in ONE copy; device-resident y / variances
    # are copied on the stream into their slots of the same device buffer, so the pointers bound below never change.
    # X always takes the staging path: its structure is counted on a host copy anyway.
    plan.stage_X(X, np.ascontiguousarray(host(X)))
    h = plan.h_in
    device_inputs = []
    for src, dst, off, per_lfm in ((y, plan.yd, plan.oy, per_lfm_y), (variances, plan.vd, plan.ov, per_lfm_var)):
        if dst is None:
            continue
        if on_device(src):
            device_inputs.append((dst, (src[lo:hi] if per_lfm else src).detach().reshape(-1)))
        else:
            h[off:off + dst.numel()] = (host(src)[lo:hi] if per_lfm else host(src)).reshape(-1)
    h[plan.oth:plan.oth + Bl * P] = theta0_all[lo:hi].reshape(-1)
    main = torch.cuda.current_stream()
    s = main.cuda_stream
    plan.ev0.record(main)
    plan.d_in.copy_(plan.pin_in, non_blocking=True)
    for dst, src in device_inputs:
        dst.copy_(src)
    st.reset(plan.th0)
    if Bl == 0:   # lfm_batched_fit_init rejects B = 0: an empty shard only resets its keys, then joins every collective
        plan.keys.fill_(torch.iinfo(torch.int64).max)
    launch = ops._bind_fit(st, plan.Xd, plan.yd, plan.y_stride, plan.vd, plan.var_stride, jitter, lr, b1, b2, eps,
                           fix_params, num_steps_per_epoch, plan.keys if trace else None,
                           queue_chunk if trace and chunk >= num_iters else 0)
    mark()
    multi = world > 1
    side = _side_stream(device) if multi and not trace else None
    keys_ptr = plan.keys.data_ptr()
    done = 0
    for c in range((num_iters + chunk - 1) // chunk):
        steps = min(chunk, num_iters - done)
        if Bl:
            launch(s, done, steps, None if trace else keys_ptr + 8 * c)
        done += steps
        if side is not None:
            e = plan.chunk_events[c]
            e.record(main)
            with torch.cuda.stream(side):
                side.wait_event(e)
                if comm is not None:
                    comm.allreduce_min_i64(plan.key_views[c], stream=side)
                else:
                    dist.all_reduce(plan.key_views[c], op=dist.ReduceOp.MIN)
    mark()
    if side is not None:
        main.wait_stream(side)
    # ---- global winner: one launch packs the shard's [loss, id, theta(P)], ONE all-gather, ONE device->host copy ------
    have = Bl > 0 and num_iters > 0
    ops.batched_best(st.hist if have else None, num_iters - 1 if have else 0, st.theta if have else None, float(lo),
                     plan.packed)
    gathered_on_host = None
    if multi:
        if comm is not None:
            comm.allgather_f64(plan.mine, plan.allp.view(-1))
        elif dist.get_backend() == "nccl":
            dist.all_gather_into_tensor(plan.allp.view(-1), plan.mine)
        else:  # gloo: gather on the host
            buf = [torch.empty(plan.row, dtype=torch.float64) for _ in range(world)]
            dist.all_gather(buf, plan.mine.cpu())
            gathered_on_host = torch.stack(buf).numpy()
    else:
        plan.allp[0].copy_(plan.mine)
    # ONE device->host copy of [theta | history | info | extra] into a pinned block of torch's caching host allocator;
    # the arrays handed back are views of it (they keep it alive), nothing is copied again on the host
    out = torch.empty(st.blob.numel(), dtype=torch.float64, pin_memory=True)
    out.copy_(st.blob, non_blocking=True)
    plan.ev1.record(main)
    main.synchronize()
    a = out.numpy()
    c0, c1, c2 = st._cuts
    theta = a[:c0].reshape(Bl, P)
    hist = a[c0:c1].reshape(st.hist.shape)
    info = a[c1:c2].view("int32")[:Bl]
    ex = a[c2:]
    row = plan.row
    allp_h = gathered_on_host if gathered_on_host is not None else ex[plan.n_extra - world * row:].reshape(world, row)
    if trace:
        keys_h = allp_h[:, P + 2:].copy().view(np.int64).min(axis=0)[:num_iters]   # MIN over ranks, per step
    else:
        keys_h = ex[row:row + plan.nkeys].view(np.int64)[:(num_iters + chunk - 1) // chunk]
    best = reduce_best_gathered(allp_h)
    best_id = int(best[1]) if np.isfinite(best[0]) else -1
    best_theta = None
    if best_id >= 0:
        owner = int(np.flatnonzero((allp_h[:, 0] == best[0]) & (allp_h[:, 1] == best[1]))[0])
        best_theta = allp_h[owner, 2:P + 2].copy()
    mark()
    if timing:
        global LAST_TIMING
        LAST_TIMING = [round(1e3 * (t1 - t0), 3) for t0, t1 in zip(tmarks[:-1], tmarks[1:])]
    device_ms = float(plan.ev0.elapsed_time(plan.ev1)) if Bl else float("nan")
    return MultiStartResult(theta, hist, info, lo, hi, float(best[0]), best_id, best_theta,
                            ops.loss_key_to_float(keys_h), device_ms)
