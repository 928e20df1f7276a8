"""Batched multi-start fits sharded over GPUs (BASELINE config 4; SURVEY.md 8e).

``B`` independent ``JaxTrainer.fit`` loops (reference ``src/trainer.py:162-228``) that share (X, y)
and differ in their start point.  Restart b lives on rank ``b * world // B`` (contiguous shards); no
data-path collective is needed because the restarts are independent.  One small all-reduce per
optimiser chunk keeps every rank informed of the global best objective (MIN over a packed
(loss, restart-id) key) and of a few SUM statistics; it runs on a side stream and is consumed one
chunk late so that it never sits on the critical path (NCCL over NVLink on the GPU box, gloo in the
CPU tests).
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


LAST_TIMING = None
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


def pack_best(loss: np.ndarray, ids: np.ndarray) -> np.ndarray:
    """(loss, id) pairs -> [best_loss, id_of_best] for a MIN all-reduce; NaN losses never win."""
    loss = np.where(np.isfinite(loss), loss, np.inf)
    if loss.size == 0:
        return np.array([np.inf, -1.0])
    k = int(np.argmin(loss))
    return np.array([loss[k], float(ids[k])])


def reduce_best(local: np.ndarray, dist=None):
    """All-reduce of the packed best: MIN on the loss, then MIN on the id among ranks that hold it."""
    import torch

    if dist is None or not dist.is_initialized() or dist.get_world_size() == 1:
        return local
    dev = "cuda" if dist.get_backend() == "nccl" else "cpu"
    t = torch.tensor([local[0]], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    best = float(t.item())
    cand = local[1] if local[0] == best else float("inf")
    t2 = torch.tensor([cand], dtype=torch.float64, device=dev)
    dist.all_reduce(t2, op=dist.ReduceOp.MIN)
    return np.array([best, float(t2.item())])


def reduce_best_gathered(allp: np.ndarray) -> np.ndarray:
    """Rows [loss, id, ...] gathered from every rank -> [best_loss, id_of_best]: MIN on the loss, then the
    smallest id among the rows that hold it (the same rule as `reduce_best`); NaN / inf never win."""
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


_STAGE = {}


def _stage_to_device(device, arrays):
    """Host arrays -> device views through ONE pinned staging buffer and ONE host->device copy (cached per size)."""
    import torch

    sizes = [int(a.size) for a in arrays]
    total = sum((n + 1) & ~1 for n in sizes)
    key = (device.index if device.index is not None else torch.cuda.current_device(), total)
    bufs = _STAGE.get(key)
    if bufs is None:
        if len(_STAGE) > 16:
            _STAGE.clear()
        bufs = (torch.empty(max(total, 2), dtype=torch.float64, pin_memory=True),
                torch.empty(max(total, 2), dtype=torch.float64, device=device))
        _STAGE[key] = bufs
    pinned, dbuf = bufs
    hp = pinned.numpy()
    views, off = [], 0
    for a, n in zip(arrays, sizes):
        hp[off:off + n] = np.asarray(a, dtype=np.float64).reshape(-1)
        views.append(dbuf[off:off + n].view(*a.shape))
        off += (n + 1) & ~1
    dbuf.copy_(pinned, non_blocking=True)
    return views


_PLANS = {}


class _MsfPlan:
    """Everything of one rank's share of a multi-start fit that depends on SHAPES only, built once and reused by every
    later fit of the same shape: the pinned staging buffer and its device twin ([X | y | start points], one copy), the
    fit state with the result rows behind it (one allocation, one read-back), the structure cache and task queue of
    the kernels, the events, and every pointer the C-ABI calls take.  What is left per fit on the host is three numpy
    copies into the staging buffer and five stream-ordered calls -- the fit kernel is in flight ~30 us after
    `multi_start_fit` is entered instead of ~200 us (`tools/msf_timeline.py`: the device used to wait for the host)."""

    def __init__(self, device, N, G, Bl, per_lfm_y, num_iters, chunk, trace, world, var_rows=0):
        """`var_rows`: 0 without measurement variances, 1 with one vector shared by the shard, Bl with one row per LFM:
        they ride in the same staging buffer and copy, [X | y | variances | start points]."""
        import torch

        from . import ops

        P = 3 * G + 2
        ev = lambda n: (int(n) + 1) & ~1
        ny = Bl * N if per_lfm_y else N
        nv = var_rows * N
        self.N, self.G, self.P, self.Bl, self.ny, self.num_iters, self.chunk, self.trace = N, G, P, Bl, ny, num_iters, chunk, trace
        self.oy, self.ov = ev(3 * N), ev(3 * N) + ev(ny)
        self.nv, self.oth = nv, self.ov + ev(nv)
        total = self.oth + ev(Bl * P)
        self.pin_in = torch.empty(total, dtype=torch.float64, pin_memory=True)
        self.h_in = self.pin_in.numpy()
        self.d_in = torch.empty(total, dtype=torch.float64, device=device)
        self.Xd = self.d_in[:3 * N].view(N, 3)
        self.yd = self.d_in[self.oy:self.oy + ny]
        self.vd = self.d_in[self.ov:self.ov + nv] if nv else None
        self.var_stride = N if var_rows > 1 else 0
        self.th0 = self.d_in[self.oth:self.oth + Bl * P].view(Bl, P)
        self.y_stride = N if per_lfm_y else 0
        self.nchunks = max((num_iters + chunk - 1) // chunk, 1)
        nkeys = max(num_iters, 1) if trace else self.nchunks
        row = P + 2 + (nkeys if trace else 0)
        self.row, self.nkeys = row, nkeys
        self.n_extra = row + (0 if trace else nkeys) + world * row
        key_off = (P + 2) if trace else row
        self.st = st = ops.BatchedFitState(None, G, num_iters, extra_doubles=self.n_extra, n_keys=nkeys, keys_offset=key_off,
                                           B=Bl, device=device)
        extra = st.extra
        self.mine = extra[:row]
        self.packed = self.mine[:P + 2]
        self.keys = (self.mine[P + 2:] if trace else extra[row:row + nkeys]).view(torch.int64)
        self.key_views = None if trace else [self.keys[c:c + 1] for c in range(self.nchunks)]
        self.allp = extra[self.n_extra - world * row:].view(world, row)
        self.allp_flat = self.allp.view(-1)
        self.ev0, self.ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.chunk_events = [torch.cuda.Event() for _ in range(self.nchunks)] if world > 1 and not trace else None
        self.X_bytes = None
        self.hint = self.tg = 0
        self.struct = None
        self.queue_ws, self.qb = None, 0

    def stage_X(self, Xh):
        """X into the staging buffer; the checks and counts that depend on its contents run once per distinct X."""
        import torch

        from . import ops

        b = Xh.tobytes()
        if b == self.X_bytes:
            return
        ops._check_training_flags(Xh)
        self.hint, self.tg = ops.unique_rows(Xh), int(ops.distinct_times(Xh))
        self.h_in[:3 * self.N] = Xh.reshape(-1)
        l = ops._lib.lib()
        nb = int(l.lfm_batched_structure_bytes(self.N, self.G, self.hint, self.tg))
        if self.struct is None or self.struct.numel() < max(nb, 16):
            self.struct = torch.empty(max(nb, 16), dtype=torch.uint8, device=self.d_in.device)
        self.X_bytes = b

    def queue(self, queue_chunk):
        import torch

        from . import ops

        qb = int(ops._lib.lib().lfm_batched_queue_bytes(self.Bl, self.num_iters, int(queue_chunk)))
        if qb > 0 and (self.queue_ws is None or self.queue_ws.numel() < qb):
            self.queue_ws = torch.empty(qb, dtype=torch.uint8, device=self.d_in.device)
        self.qb = qb
        return qb


def _msf_planned(Xh, yh, theta0_all, lo, hi, per_lfm_y, jitter, num_iters, lr, fix_params, num_steps_per_epoch, chunk,
                 b1, b2, eps, trace, comm, queue_chunk, dist, rank, world, device, timing, vh=None, per_lfm_var=False):
    """The host-buffer path of `multi_start_fit` over a cached `_MsfPlan` (same results, same collectives)."""
    import time

    import torch

    from . import ops

    B, P = theta0_all.shape
    G = (P - 2) // 3
    N = Xh.shape[0]
    Bl = hi - lo
    tmarks = [time.perf_counter()]

    def mark():
        if timing:
            torch.cuda.synchronize()
            tmarks.append(time.perf_counter())

    var_rows = 0 if vh is None else (Bl if per_lfm_var else 1)
    key = (device.index if device.index is not None else torch.cuda.current_device(), N, G, Bl, per_lfm_y, num_iters, chunk,
           trace, world, vh is not None, per_lfm_var)
    plan = _PLANS.get(key)
    if plan is None:
        if len(_PLANS) > 8:
            _PLANS.clear()
        plan = _PLANS[key] = _MsfPlan(device, N, G, Bl, per_lfm_y, num_iters, chunk, trace, world, var_rows)
    lib = ops._lib.lib()
    check = ops._lib.check
    st = plan.st
    plan.stage_X(Xh)
    h = plan.h_in
    h[plan.oy:plan.oy + plan.ny] = (yh[lo:hi] if per_lfm_y else yh).reshape(-1)
    if vh is not None:
        h[plan.ov:plan.ov + plan.nv] = (vh[lo:hi] if per_lfm_var else vh).reshape(-1)
    h[plan.oth:plan.oth + Bl * P] = theta0_all[lo:hi].reshape(-1)
    main = torch.cuda.current_stream()
    s = main.cuda_stream
    plan.ev0.record(main)
    plan.d_in.copy_(plan.pin_in, non_blocking=True)
    check(lib.lfm_batched_fit_init(s, Bl, G, plan.th0.data_ptr(), *st._init_tail), "lfm_batched_fit_init")
    mark()
    multi = world > 1
    side = _side_stream(device) if multi and not trace else None
    keys_ptr = plan.keys.data_ptr()
    common = (Bl, N, G, plan.Xd.data_ptr(), plan.yd.data_ptr(), plan.y_stride, st.u.data_ptr(), st.adam.data_ptr(),
              float(jitter), float(lr), float(b1), float(b2), float(eps))
    tail = (int(bool(fix_params)), int(num_steps_per_epoch), plan.hint, plan.tg, st.hist.data_ptr(), st.hist.shape[1],
            st.theta.data_ptr(), st.info.data_ptr())
    done = 0
    for c in range((num_iters + chunk - 1) // chunk):
        steps = min(chunk, num_iters - done)
        best_key = None if trace else keys_ptr + 8 * c
        step_keys = keys_ptr if trace else None
        qb = plan.queue(queue_chunk) if (trace and chunk >= num_iters and queue_chunk > 0 and done == 0) else 0
        if plan.vd is not None:   # one entry point for the chunked and the queue launches
            check(lib.lfm_batched_fit_het(s, *common[:6], plan.vd.data_ptr(), plan.var_stride, *common[6:], done, steps,
                                          num_iters, *tail, best_key, step_keys, plan.struct.data_ptr(),
                                          int(queue_chunk) if qb > 0 else 0, plan.queue_ws.data_ptr() if qb > 0 else None,
                                          qb), "lfm_batched_fit_het")
        elif qb > 0:
            check(lib.lfm_batched_fit_queue(s, *common, num_iters, *tail, best_key, step_keys, plan.struct.data_ptr(),
                                            int(queue_chunk), plan.queue_ws.data_ptr(), qb), "lfm_batched_fit_queue")
        else:
            check(lib.lfm_batched_fit_trace(s, *common, done, steps, num_iters, *tail, best_key, step_keys,
                                            plan.struct.data_ptr()), "lfm_batched_fit_trace")
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
    if num_iters > 0:
        check(lib.lfm_batched_best(s, Bl, P, st.hist.data_ptr(), st.hist.stride(0), num_iters - 1, st.theta.data_ptr(),
                                   float(lo), plan.packed.data_ptr()), "lfm_batched_best")
    else:
        check(lib.lfm_batched_best(s, 0, P, None, 1, 0, None, float(lo), plan.packed.data_ptr()), "lfm_batched_best")
    gathered_on_host = None
    if multi:
        if comm is not None:
            comm.allgather_f64(plan.mine, plan.allp_flat)
        elif dist.get_backend() == "nccl":
            dist.all_gather_into_tensor(plan.allp_flat, plan.mine)
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
    hist = a[c0:c1].reshape(Bl, -1)
    info = a[c1:c2].view("int32")[:Bl]
    ex = a[c2:]
    n_extra, row, nkeys = plan.n_extra, plan.row, plan.nkeys
    allp_h = gathered_on_host if gathered_on_host is not None else ex[n_extra - world * row:].reshape(world, row)
    if trace:
        keys_h = allp_h[:, P + 2:].copy().view(np.int64).min(axis=0)[:num_iters]   # MIN over ranks, per step
    else:
        keys_h = ex[row:row + nkeys].view(np.int64)[:(num_iters + chunk - 1) // chunk]
    best = reduce_best_gathered(allp_h)
    best_id = int(best[1]) if np.isfinite(best[0]) else -1
    best_theta = None
    if best_id >= 0:
        owner = int(np.flatnonzero((allp_h[:, 0] == best[0]) & (allp_h[:, 1] == best[1]))[0])
        best_theta = allp_h[owner, 2:P + 2].copy()
    mark()
    if timing:
        global LAST_TIMING
        LAST_TIMING = [round(1e3 * (b - a_), 3) for a_, b in zip(tmarks[:-1], tmarks[1:])]
    device_ms = float(plan.ev0.elapsed_time(plan.ev1))
    return MultiStartResult(theta, hist, info, lo, hi, float(best[0]), best_id, best_theta,
                            ops.loss_key_to_float(keys_h), device_ms)


def multi_start_fit(X, y, theta0_all, jitter: float, *, num_iters: int = 150, lr: float = 0.01,
                    fix_params: bool = True, num_steps_per_epoch: int = 1000, chunk: Optional[int] = 1,
                    b1: float = 0.9, b2: float = 0.999, eps: float = 1e-8, trace: bool = False,
                    comm=None, queue_chunk: int = 10, variances=None) -> MultiStartResult:
    """Fit all restarts of this rank's shard on the current CUDA device.

    `theta0_all` is the (B, P) array of constrained start points of the WHOLE job (every rank passes
    the same array); the function slices its own shard.  `y` is (N,) -- B restarts of one data set -- or
    (B, N): LFM b fits y[b] on the shared design X (replicas, gene subsets of equal size, candidate transcription
    factors); the "winner" is then the LFM with the smallest final NLML over all data sets.

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
    over a device-side queue of `queue_chunk`-step tasks (``lfm_batched_fit_queue``): used by the library where a static
    one-CTA-per-LFM assignment would leave SMs unevenly loaded (e.g. 512 LFMs per GPU), ignored elsewhere; 0 = never.
    `comm`: a ``dis_project_b200.comm.LfmComm`` -- the collectives then run through the C-ABI's own NCCL communicator
    (``lfm_comm_*``) and rank / world come from it; default: ``torch.distributed``.
    `variances`: None, or the measurement variances of the heteroscedastic objective, Sigma = K + diag(variances) +
    (jitter + sigma^2) I (the third output of ``dataset_3d``): (N,) / (N, 1) shared by every LFM, or (B, N) with one row
    per LFM, sliced per shard like `y` (``lfm_batched_fit_het``, include/lfm_b200.h).
    """
    import torch
    import torch.distributed as dist

    from . import ops

    import os
    import time
    timing = os.environ.get("LFM_MSF_TIMING") == "1"   # debug: synchronising phase timers (tools/batched_scale.py)
    tmarks = [time.perf_counter()]

    def mark():
        if timing:
            torch.cuda.synchronize()
            tmarks.append(time.perf_counter())

    distributed = comm is not None or (dist.is_available() and dist.is_initialized())
    if comm is not None:
        rank, world = comm.rank, comm.world
    else:
        rank = dist.get_rank() if distributed else 0
        world = dist.get_world_size() if distributed else 1
    theta0_all = np.asarray(theta0_all, dtype=np.float64)
    B, P = theta0_all.shape
    G = (P - 2) // 3
    lo, hi = shard_bounds(B, rank, world)
    if chunk is None or chunk <= 0:
        chunk = max(num_iters, 1)
    ops._lib.require_device()
    device = X.device if isinstance(X, torch.Tensor) and X.is_cuda else torch.device("cuda", torch.cuda.current_device())
    yh = y if isinstance(y, torch.Tensor) else np.asarray(y, dtype=np.float64)
    per_lfm_y = yh.ndim == 2 and yh.shape[0] == B and yh.shape[1] == (X.shape[0]) and B != 1
    vh, per_lfm_var = None, False
    if variances is not None:
        vh = variances if isinstance(variances, torch.Tensor) else np.asarray(variances, dtype=np.float64)
        per_lfm_var = ops._variance_layout(vh.shape, B, X.shape[0])
    host_inputs = not isinstance(X, torch.Tensor) and not isinstance(yh, torch.Tensor) and not isinstance(vh, torch.Tensor)
    hint = tg = None
    if host_inputs and hi > lo and os.environ.get("LFM_MSF_PLAN", "1") != "0":
        Xh = np.ascontiguousarray(np.asarray(X, dtype=np.float64))
        if Xh.ndim != 2 or Xh.shape[1] != 3:
            raise ValueError(f"x must have shape (n, 3) = [time, gene_index, flag] (dataset.py:391), got {Xh.shape}")
        return _msf_planned(Xh, yh, theta0_all, lo, hi, per_lfm_y, jitter, num_iters, lr, fix_params, num_steps_per_epoch,
                            chunk, b1, b2, eps, trace, comm, queue_chunk, dist if distributed and comm is None else None,
                            rank, world, device, timing, vh, per_lfm_var)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    if host_inputs:
        # everything this rank needs crosses PCIe in ONE copy: X, its observations, its start points
        Xh = np.ascontiguousarray(np.asarray(X, dtype=np.float64))
        ops._check_training_flags(Xh)
        hint, tg = ops.unique_rows(Xh), ops.distinct_times(Xh)  # from the host copy: no device->host round trip
        ysel = np.ascontiguousarray(yh[lo:hi]) if per_lfm_y else yh.reshape(-1)
        staged = [Xh, ysel, np.ascontiguousarray(theta0_all[lo:hi])]
        if vh is not None:
            staged.append(np.ascontiguousarray(vh[lo:hi]) if per_lfm_var else vh.reshape(-1))
        Xd, yd, th0, *vd = _stage_to_device(device, staged)
        vd = vd[0] if vd else None
        Xd = ops._rows3(Xd, "x")
    else:
        Xd = ops._rows3(X, "x")
        yd = ops._dev(yh[lo:hi]) if per_lfm_y else ops._dev(yh).reshape(-1)
        th0 = theta0_all[lo:hi]
        vd = None if vh is None else (ops._dev(vh[lo:hi]) if per_lfm_var else ops._dev(vh).reshape(-1))
    nchunks = max((num_iters + chunk - 1) // chunk, 1)
    nkeys = max(num_iters, 1) if trace else nchunks
    # behind the state of the shard, in the same allocation: what this rank contributes to the final all-gather --
    # [loss, id, theta] of the shard's winner (P + 2) and, with trace, the best objective of every step -- then the
    # per-chunk best-objective words (without trace) and the gathered rows of every rank: read back in ONE copy
    row = P + 2 + (nkeys if trace else 0)
    n_extra = row + (0 if trace else nkeys) + world * row
    key_off = (P + 2) if trace else row
    st = ops.BatchedFitState(th0, G, num_iters, extra_doubles=n_extra, n_keys=nkeys, keys_offset=key_off) if hi > lo else None
    if st is not None and hint is not None:
        st.unique_hint, st.time_grid = hint, tg
    extra = st.extra if st is not None else torch.empty(n_extra, dtype=torch.float64, device=device)
    mine = extra[:row]
    packed = mine[:P + 2]
    keys = (mine[P + 2:] if trace else extra[row:row + nkeys]).view(torch.int64)
    if st is None:
        keys.fill_(torch.iinfo(torch.int64).max)   # (with a shard the state's initialisation launch has done it)
    allp = extra[n_extra - world * row:].view(world, row)
    main = torch.cuda.current_stream()
    multi = distributed and world > 1
    side = _side_stream(device) if multi and not trace else None
    done = 0
    mark()
    for c in range((num_iters + chunk - 1) // chunk):
        steps = min(chunk, num_iters - done)
        if st is not None:
            ops.batched_fit_steps(st, Xd, yd, jitter, steps, lr=lr, b1=b1, b2=b2, eps=eps, fix_params=fix_params,
                                  steps_per_epoch=num_steps_per_epoch, best_key=None if trace else keys[c:c + 1],
                                  step_keys=keys if trace else None,
                                  queue_chunk=queue_chunk if trace and chunk >= num_iters else 0, variances=vd)
        done += steps
        if side is not None:
            ev = torch.cuda.Event()
            ev.record(main)
            with torch.cuda.stream(side):
                side.wait_event(ev)
                if comm is not None:
                    comm.allreduce_min_i64(keys[c:c + 1], stream=side)
                else:
                    dist.all_reduce(keys[c:c + 1], op=dist.ReduceOp.MIN)
    mark()
    if side is not None:
        main.wait_stream(side)
    # ---- global winner: one launch packs the shard's [loss, id, theta(P)], ONE all-gather, ONE device->host copy ------
    have = st is not None and num_iters > 0
    ops.batched_best(st.hist if have else None, num_iters - 1 if have else 0, st.theta if have else None, float(lo), packed)
    gathered_on_host = None
    if multi:
        if comm is not None:
            comm.allgather_f64(mine, allp.view(-1))
        elif dist.get_backend() == "nccl":
            dist.all_gather_into_tensor(allp.view(-1), mine)
        else:  # gloo (CPU tests): gather on the host
            buf = [torch.empty(row, dtype=torch.float64) for _ in range(world)]
            dist.all_gather(buf, mine.cpu())
            gathered_on_host = torch.stack(buf).numpy()
    else:
        allp[0].copy_(mine)
    if st is not None:
        theta, hist, info, ex = ops.batched_to_host(st, after_copy=ev1)
    else:
        theta, hist, info = np.zeros((0, P)), np.zeros((0, num_iters)), np.zeros(0, dtype=np.int32)
        ex = extra.cpu().numpy()
    allp_h = gathered_on_host if gathered_on_host is not None else ex[n_extra - world * row:].reshape(world, row)
    if trace:
        keys_h = allp_h[:, P + 2:].copy().view(np.int64).min(axis=0)[:num_iters]   # MIN over ranks, per step
    else:
        keys_h = ex[row:row + nkeys].view(np.int64)[:(num_iters + chunk - 1) // chunk]
    best = reduce_best_gathered(allp_h)
    best_id = int(best[1]) if np.isfinite(best[0]) else -1
    best_theta = None
    if best_id >= 0:
        owner = int(np.flatnonzero((allp_h[:, 0] == best[0]) & (allp_h[:, 1] == best[1]))[0])
        best_theta = allp_h[owner, 2:P + 2].copy()
    mark()
    if timing:
        global LAST_TIMING
        LAST_TIMING = [round(1e3 * (b - a), 3) for a, b in zip(tmarks[:-1], tmarks[1:])]
    device_ms = float(ev0.elapsed_time(ev1)) if st is not None else float("nan")
    return MultiStartResult(theta, hist, info, lo, hi, float(best[0]), best_id, best_theta,
                            ops.loss_key_to_float(keys_h), device_ms)
