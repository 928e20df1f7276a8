#!/usr/bin/env python
"""Benchmark of the LFM hot path (BASELINE.json metric: NLML+grad evaluations / second, fp64).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload at every N: BASELINE config 2, synthetic LFM 50 genes x 80 time points (N = 4000), one
"step" = one NLML + gradient evaluation at the reference's initial hyper-parameters.  A single
large-N evaluation does not shard (north_star: "no cross-GPU split"), so --gpus N runs N independent
replicas (weak scaling, no data-path collective); the batched multi-start path, which does shard,
is reported beside it under "secondary" (4096 p53-shaped restarts x 150 Adam steps over all ranks
with its best-objective all-reduce every 10 steps and every step, median of 7), together with the N = 32768
evaluation (config 3, 3 repetitions, its own roofline object) and the 102 400-point posterior (config 5) on rank 0.

`--impl reference` times the CPU restatement of the reference (oracle/, numpy/scipy/LAPACK with all
host threads) on the same config; rank 0 only.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

if "reference" in sys.argv[1:]:
    # The CPU arm uses every host core.  torch.distributed.run exports OMP_NUM_THREADS=1 to its workers, which would
    # throttle LAPACK inside the oracle (round 1: 1.19 -> 0.66 evaluations/s under torchrun): restore the thread
    # counts BEFORE numpy / scipy load their BLAS, so that the reference arm is the same measurement at every --gpus N.
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        os.environ[_v] = str(os.cpu_count() or 1)

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

G_C2, T_C2 = 50, 80          # config 2: N = 4000
G_C3, T_C3 = 256, 128        # config 3: N = 32768
JITTER = 1e-4
METRIC = "LFM NLML+grad evals/sec (fp64), N=4000 (50 genes x 80 time points)"
UNIT = "evals/s"
CONFIG = {"workload": "config 2: synthetic LFM 50 genes x 80 time points (N=4000), NLML+grad at the reference's "
                      "initial hyper-parameters", "N": 4000, "G": G_C2, "T": T_C2,
          "launch": "one CUDA-graph replay per evaluation (ops.NlmlGradPlan / lfm_plan_launch); e2e: lfm_nlml_grad_host",
          "parallelism": "replicas only (one independent LFM per GPU; a single large-N Cholesky does not shard)",
          "l2": "256 MB buffer written between timed iterations (L2 flush); working set 268 MB > 126 MB L2",
          "scheduling": "factorisation streams in green contexts when the driver exports them (8-SM chain partition, 140-SM "
                        "bulk partition with panel, early-update, late-update, inverse and filler streams at three priorities, 88-SM sub-partition for the top-node product of the inverse; LFM_SM_PARTITION=0 "
                        "= stream priorities only)"}


# synthetic inputs built here so that the product arm never imports oracle/
class _Inputs:
    @staticmethod
    def make_problem(G, T, seed=42):
        times = np.linspace(0.0, 12.0, T)
        X = np.stack((np.tile(times, G), np.repeat(np.arange(G), T).astype(np.float64), np.ones(G * T)), axis=-1)
        rng = np.random.default_rng(seed)
        d = rng.uniform(0.2, 1.0, G)
        b = rng.uniform(0.01, 0.1, G)
        # y = mean + smooth latent response + unit noise: cheap O(N) draw with the right scales
        f = np.interp(times, np.linspace(0, 12, 7), [0.18, 1.18, 1.62, 0.82, 0.69, -0.18, 0.51])
        y = np.repeat(b / d, T) + np.tile(f, G) * np.repeat(rng.uniform(0.5, 1.5, G), T) + rng.standard_normal(G * T)
        theta = np.concatenate([np.full(G, 0.4), np.full(G, 1.0), np.full(G, 0.05), [2.5, 1.0]])
        return X, y, theta



def clocks_start(path):
    q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    try:
        fh = open(path, "w")
        return subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                stdout=fh, stderr=subprocess.DEVNULL)
    except Exception:
        return None


def clocks_parse(path, dev_index):
    sm, mx, reasons = [], [], set()
    try:
        for line in open(path):
            p = [c.strip() for c in line.split(",")]
            if len(p) < 9 or not p[0].isdigit() or int(p[0]) != dev_index:
                continue
            sm.append(float(p[1])); mx.append(float(p[2]))
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
    except Exception:
        pass
    if not sm:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
    # "under load": the upper half of the samples (idle samples before/after the region drop out)
    load = sorted(sm)[len(sm) // 2:]
    return {"sm_mhz": float(np.median(load)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
            "samples": len(sm)}


def dump_outputs(path, nlml_grad, info):
    """--dump-outputs: what the last timed step returned, as float64 .npy files.  The inputs are seeded, so two builds
    (or a build and --impl reference) can be compared output for output."""
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "nlml_grad.npy"), np.asarray(nlml_grad, dtype=np.float64).reshape(-1))
    np.save(os.path.join(path, "info.npy"), np.asarray(info, dtype=np.float64).reshape(-1))


def run_reference(args):
    """CPU arm: the oracle restatement of the reference path on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import lfm_oracle as o
    X, y, theta = _Inputs.make_problem(G_C2, T_C2)
    p = o.Params.unpack(theta, JITTER)
    cores = os.cpu_count() or 1
    blas_threads = None
    try:  # belt and braces: if a BLAS was already initialised with fewer threads, raise its limit
        import threadpoolctl
        threadpoolctl.threadpool_limits(limits=cores)
        blas_threads = max([m.get("num_threads", 0) for m in threadpoolctl.threadpool_info()] or [0])
    except Exception:
        pass
    for _ in range(args.warmup):
        o.nlml_and_grad(p, X, y, threads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        v, g = o.nlml_and_grad(p, X, y, threads=cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, np.concatenate([[v], g]), 0)   # the oracle raises where the device reports info > 0
    val = args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "steps_executed": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": CONFIG,
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "blas_threads": blas_threads, "kind": "port",
                             "sample": f"{args.steps} full NLML+grad evaluations at N=4000 (oracle/lfm_oracle.py, "
                                       "numpy+scipy+LAPACK, row chunks over all host threads)"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-secondary", action="store_true", help="skip the batched / N=32768 secondary measurements")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (rank 0) as float64 .npy files to DIR: "
                         "nlml_grad.npy (NLML, then the gradient) and info.npy (factorisation status, 0 = success)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # stdout carries ONE JSON line: NCCL prints its version banner to stdout while the communicator comes
        # up (whenever NCCL_DEBUG >= VERSION), so fd 1 points at stderr until the first collective has run
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    from dis_project_b200 import _lib, ops
    from dis_project_b200.batched import make_restarts, multi_start_fit
    from dis_project_b200.dataset import JaxP53Data, dataset_3d

    _lib.require_device()
    lib = _lib.lib()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- inputs resident in HBM --------------------------------------------------------------------
    Xh, yh, thh = _Inputs.make_problem(G_C2, T_C2, seed=42 + rank)  # every replica its own data
    N = Xh.shape[0]
    P = 3 * G_C2 + 2
    X, y, th = (torch.as_tensor(a).to(dev) for a in (Xh, yh, thh))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    # the public API for repeated evaluations at fixed (X, y): a CUDA-graph evaluation plan (what JaxTrainer's
    # objective uses); every step writes theta into the bound buffer and replays ~270 kernel launches
    plan = ops.NlmlGradPlan(X, y, G_C2, JITTER)

    def step():
        return plan(th)

    # ---- FP64 roofline denominator: cuBLAS Dgemm, measured here (MEASURED_PEAKS.json has no FP64 entry) ----
    peak_tf = None
    if rank == 0:
        n = 8192
        A = torch.randn(n, n, dtype=torch.float64, device=dev)
        Bm = torch.randn(n, n, dtype=torch.float64, device=dev)
        torch.matmul(A, Bm)
        best = 1e9
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch.matmul(A, Bm); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1) * 1e-3)
        peak_tf = 2 * n**3 / best / 1e12
        del A, Bm
        torch.cuda.empty_cache()

    # ---- warm-up, then the timed region ---------------------------------------------------------------
    for _ in range(args.warmup):
        out, info = step()
    torch.cuda.synchronize()
    assert int(info.item()) == 0 and bool(torch.isfinite(out).all()), "warm-up evaluation failed"
    clk_path = os.path.join(tempfile.gettempdir(), f"lfm_clocks_{rank}.csv")
    clk = clocks_start(clk_path) if rank == 0 else None
    time.sleep(0.3 if clk else 0.0)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    launches0 = lib.lfm_debug_launch_count()
    wall0 = time.perf_counter()
    for e0, e1 in evs:
        flush.zero_()           # L2 flush between timed iterations (outside the per-step events)
        e0.record()
        out, info = step()
        e1.record()
    barrier()
    wall = time.perf_counter() - wall0
    launches = lib.lfm_debug_launch_count() - launches0
    dev_s = sum(e0.elapsed_time(e1) for e0, e1 in evs) * 1e-3
    dev_s = max_over_ranks(dev_s)
    value = world * args.steps / dev_s
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out.cpu().numpy(), info.cpu().numpy())

    # ---- e2e: the host-buffer C-ABI call (H2D of X, y, theta and D2H of NLML+grad inside the timed region) ----
    import ctypes as C
    h = C.c_void_p()
    _lib.check(lib.lfm_handle_create(C.byref(h)), "lfm_handle_create")
    out_h = np.empty(1 + P)
    info_h = C.c_int(0)

    def host_step():
        _lib.check(lib.lfm_nlml_grad_host(h, N, G_C2, Xh.ctypes.data, yh.ctypes.data, thh.ctypes.data, JITTER, 0,
                                          out_h.ctypes.data, C.byref(info_h)), "lfm_nlml_grad_host")

    for _ in range(args.warmup):
        host_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        host_step()
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    e2e_val = world * args.steps / e2e_s
    assert abs(out_h[0] - float(out[0].item())) <= 1e-9 * abs(out_h[0]), "host and device entry points disagree"
    lib.lfm_handle_destroy(h)
    if clk:
        clk.terminate(); clk.wait()

    # ---- roofline of the dominant kernel (lfm_dgemm_kernel, DMMA): CUDA events around every launch -----------
    roof = None
    if rank == 0:
        lib.lfm_debug_profile_begin()
        pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        pe0.record()
        for _ in range(args.steps):
            ops.nlml_grad(X, y, th, JITTER, G_C2)   # stream launches: per-launch events cannot be taken inside a graph
        pe1.record()
        ms, fl, nl = C.c_double(0), C.c_double(0), C.c_longlong(0)
        _lib.check(lib.lfm_debug_profile_end(C.byref(ms), C.byref(fl), C.byref(nl)), "profile_end")
        cms, cfl, cnl = C.c_double(0), C.c_double(0), C.c_longlong(0)
        _lib.check(lib.lfm_debug_profile_chain(C.byref(cms), C.byref(cfl), C.byref(cnl)), "profile_chain")
        # SURVEY 8(d): N^3/3 (POTRF) + 2N^3/3 (explicit inverse) algorithmic FLOP per evaluation.  The 16 x 128-tile
        # launches of the look-ahead chain are a separate instantiation (8 CTAs, latency-bound by design); their
        # share of the algorithmic flops is removed from the numerator and their time reported beside it.
        alg_flops = float(N) ** 3
        exec_total = fl.value + cfl.value
        alg_bulk = alg_flops * (fl.value / exec_total) if exec_total > 0 else alg_flops
        gemm_s = ms.value * 1e-3 / args.steps
        achieved = alg_bulk / gemm_s / 1e12
        # DRAM traffic cannot be measured outside a profiler: the figure is the ncu --set full capture committed under
        # profiles/ (newest round available), labelled as such
        traffic, traffic_src = None, None
        for name in ("roofline_r2.json", "roofline_r1.json"):
            try:
                traffic = json.load(open(os.path.join(ROOT, "profiles", name))).get("dgemm_dram_bytes_per_launch")
                traffic_src = f"profiles/{name} (ncu --set full: dram__bytes_read.sum + dram__bytes_write.sum averaged over the " \
                              "GEMM launches of one evaluation; not measured in this run)"
                break
            except Exception:
                continue
        prof_step_s = pe0.elapsed_time(pe1) * 1e-3 / args.steps
        roof = {"bound": "tensor", "kernel": "lfm_dgemm_kernel (mma.sync m8n8k4 f64 = SASS DMMA), bulk tile variants",
                "achieved": achieved,
                "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf if peak_tf else None, "traffic": traffic,
                "traffic_source": traffic_src,
                "traffic_note": "both N x N matrices of an evaluation (2 x 134 MB) cycle through the 126 MB L2 between launches; the "
                                "GEMM launches of one evaluation move about 3.5x the 8 N^2 = 128 MB algorithmic bytes through DRAM, "
                                "which at the measured HBM rate is ~70 us of a 3.4 ms step: not the bound, the DMMA pipe and the "
                                "dependent chain of the factorisation are",
                "peak_source": "cuBLAS Dgemm 8192^3 best of 5, measured in this run (MEASURED_PEAKS.json has no FP64 figure)",
                "algorithmic_flops_per_eval": alg_flops, "algorithmic_flops_in_these_launches": alg_bulk,
                "executed_flops_per_eval": fl.value / args.steps,
                "launches_per_eval": nl.value / args.steps, "kernel_s_per_eval": gemm_s,
                "kernel_share_of_step": gemm_s / prof_step_s,
                "profiled_pass_ms_per_eval": prof_step_s * 1e3,
                "profiled_pass_note": "the share is taken inside the PROFILED pass: stream launches with two event records per GEMM "
                                      "launch, issued from Python -- that pass is host-launch-bound (its time per evaluation is "
                                      "beside this note and varies with the box's host, 3.6-5.4 ms against the ~3.2 ms of a "
                                      "graph replay), so the share moves between ~0.6 and ~0.9 while kernel_s_per_eval does not",
                "kernel_s_per_eval_summed": lib.lfm_debug_profile_sum_ms() * 1e-3 / args.steps,
                "note": "the factorisation launches on several streams and launches overlap: kernel_s_per_eval is the "
                        "length of the union of the launch intervals (CUDA-event timestamps), the plain sum is beside it",
                "chain_tile_launches": {"kernel": "lfm_dgemm_kernel<.,.,1,4,2> (16 x 128 tiles; only with LFM_CHAIN_FUSED=0 -- by "
                                                  "default the chain step is lfm_chain_step_kernel, one 8-CTA cluster "
                                                  "launch per 128 columns, outside this accounting)",
                                        "launches_per_eval": cnl.value / args.steps,
                                        "kernel_s_per_eval": cms.value * 1e-3 / args.steps,
                                        "executed_flops_per_eval": cfl.value / args.steps},
                "step_tflops": alg_flops / (dev_s / args.steps) / 1e12,
                "step_frac_of_peak": alg_flops / (dev_s / args.steps) / 1e12 / peak_tf if peak_tf else None}

    # ---- secondary: batched multi-start (config 4, sharded) and N = 32768 (configs 3 and 5) -------------------
    def stats(xs):
        xs = sorted(xs)
        return {"median": float(np.median(xs)), "min": xs[0], "max": xs[-1], "repetitions": len(xs)}

    secondary = {}
    if not args.no_secondary:
        data = JaxP53Data.synthetic()
        xb, yb, _ = dataset_3d(data)
        TH = make_restarts(np.concatenate([np.full(5, 0.4), np.ones(5), np.full(5, 0.05), [2.5, 1.0]]), 4096)
        secondary["batched"] = {}
        # the collectives of the sharded path run through the C-ABI's own NCCL communicator (lfm_comm_*, include/lfm_b200.h),
        # its id broadcast over the process group; measured at 8 GPUs (tools/msf_modes.py): 4.59 ms against 4.79 ms through
        # torch.distributed for the same fit
        lcomm = None
        if world > 1:
            from dis_project_b200.comm import LfmComm
            lcomm = LfmComm.from_torch_distributed()
        # chunk = 10: best-objective all-reduce every 10 optimiser steps; chunk = 1: every step (north_star: "one NCCL
        # allreduce of best-objective ... state per step").  Median of 7 after a full-size warm-up each.
        modes = (("chunk10", dict(chunk=10), "best-objective MIN all-reduce (8 bytes, side stream) every 10 optimiser steps"),
                 ("chunk1", dict(chunk=1), "best-objective MIN all-reduce every optimiser step (north_star's literal wording): "
                                           "one launch + one collective per step"),
                 ("trace", dict(chunk=None, trace=True), "best objective of EVERY step recorded by the kernels (step_keys), whole "
                                                         "fit in one launch, the per-step reduction over ranks rides in the ONE "
                                                         "all-gather that moves the winners"))
        for name, kw, what in modes:
            multi_start_fit(xb, yb.reshape(-1), TH, JITTER, num_iters=150, comm=lcomm, **kw)   # allocator, pinned buffers, NCCL
            times, dev_times = [], []
            for _ in range(7):
                barrier()
                t0 = time.perf_counter()
                res = multi_start_fit(xb, yb.reshape(-1), TH, JITTER, num_iters=150, comm=lcomm, **kw)
                times.append(max_over_ranks(time.perf_counter() - t0))
                dev_times.append(max_over_ranks(res.device_ms * 1e-3))
            st_ = stats(times)
            secondary["batched"][name] = {
                "workload": "config 4: 4096 p53-shaped restarts (N=105, G=5) x 150 Adam steps, sharded over "
                            f"{world} GPU(s); {what}",
                "seconds": st_, "device_seconds": stats(dev_times),
                "restarts_per_s": 4096 / st_["median"], "evals_per_s": 4096 * 150 / st_["median"],
                "best_nlml": res.best_loss, "restarts_per_gpu": res.hi - res.lo, "best_trace_entries": int(res.best_trace.shape[0]),
                "collectives": "lfm_comm_* (C-ABI, NCCL)" if lcomm is not None else "none (one GPU)",
                "warps_per_lfm": int(_lib.lib().lfm_batched_team_size(
                    res.hi - res.lo, xb.shape[0], 5, ops.unique_rows(xb), ops.distinct_times(xb))),
                "timed": "seconds: host wall clock around multi_start_fit (host buffers in, numpy results out, barrier before, "
                         "max over ranks), median of 7; device_seconds: CUDA events on the launching stream from the first "
                         "enqueued operation (host-to-device copy of this rank's inputs) to the last (device-to-host copy of its "
                         "results), max over ranks, same 7 runs"}
        # kept at the top level for continuity with round 1 (chunk = 10)
        secondary["batched"].update({k: secondary["batched"]["chunk10"][k] for k in ("restarts_per_s", "evals_per_s", "best_nlml",
                                                                                     "restarts_per_gpu", "warps_per_lfm")})
        secondary["batched"]["seconds"] = secondary["batched"]["chunk10"]["seconds"]["median"]
        if lcomm is not None:
            lcomm.close()
        if rank == 0:
            try:
                X3h, y3h, th3h = _Inputs.make_problem(G_C3, T_C3)
                X3, y3, th3 = (torch.as_tensor(a).to(dev) for a in (X3h, y3h, th3h))
                N3 = float(X3h.shape[0])
                ops.nlml_grad(X3, y3, th3, JITTER, G_C3)
                torch.cuda.synchronize()
                t3 = []
                for _ in range(3):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(); o3, i3 = ops.nlml_grad(X3, y3, th3, JITTER, G_C3); e1.record(); torch.cuda.synchronize()
                    t3.append(e0.elapsed_time(e1) * 1e-3)
                st3 = stats(t3)
                s3 = st3["median"]
                # one more evaluation with CUDA events around every GEMM launch: the roofline object of config 3
                lib.lfm_debug_profile_begin()
                pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                pe0.record(); ops.nlml_grad(X3, y3, th3, JITTER, G_C3); pe1.record()
                ms3, fl3, nl3 = C.c_double(0), C.c_double(0), C.c_longlong(0)
                _lib.check(lib.lfm_debug_profile_end(C.byref(ms3), C.byref(fl3), C.byref(nl3)), "profile_end")
                vbuf = C.create_string_buffer(1 << 14)
                lib.lfm_debug_profile_variants(vbuf, len(vbuf))
                variants = json.loads(vbuf.value.decode() or "[]")
                for v in variants:
                    v["tflops_executed"] = v["executed_flops"] / (v["ms_sum"] * 1e-3) / 1e12 if v["ms_sum"] > 0 else None
                prof_s = pe0.elapsed_time(pe1) * 1e-3
                ach3 = N3**3 / s3 / 1e12
                secondary["n32768"] = {
                    "workload": "config 3: 256 genes x 128 time points (N=32768) NLML+grad",
                    "evals_per_s": 1.0 / s3, "seconds": st3, "dense_tflops": ach3,
                    "frac_of_dgemm_peak": ach3 / peak_tf if peak_tf else None,
                    "info": int(i3.item()), "finite": bool(torch.isfinite(o3).all()),
                    "roofline": {"bound": "tensor", "kernel": "lfm_dgemm_kernel<.,.,4,4,4> (128 x 128 tiles, 16 warps; DMMA)",
                                 "achieved": ach3, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach3 / peak_tf if peak_tf else None,
                                 "achieved_definition": "algorithmic N^3 FLOP of an evaluation / median evaluation time (whole step: "
                                                        "Sigma build, gradient contraction and reductions included in the time)",
                                 "algorithmic_flops_per_eval": N3**3, "executed_flops_gemm": fl3.value,
                                 "gemm_launches": nl3.value, "gemm_kernel_s_union": ms3.value * 1e-3,
                                 "gemm_share_of_step": ms3.value * 1e-3 / prof_s, "profiled_step_s": prof_s,
                                 "gemm_tflops_executed": fl3.value / (ms3.value * 1e-3) / 1e12 if ms3.value > 0 else None,
                                 "by_variant": variants, "traffic": None,
                                 "peak_source": "cuBLAS Dgemm 8192^3 best of 5, measured in this run"}}
                # config 5: latent posterior mean / variance at 102 400 test times from the same N = 32768 LFM
                TS = 102400
                Xs = torch.stack((torch.linspace(0, 13, TS, dtype=torch.float64, device=dev),
                                  torch.full((TS,), -1.0, dtype=torch.float64, device=dev),
                                  torch.zeros(TS, dtype=torch.float64, device=dev)), dim=1).contiguous()
                var3 = torch.as_tensor(np.random.default_rng(7).uniform(0.01, 0.1, X3h.shape[0])).to(dev)
                ops.release_workspaces()
                torch.cuda.empty_cache()
                ops.latent_posterior(X3, y3, var3, th3, JITTER, Xs[:4096], G_C3)  # warm-up (small T*)
                torch.cuda.synchronize()
                t5 = []
                for _ in range(2):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(); pm, pv, pi = ops.latent_posterior(X3, y3, var3, th3, JITTER, Xs, G_C3); e1.record()
                    torch.cuda.synchronize()
                    t5.append(e0.elapsed_time(e1) * 1e-3)
                st5 = stats(t5)
                s5 = st5["median"]
                fl5 = 32768.0**2 * TS + 2.0 * 32768.0**3 / 3.0
                secondary["posterior_100k"] = {
                    "workload": "config 5: latent posterior mean+variance at 102400 test times from the N=32768 LFM "
                                "(factorisation + inverse factor included)",
                    "seconds": st5, "test_points_per_s": TS / s5, "dense_tflops": fl5 / s5 / 1e12,
                    "frac_of_dgemm_peak": fl5 / s5 / 1e12 / peak_tf if peak_tf else None, "info": int(pi.item()),
                    "finite": bool(torch.isfinite(pm).all() and torch.isfinite(pv).all()),
                    "var_min": float(pv.min().item()), "var_max": float(pv.max().item())}
                del X3, y3, th3, Xs, var3
                ops.release_workspaces()
                torch.cuda.empty_cache()
            except Exception as exc:  # pragma: no cover
                secondary["n32768"] = {"error": repr(exc)}
        try:   # oracle parity of configs 3 and 5 at full size, measured by tools/fullsize_parity.py (minutes of CPU time)
            secondary["fullsize_parity"] = dict(json.load(open(os.path.join(ROOT, "profiles", "fullsize_parity_r2.json"))),
                                                source="profiles/fullsize_parity_r2.json (tools/fullsize_parity.py; not re-run here)")
        except Exception:
            pass
        barrier()

    # ---- CPU baseline beside it (rank 0, N = 1 only) -----------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import lfm_oracle as o
        cores = os.cpu_count() or 1
        pc = o.Params.unpack(thh, JITTER)
        o.nlml_and_grad(pc, Xh, yh, threads=cores)
        t0 = time.perf_counter()
        reps = 2
        for _ in range(reps):
            vc, gc = o.nlml_and_grad(pc, Xh, yh, threads=cores)
        ct = (time.perf_counter() - t0) / reps
        cpu = {"value": 1.0 / ct, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{reps} full NLML+grad evaluations at N=4000 (oracle/lfm_oracle.py: numpy/scipy/LAPACK, all host threads)",
               "parity_rel_err_nlml": abs(vc - out_h[0]) / abs(vc),
               "parity_rel_err_grad": float(np.max(np.abs(gc - out_h[1:])) / np.max(np.abs(gc)))}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * dev_s / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": CONFIG,
                "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int((4 * N + P) * 8),
                        "d2h_bytes_per_step": int((1 + P) * 8 + 4), "ms_per_step": 1e3 * e2e_s / args.steps,
                        "api": "lfm_nlml_grad_host (C-ABI, host buffers)"},
                "gpu_launches": int(launches), "wall_s_timed_region": wall,
                "clocks": clocks_parse(clk_path, local), "roofline": roof, "cpu_baseline": cpu, "secondary": secondary}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
