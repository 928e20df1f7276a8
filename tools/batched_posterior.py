"""Batched posteriors after a 4096-restart fit (config 4): the p53 data of `JaxP53Data.synthetic()` / `dataset_3d`
(G = 5, T = 7, R = 3, N = 105), `multi_start_fit` of 4096 restarts (150 Adam steps, `trace=True, chunk=None`), then
the posteriors of every fitted LFM from `MultiStartResult.theta`, all in one process:

  - ops.batched_latent_posterior at generate_test_times(100);
  - ops.batched_gene_posterior at generate_test_times_pred(100, 5) (T* = 500), mean and variance;
  - ops.batched_gene_posterior with the full covariance, at --cov-batch LFMs;
  - ops.latent_posterior + ops.gene_posterior called once per LFM over the first --loop LFMs (per-LFM time);
  - the fit itself.

Times are CUDA-event medians of --reps calls after one warm-up (inputs already on the device, the unique-row count of X read per call as ops does; the fit as
`MultiStartResult.device_ms`, plus its wall clock).  Every batched row is checked against the single-LFM path (max
relative error per row and quantity, 1e-9 required).  Prints one JSON line with the card name and power limit read in
the same process (quoted by profiles/batched_posterior_r1.md)."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np
import torch

from dis_project_b200 import _lib, ops
from dis_project_b200.batched import make_restarts, multi_start_fit
from dis_project_b200.dataset import JaxP53Data, dataset_3d
from dis_project_b200.utils import generate_test_times, generate_test_times_pred


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def timed(fn, reps):
    """CUDA-event time of fn() (ms): one warm-up, then the median, min and max of `reps` calls."""
    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return {"median": float(np.median(ms)), "min": float(np.min(ms)), "max": float(np.max(ms))}


def rowerr(a, b):
    """max relative error of each row (normalised by the row's largest magnitude)."""
    a, b = np.asarray(a), np.asarray(b)
    a, b = a.reshape(a.shape[0], -1), b.reshape(b.shape[0], -1)
    return np.max(np.abs(a - b), axis=1) / np.maximum(np.max(np.abs(b), axis=1), 1e-300)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--restarts", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--cov-batch", type=int, default=256)
    ap.add_argument("--loop", type=int, default=64)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    _lib.require_device()
    x, y, var = dataset_3d(JaxP53Data.synthetic())
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64).reshape(-1)
    var = np.ascontiguousarray(var, dtype=np.float64).reshape(-1)
    G, B, jit = 5, args.restarts, 1e-4
    theta0 = np.concatenate([np.full(G, 0.4), np.ones(G), np.full(G, 0.05), [2.5, 1.0]])
    TH0 = make_restarts(theta0, B)
    out = {"card": card(), "N": int(x.shape[0]), "unique_rows": ops.unique_rows(x), "restarts": B, "reps": args.reps}

    # the fit that produces the parameters
    fit_dev, fit_wall = [], []
    res = multi_start_fit(x, y, TH0, jit, num_iters=150, chunk=None, trace=True)   # warm-up
    for _ in range(args.reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = multi_start_fit(x, y, TH0, jit, num_iters=150, chunk=None, trace=True)
        fit_wall.append(1e3 * (time.perf_counter() - t0))
        fit_dev.append(float(res.device_ms))
    out["fit_ms"] = {"device_median": float(np.median(fit_dev)), "wall_median": float(np.median(fit_wall)),
                     "failed_fits": int(np.count_nonzero(res.info))}

    dev = torch.device("cuda:0")
    X, Y, V = (torch.as_tensor(a, device=dev) for a in (x, y, var))
    TH = torch.as_tensor(np.ascontiguousarray(res.theta), device=dev)
    xs, xg = generate_test_times(100), generate_test_times_pred(100, G)
    XS, XG = torch.as_tensor(xs, device=dev), torch.as_tensor(xg, device=dev)
    out["Tstar_latent"], out["Tstar_gene"] = int(xs.shape[0]), int(xg.shape[0])

    lat = lambda: ops.batched_latent_posterior(X, Y, V, TH, jit, XS, G)
    gen = lambda: ops.batched_gene_posterior(X, Y, V, TH, jit, XG, G)
    nc = min(args.cov_batch, B)
    cov = lambda: ops.batched_gene_posterior(X, Y, V, TH[:nc], jit, XG, G, full_cov=True)
    nl = min(args.loop, B)

    def loop():
        for b in range(nl):
            ops.latent_posterior(X, Y, V, TH[b], jit, XS, G)
            ops.gene_posterior(X, Y, V, TH[b], jit, XG, G, full_cov=False)

    t = {"latent_batched": timed(lat, args.reps), "gene_batched": timed(gen, args.reps)}
    t["latent_plus_gene_batched_median"] = t["latent_batched"]["median"] + t["gene_batched"]["median"]
    t["gene_full_cov_batched"] = timed(cov, args.reps)
    t["gene_full_cov_batch"] = nc
    lp = timed(loop, max(1, args.reps // 2))
    t["single_loop"] = lp
    t["single_loop_lfms"] = nl
    t["single_per_lfm_ms"] = lp["median"] / nl
    t["single_loop_extrapolated_to_batch_ms"] = lp["median"] / nl * B
    t["batched_over_fit"] = t["latent_plus_gene_batched_median"] / out["fit_ms"]["device_median"]
    out["time_ms"] = t

    # every batched row against the single-LFM path
    m, v, info = (a.cpu().numpy() for a in lat())
    gm, _, gv, ginfo = gen()
    gm, gv, ginfo = gm.cpu().numpy(), gv.cpu().numpy(), ginfo.cpu().numpy()
    gcc = cov()[1].cpu().numpy()
    ok = (info == 0) & (ginfo == 0)
    err = {k: 0.0 for k in ("latent_mean", "latent_var", "gene_mean", "gene_var", "gene_cov")}
    for b in np.flatnonzero(ok):
        m1, v1, _ = (a.cpu().numpy() for a in ops.latent_posterior(X, Y, V, TH[b], jit, XS, G))
        g1, c1, w1, _ = ops.gene_posterior(X, Y, V, TH[b], jit, XG, G, full_cov=b < nc)
        g1, w1 = g1.cpu().numpy(), w1.cpu().numpy()
        err["latent_mean"] = max(err["latent_mean"], float(rowerr(m[b:b + 1], m1[None])[0]))
        err["latent_var"] = max(err["latent_var"], float(rowerr(v[b:b + 1], v1[None])[0]))
        err["gene_mean"] = max(err["gene_mean"], float(rowerr(gm[b:b + 1], g1[None])[0]))
        err["gene_var"] = max(err["gene_var"], float(rowerr(gv[b:b + 1], w1[None])[0]))
        if b < nc:
            err["gene_cov"] = max(err["gene_cov"], float(rowerr(gcc[b:b + 1], c1.cpu().numpy()[None])[0]))
    out["check"] = {"rows_compared": int(ok.sum()), "rows_failed_info": int((~ok).sum()), "max_rel_err": err,
                    "all_within_1e-9": bool(max(err.values()) < 1e-9)}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    if not out["check"]["all_within_1e-9"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
