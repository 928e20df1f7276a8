"""Cost of the measurement variances in the batched fits (config 4): `multi_start_fit` on the p53 data of
`JaxP53Data.synthetic()` / `dataset_3d`, 150 Adam steps, `trace=True, chunk=None`, with and without `variances=` (the
third output of `dataset_3d`), alternating in one process: one warm-up of each, then `--reps` pairs; median wall clock
(host clock around the call, which ends in a device synchronise) and median device time (`MultiStartResult.device_ms`).
Two loads: 4096 restarts on one GPU, and the 512-restart shard that one rank of eight fits.  Prints one JSON line with
the card name and power limit read in the same process (quoted by profiles/batched_het_r3.md)."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np
import torch

from dis_project_b200 import _lib
from dis_project_b200.batched import make_restarts, multi_start_fit
from dis_project_b200.dataset import JaxP53Data, dataset_3d


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    _lib.require_device()
    x, y, var = dataset_3d(JaxP53Data.synthetic())
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64).reshape(-1)
    var = np.ascontiguousarray(var, dtype=np.float64).reshape(-1)
    G = 5
    theta0 = np.concatenate([np.full(G, 0.4), np.ones(G), np.full(G, 0.05), [2.5, 1.0]])
    TH_all = make_restarts(theta0, 4096)
    out = {"card": card(), "N": int(x.shape[0]), "unique_rows": int(_lib.lib().lfm_count_unique_rows(x.shape[0], x.ctypes.data)),
           "steps": 150, "reps": args.reps, "loads": {}}
    for B in (4096, 512):
        TH = np.ascontiguousarray(TH_all[:B])
        team = int(_lib.lib().lfm_batched_team_size(B, x.shape[0], G, out["unique_rows"], 7))
        runs = {"plain": dict(variances=None), "het": dict(variances=var)}
        res = {k: {"wall_ms": [], "device_ms": []} for k in runs}
        best = {}
        for k, kw in runs.items():   # warm-up: module load, plan construction, occupancy queries
            r = multi_start_fit(x, y, TH, 1e-4, num_iters=150, chunk=None, trace=True, **kw)
            best[k] = (float(r.best_loss), int(r.best_id), int(np.count_nonzero(r.info)))
        for _ in range(args.reps):
            for k, kw in runs.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                r = multi_start_fit(x, y, TH, 1e-4, num_iters=150, chunk=None, trace=True, **kw)
                res[k]["wall_ms"].append(1e3 * (time.perf_counter() - t0))
                res[k]["device_ms"].append(float(r.device_ms))
        load = {"restarts": B, "warps_per_lfm_plain": team, "best": best}
        for k in runs:
            load[k] = {m: {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v))}
                       for m, v in res[k].items()}
        load["het_over_plain_wall"] = load["het"]["wall_ms"]["median"] / load["plain"]["wall_ms"]["median"]
        load["het_over_plain_device"] = load["het"]["device_ms"]["median"] / load["plain"]["device_ms"]["median"]
        out["loads"][str(B)] = load
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
