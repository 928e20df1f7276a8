"""Kernel time of a 150-step p53 fit of B LFMs on one GPU: separate launches of 10 steps (static one-CTA-per-LFM
assignment) against ONE launch with persistent workers + task queue (lfm_batched_fit_het with queue_ws), team of four warps per LFM."""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from dis_project_b200 import ops
from dis_project_b200.batched import make_restarts
from dis_project_b200.dataset import JaxP53Data, dataset_3d
x, y, _ = dataset_3d(JaxP53Data.synthetic()); y = y.reshape(-1)
TH = make_restarts(np.concatenate([np.full(5, 0.4), np.ones(5), np.full(5, 0.05), [2.5, 1.0]]), 4096)
X = torch.as_tensor(x).cuda(); Y = torch.as_tensor(y).cuda()
os.environ["LFM_BATCHED_TEAM"] = sys.argv[1] if len(sys.argv) > 1 else "4"

def fit(B, queue_chunk, chunk=10):
    st = ops.BatchedFitState(TH[:B], 5, 150)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    if queue_chunk:
        ops.batched_fit_steps(st, X, Y, 1e-4, 150, queue_chunk=queue_chunk)
    else:
        for c in range(0, 150, chunk):
            ops.batched_fit_steps(st, X, Y, 1e-4, chunk)
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1), st

for B in (148, 296, 333, 444, 512, 550, 592, 1024):
    row = {"B": B}
    _, ref = fit(B, 0)
    row["static_chunk10_ms"] = round(min(fit(B, 0)[0] for _ in range(3)), 3)
    for q in (0, 1):
        os.environ["LFM_BATCHED_QUEUE"] = str(q)   # 0: the workspace is ignored (one plain launch of 150 steps); 1: forced
        for qc in ((10,) if q == 0 else (5, 10, 15, 30)):
            t, st = fit(B, qc)
            t = min(t, *(fit(B, qc)[0] for _ in range(2)))
            row[("queue" if q else "plain150") + f"_chunk{qc}_ms"] = round(t, 3)
            if q and qc == 10:
                row["queue_equals_static"] = bool(torch.equal(st.hist, ref.hist))
    os.environ.pop("LFM_BATCHED_QUEUE")
    row["auto_ms"] = round(min(fit(B, 10)[0] for _ in range(3)), 3)
    print(json.dumps(row), flush=True)
