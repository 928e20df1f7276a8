"""Rate of the trailing update C -= P P^T (lower tiles) for the shapes of the blocked Cholesky."""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from dis_project_b200 import _lib
l = _lib.lib(); dev = torch.device("cuda:0"); st = torch.cuda.current_stream().cuda_stream
n = 4096
A = torch.randn(n, n, dtype=torch.float64, device=dev)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
def t(m, K, cold):
    ts = []
    for it in range(6):
        if cold: flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.check(l.lfm_debug_syrk(st, m, K, A.data_ptr() + 8 * (n - m) * n, n, A.data_ptr() + 8 * ((n - m) * n + K), n), "syrk")
        e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts[2:]))
for K in (128, 256, 512):
    for m in (512, 1024, 2048, 3072, 3840):
        if m + K > n: continue
        for cold in (0, 1):
            ms = t(m, K, cold)
            fl = (m / 128) * (m / 128 + 1) / 2 * 128 * 128 * K * 2
            print(json.dumps({"K": K, "m": m, "cold": cold, "us": ms * 1e3, "tflops": fl / ms / 1e9}), flush=True)
