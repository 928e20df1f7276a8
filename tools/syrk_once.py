"""One rank-128 trailing update C -= P P^T (lower tiles, m = 3840, the tile variant lfm_dgemm's heuristic picks) after two
warm-ups: target for `ncu --set full` (`ncu -k regex:lfm_dgemm_kernel -s 2 -c 1 ...`)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from dis_project_b200 import _lib
l = _lib.lib(); dev = torch.device("cuda:0"); st = torch.cuda.current_stream().cuda_stream
n, m, K = 4096, 3840, int(sys.argv[1]) if len(sys.argv) > 1 else 128
A = torch.randn(n, n, dtype=torch.float64, device=dev)
for _ in range(3):
    _lib.check(l.lfm_debug_syrk(st, m, K, A.data_ptr() + 8 * (n - m) * n, n, A.data_ptr() + 8 * ((n - m) * n + K), n), "syrk")
    torch.cuda.synchronize()
print("ok")
