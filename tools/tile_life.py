"""What a tile's life is made of in the rank-128 trailing update (the tile variant lfm_dgemm's heuristic picks): per-CTA debug
words of lfm_debug_syrk_stamps (SM id, clock64 at entry / first operand unit landed / last DMMA issued / stores issued,
globaltimer at entry / exit).  Prints the distribution of the phases over the CTAs of the launch and, per SM, the gaps between
one CTA leaving a slot and the next one entering."""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from dis_project_b200 import _lib
l = _lib.lib(); dev = torch.device("cuda:0"); st = torch.cuda.current_stream().cuda_stream
n, m = 4096, int(sys.argv[1]) if len(sys.argv) > 1 else 3840
K = int(sys.argv[2]) if len(sys.argv) > 2 else 128
A = torch.randn(n, n, dtype=torch.float64, device=dev)
T = (m // 64) * (m // 64 + 1) // 2   # 8 words per CTA for the smallest tiles; the rows the launch wrote are kept below
S = torch.zeros(T * 8, dtype=torch.int64, device=dev)
def run(stamps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    if stamps:
        _lib.check(l.lfm_debug_syrk_stamps(st, m, K, A.data_ptr() + 8 * (n - m) * n, n, A.data_ptr() + 8 * ((n - m) * n + K), n, S.data_ptr()), "syrk")
    else:
        _lib.check(l.lfm_debug_syrk(st, m, K, A.data_ptr() + 8 * (n - m) * n, n, A.data_ptr() + 8 * ((n - m) * n + K), n), "syrk")
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3
for _ in range(3): run(False)
plain, stamped = round(min(run(False) for _ in range(4)), 1), round(min(run(True) for _ in range(4)), 1)
s = S.cpu().numpy().reshape(T, 8)
s = s[s[:, 6] != 0]   # CTAs of the launch (exit globaltimer written)
T = len(s)
print("launch us: plain", plain, "with stamps", stamped, "tiles", T)
smid, t0, t1, t2, t3, g0, g1 = (s[:, i] for i in range(7))
q = lambda x: [int(v) for v in np.percentile(x, [5, 25, 50, 75, 95])]
print("cycles, percentiles 5/25/50/75/95 over the CTAs")
print("  entry -> address set-up done:", q(s[:, 7] - t0), " -> first unit landed:", q(t1 - s[:, 7]))
print("  entry -> first unit landed (prologue):", q(t1 - t0))
print("  first unit -> last DMMA issued (mainloop):", q(t2 - t1))
print("  last DMMA -> stores issued (epilogue):", q(t3 - t2))
print("  whole CTA:", q(t3 - t0), " ns by globaltimer:", q(g1 - g0))
span = g1.max() - g0.min()
print("launch span by globaltimer ns:", int(span))
# per SM: CTAs sorted by entry; busy time of the SM = union of CTA lifetimes; slot gaps
gaps, idle1, idle0 = [], 0.0, 0.0
tot = 0.0
for sm in np.unique(smid):
    idx = np.where(smid == sm)[0]
    ev = sorted([(g0[i], +1) for i in idx] + [(g1[i], -1) for i in idx])
    cur, last = 0, g0.min()
    occ = {0: 0, 1: 0, 2: 0}
    for t, d in ev:
        occ[min(cur, 2)] += t - last
        last = t; cur += d
    occ[0] += g1.max() - last
    tot += span; idle0 += occ[0]; idle1 += occ[1]
print("share of SM time with 0 / 1 / 2 resident CTAs: %.3f / %.3f / %.3f" % (idle0 / tot, idle1 / tot, 1 - (idle0 + idle1) / tot))
first = np.array([g0[np.where(smid == sm)[0]].min() for sm in np.unique(smid)]) - g0.min()
last = g1.max() - np.array([g1[np.where(smid == sm)[0]].max() for sm in np.unique(smid)])
print("ns from launch start to an SM's first CTA:", q(first), " from an SM's last CTA to launch end:", q(last))
print("CTAs per SM:", q(np.bincount(smid.astype(int))[np.unique(smid).astype(int)]))
