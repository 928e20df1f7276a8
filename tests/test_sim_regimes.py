"""The SIM covariance beyond the p53 regime, against a high-precision reference.

The other parity tests draw their parameters from D in [0.2, 1], l in [0.8, 3.2] and times in [0, 12], and most of them
compare the CUDA path with the oracle, which evaluates the same formulas: a defect the two share is invisible there.
The multi-start fits go further (l is bounded to (0.5, 3.5) by the sigmoid, D is not), and so do real data sets
(absolute timestamps, irregular and per-gene time grids).  This file

  * writes h, k_xx, k_xf, k_ff and the partials of h literally from src/model.py:197-369 in mpmath, at a working
    precision chosen per point and checked by a second evaluation with 30 more digits (erf(-9.28) + erf(9.86) loses
    every digit at 40 digits: a fixed precision is not a reference),
  * checks the oracle against it in a set of named regimes (CPU), entry by entry on the scale sqrt(Sigma_ii Sigma_jj),
    never on the largest entry, and the gradient component by component,
  * checks every CUDA path against the oracle in the same regimes (GPU): the covariance entry points, the dense and
    time-grid NLML + gradient, the evaluation plan, the batched kernels (one warp, teams of four and eight warps, one
    CTA per LFM) and their dispatch edges, and the four posteriors.

The gamma regimes (gamma = D l / 2 >= 4.4) fail with the literal second erf sum of h, erf(t/l - gamma) + erf(gamma),
which cancels for t/l < gamma and is then multiplied by exp(gamma^2)."""
import math
import zlib
from dataclasses import dataclass
from typing import Tuple

import mpmath as mp
import numpy as np
import pytest

from oracle import lfm_oracle as o

JITTER = 1e-4
SIGMA = 1.0
ENTRY_TOL = 1e-13        # |K_hat_ij - K_ij| <= ENTRY_TOL sqrt(Sigma_ii Sigma_jj)
SELF_CHECK = 1e-22       # the reference at its precision and at 30 more digits agree to this (relative to the scale)


# ---- regimes ---------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Regime:
    name: str
    d: Tuple[float, ...]
    l: float
    times: Tuple[Tuple[float, ...], ...]     # one time set per gene (equal sizes: the mean is positional, model.py:145)
    s: Tuple[float, ...] = (0.7, 1.3, 1.0)
    b: Tuple[float, ...] = (0.05, 0.08, 0.03)

    @property
    def G(self):
        return len(self.d)

    def params(self):
        return o.Params(d=np.array(self.d), s=np.array(self.s[:self.G]), b=np.array(self.b[:self.G]), l=self.l,
                        sigma=SIGMA, jitter=JITTER)

    def x(self):
        rows = [(t, g, 1.0) for g, ts in enumerate(self.times) for t in ts]
        return np.array(rows, dtype=np.float64)

    def latent(self):
        """Latent test rows inside and outside the data's time range (at most 3 beyond it, so that D |t - t'| stays
        below the 709 where exp overflows in every regime)."""
        ts = np.concatenate(self.times)
        lo, hi = float(ts.min()), float(ts.max())
        out = min(0.2 * (hi - lo), 3.0)
        t = np.array([lo - out, lo, lo + 0.37 * (hi - lo), lo + 0.81 * (hi - lo), hi, hi + out])
        return np.stack([t, -np.ones_like(t), np.zeros_like(t)], axis=1)


def _shared(ts, G=3):
    return tuple(tuple(float(t) for t in ts) for _ in range(G))


P53_T = _shared(np.linspace(0.0, 12.0, 7))
REGIMES = [Regime("p53", (0.25, 0.55, 0.95), 2.5, P53_T)]
for _gam in (3.5, 4.4, 5.25, 7.0, 8.75):
    for _l in (3.499, 2.5):
        _dm = 2 * _gam / _l
        REGIMES.append(Regime(f"gamma{_gam}_l{_l}", (0.3, _dm / 2, _dm), _l, P53_T))
REGIMES += [
    Regime("l_low", (0.2, 2.0, 6.0), 0.501, P53_T),
    Regime("tiny_d", (0.01, 0.4, 3.0), 3.0, P53_T),
    # absolute timestamps: max D t = 748 > 600 selects the batched kernels' direct evaluation ("slow"), and beyond 745
    # exp(-D t) underflows, so that the factored exp(-D t_b) / exp(-D t_a) would be 0 * inf; the control stays at 590
    Regime("offset", (0.3, 0.6, 1.05), 2.5, _shared(np.linspace(700.0, 712.0, 7))),
    Regime("offset_control", (0.3, 0.6, 590.0 / 712.0), 2.5, _shared(np.linspace(700.0, 712.0, 7))),
    Regime("long", (0.05, 0.5, 1.0), 3.0, _shared(np.linspace(0.0, 650.0, 8))),
    Regime("negative", (0.2, 0.6, 1.2), 2.0, _shared(np.linspace(-6.0, 6.0, 7))),
    Regime("logspaced", (0.1, 1.0, 3.0), 1.2, _shared([0, 0.25, 0.5, 1, 2, 4, 8, 12])),
    Regime("disjoint", (0.4, 1.5, 3.0), 2.8, ((0.0, 2.4, 4.8, 7.2, 9.6, 12.0), (0.5, 1.7, 3.1, 5.9, 8.3, 11.6),
                                               (0.2, 2.2, 4.4, 6.6, 9.9, 12.5))),
]
BY_NAME = {r.name: r for r in REGIMES}
NAMES = [r.name for r in REGIMES]


def problem(r: Regime, seed=0):
    """(p, x, y, variances): y drawn from the model's prior at the regime's own parameters."""
    p = r.params()
    x = r.x()
    rng = np.random.default_rng(seed)
    S = o.sigma_matrix(p, x)
    y = o.mean_function(p, x) + np.linalg.cholesky(S) @ rng.standard_normal(x.shape[0])
    var = rng.uniform(0.01, 0.1, x.shape[0])
    return p, x, y, var


def sigma_scale(p, rows):
    """sqrt(Sigma_ii Sigma_jj) per entry: Sigma_ii = K_ii + sigma^2 on gene rows, k_ff(t, t) + jitter on latent rows."""
    kd = np.array([o.cross_covariance(p, rows[i:i + 1], rows[i:i + 1])[0, 0] for i in range(rows.shape[0])])
    sd = np.where(rows[:, 2] == 1, kd + p.sigma ** 2, 1.0 + p.jitter)
    return np.sqrt(np.outer(sd, sd))


# ---- high-precision reference (src/model.py:197-369, literally) -------------------------------------------------------
def _digits(*log_mult):
    """Working precision for a point: 30 digits beyond the largest factor, exp(max(log_mult)), that multiplies an erf sum.
    An erf sum that cancels down to erfc(x) ~ exp(-x^2) is computed to an absolute 10^-dps like any other, and what
    reaches the entry is that error times its factor (exp(gamma^2) exp(-D dt) or exp(gamma^2) exp(-(D_b v + D_a u))).
    The entries are compared on a scale >= sigma^2 = 1, so 30 digits beyond the factor are ample; _checked verifies it."""
    return 30 + int(math.ceil(max(0.0, *log_mult) / math.log(10)))


def _checked(f, dps, scale):
    """f() at dps and at dps + 30 digits; the two agree to SELF_CHECK * scale or the reference is not one."""
    with mp.workdps(dps):
        a = f()
    with mp.workdps(dps + 30):
        b = f()
    assert abs(a - b) <= SELF_CHECK * scale, f"reference lost its precision at {dps} digits"
    return b


def mp_h(da, db, l, u, v):
    """model.py:315-365: h(j, k, t1=u, t2=v) with D_j = da, D_k = db, gamma = D_k l / 2."""
    da, db, l, u, v = (mp.mpf(float(z)) if not isinstance(z, mp.mpf) else z for z in (da, db, l, u, v))
    g = db * l / 2
    td = v - u
    first = mp.exp(-db * td) * (mp.erf(td / l - g) + mp.erf(u / l + g))
    second = mp.exp(-(db * v + da * u)) * (mp.erf(v / l - g) + mp.erf(g))
    return mp.exp(g ** 2) / (da + db) * (first - second)


def _h_digits(da, db, l, u, v):
    g = db * l / 2
    return _digits(g * g - db * (v - u), g * g - (db * v + da * u))


def mp_kxx(p, t, j, tp, k):
    mult = lambda: mp.mpf(float(p.s[j])) * mp.mpf(float(p.s[k])) * mp.mpf(float(p.l)) * mp.sqrt(mp.pi) / 2
    return lambda: mult() * (mp_h(p.d[k], p.d[j], p.l, tp, t) + mp_h(p.d[j], p.d[k], p.l, t, tp))


def mp_kxf(p, tg, j, tl):
    def f():
        d, l, s = (mp.mpf(float(z)) for z in (p.d[j], p.l, p.s[j]))
        tgm, tlm = mp.mpf(float(tg)), mp.mpf(float(tl))
        td = tgm - tlm
        g = d * l / 2
        return l * mp.sqrt(mp.pi) / 2 * s * mp.exp(g ** 2) * mp.exp(-d * td) * (mp.erf(td / l - g) + mp.erf(tlm / l + g))
    return f


def mp_cross(p, xa, xb, scale):
    """The reference's covariance between two row sets (model.py:152-195), every entry self-checked."""
    out = np.empty((xa.shape[0], xb.shape[0]))
    for i, (t, j, f1) in enumerate(xa):
        for c, (tp, k, f2) in enumerate(xb):
            j_, k_ = int(j), int(k)
            if f1 and f2:
                dps = max(_h_digits(p.d[k_], p.d[j_], p.l, tp, t), _h_digits(p.d[j_], p.d[k_], p.l, t, tp))
                fn = mp_kxx(p, t, j_, tp, k_)
            elif f1 or f2:
                tg, g, tl = (t, j_, tp) if f1 else (tp, k_, t)
                gm = p.d[g] * p.l / 2
                dps = _digits(gm * gm - p.d[g] * (tg - tl))
                fn = mp_kxf(p, tg, g, tl)
            else:
                dps = 30
                fn = lambda t=t, tp=tp: mp.exp(-(mp.mpf(float(t)) - mp.mpf(float(tp))) ** 2 / (2 * mp.mpf(float(p.l))))
            out[i, c] = float(_checked(fn, dps, scale[i, c]))
    return out


def mp_h_partials(p, a, b, u, v):
    """(H, dH/dD_a, dH/dD_b, dH/dl) of h(j=a, k=b, t1=u, t2=v) by mp.diff of the literal formula."""
    dps = _h_digits(p.d[a], p.d[b], p.l, u, v) + 10
    da, db, l = float(p.d[a]), float(p.d[b]), float(p.l)
    fns = (lambda: mp_h(da, db, l, u, v),
           lambda: mp.diff(lambda z: mp_h(z, mp.mpf(db), mp.mpf(l), mp.mpf(u), mp.mpf(v)), mp.mpf(da)),
           lambda: mp.diff(lambda z: mp_h(mp.mpf(da), z, mp.mpf(l), mp.mpf(u), mp.mpf(v)), mp.mpf(db)),
           lambda: mp.diff(lambda z: mp_h(mp.mpf(da), mp.mpf(db), z, mp.mpf(u), mp.mpf(v)), mp.mpf(l)))
    vals = []
    for f in fns:
        with mp.workdps(dps):
            x0 = f()
        with mp.workdps(dps + 30):
            x1 = f()
        assert abs(x0 - x1) <= SELF_CHECK * max(1.0, abs(x1)), f"reference lost its precision at {dps} digits"
        vals.append(x1)
    return vals


# ---- CPU: the oracle against the reference ---------------------------------------------------------------------------
@pytest.mark.parametrize("name", NAMES)
def test_oracle_covariance_entries_against_mpmath(name):
    """Every entry of the covariance of gene rows and latent rows (inside and outside the data's time range):
    k_xx, k_xf both ways round and k_ff, on the scale sqrt(Sigma_ii Sigma_jj)."""
    r = BY_NAME[name]
    p = r.params()
    rows = np.concatenate([r.x(), r.latent()])
    sc = sigma_scale(p, rows)
    K = o.cross_covariance(p, rows, rows)
    ref = mp_cross(p, rows, rows, sc)
    err = np.abs(K - ref) / sc
    assert np.all(np.isfinite(K)) and err.max() <= ENTRY_TOL, (name, float(err.max()))


# h-term partials of the oracle against mp.diff, on the covariance scale: S_a S_b (l sqrt(pi) / 2) |err| <=
# PARTIAL_TOL sqrt(Sigma(u, a) Sigma(v, b)) (1 + |u| + |v|) -- a partial of k_xx with respect to D carries a factor of the
# time.  Measured: <= 5e-15 in every regime (tiny_d), 3e-4 .. 0.15 with the literal sums at gamma >= 4.4.
PARTIAL_TOL = 1e-13


@pytest.mark.parametrize("name", NAMES)
def test_oracle_h_partials_against_mpmath(name):
    r = BY_NAME[name]
    p = r.params()
    ts = np.unique(np.concatenate(r.times))
    pick = ts[np.unique(np.linspace(0, ts.size - 1, 4).round().astype(int))]
    sd = {(a, u): o.cross_covariance(p, np.array([[u, a, 1.0]]), np.array([[u, a, 1.0]]))[0, 0] + p.sigma ** 2
          for a in range(r.G) for u in pick}
    worst = 0.0
    for a in range(r.G):
        for b in range(r.G):
            mult = p.s[a] * p.s[b] * p.l * math.sqrt(math.pi) / 2
            for u in pick:
                for v in pick:
                    got = o._h_partials(p, np.array(a), np.array(b), np.array(u), np.array(v))
                    ref = mp_h_partials(p, a, b, u, v)
                    sc = math.sqrt(sd[(a, u)] * sd[(b, v)]) * (1 + abs(u) + abs(v))
                    for gv, rv in zip(got, ref):
                        worst = max(worst, mult * abs(float(gv) - float(rv)) / sc)
    assert worst <= PARTIAL_TOL, (name, worst)


def _mp_nlml(theta, x, y, jitter, G):
    """objectives.py:64-78 over model.py:124-149,197-235 literally, at the current precision."""
    th = [mp.mpf(v) for v in theta]
    d, s, b, l, sigma = th[:G], th[G:2 * G], th[2 * G:3 * G], th[3 * G], th[3 * G + 1]
    N = x.shape[0]
    block = N // G
    K = mp.matrix(N, N)
    for i in range(N):
        for j in range(i + 1):
            t, tp = mp.mpf(float(x[i, 0])), mp.mpf(float(x[j, 0]))
            gi, gj = int(x[i, 1]), int(x[j, 1])
            v = s[gi] * s[gj] * l * mp.sqrt(mp.pi) / 2 * (mp_h(d[gj], d[gi], l, tp, t) + mp_h(d[gi], d[gj], l, t, tp))
            K[i, j] = K[j, i] = v
        K[i, i] += mp.mpf(jitter) + sigma ** 2
    L = mp.cholesky(K)
    z = mp.matrix([mp.mpf(float(y[i])) - b[i // block] / d[i // block] for i in range(N)])
    w = mp.lu_solve(L, z)
    return (N * mp.log(2 * mp.pi) + 2 * sum(mp.log(L[i, i]) for i in range(N)) + sum(w[i] ** 2 for i in range(N))) / 2


# The oracle's gradient against central differences of the mp NLML agrees to <= 1.5e-15 of the largest component in
# these regimes (measured); GRAD_FLOOR leaves a factor ~30 above that and stays far below the 1e-9 of the largest
# component that max-normalised comparisons allow on every component.
GRAD_RTOL = 1e-9
GRAD_FLOOR = 1e-13
# NLML values: the negative-time regime's Sigma has eigenvalues from 1 to 1e6, and the kernels' value differs from the
# oracle's by up to 1.4e-12 relative there (3e-15 elsewhere)
VAL_RTOL = 1e-11


def grad_close(got, ref, rtol=GRAD_RTOL, floor=GRAD_FLOOR):
    """Component by component: |got_i - ref_i| <= rtol |ref_i| + floor max|ref|.  Returns the worst ratio err / bound."""
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    bound = rtol * np.abs(ref) + floor * np.max(np.abs(ref))
    return float(np.max(np.abs(got - ref) / bound))


@pytest.mark.parametrize("name", ["gamma7.0_l2.5", "offset"])
def test_nlml_and_gradient_against_mpmath_end_to_end(name):
    """NLML and its gradient (central differences, h = 1e-30) for 3 genes x 4 times in mp at 120 digits."""
    r = BY_NAME[name]
    sub = Regime(r.name, r.d, r.l, tuple(ts[::2] for ts in r.times), r.s, r.b)
    p, x, y, _ = problem(sub, seed=5)
    theta = p.pack()
    v, g = o.nlml_and_grad(p, x, y)
    with mp.workdps(120):
        ref = _mp_nlml([float(t) for t in theta], x, y, p.jitter, sub.G)
        assert abs(float(mp.mpf(float(v)) - ref)) <= 1e-13 * abs(float(ref))
        h = mp.mpf(10) ** -30
        gref = np.empty(theta.shape[0])
        for idx in range(theta.shape[0]):
            tp = [mp.mpf(float(t)) for t in theta]
            tm = list(tp)
            tp[idx] += h
            tm[idx] -= h
            gref[idx] = float((_mp_nlml(tp, x, y, p.jitter, sub.G) - _mp_nlml(tm, x, y, p.jitter, sub.G)) / (2 * h))
    assert grad_close(g, gref) <= 1.0, (name, g, gref)


def test_literal_second_sum_is_what_the_gamma_regimes_catch():
    """LITERAL_ERF_SUMS restores the reference's literal arithmetic for both sums; at gamma = 7 that form is off by far
    more than the entry tolerance (which is why the oracle does not use it), in the p53 regime it is not."""
    for name, bad in (("gamma7.0_l2.5", True), ("p53", False)):
        r = BY_NAME[name]
        p = r.params()
        x = r.x()
        sc = sigma_scale(p, x)
        acc = o.gram(p, x)
        try:
            o.LITERAL_ERF_SUMS = True
            lit = o.gram(p, x)
        finally:
            o.LITERAL_ERF_SUMS = False
        assert (np.max(np.abs(acc - lit) / sc) > 1e3 * ENTRY_TOL) == bad, name


# ---- GPU: every CUDA path against the oracle -------------------------------------------------------------------------
def _report(name, path, err):
    print(f"REGIME {name:18s} {path:34s} {err:.2e}")


SIZES = [1, 31, 32, 33, 63, 64, 65, 127, 128, 129, 257]


def _rows(r: Regime, n, rng, flags="mixed"):
    """n rows of the regime's kind: times drawn from the regime's range (and its latent test times), genes cycled."""
    x, lat = r.x(), r.latent()
    pool = np.concatenate([x[:, 0], lat[:, 0]])
    t = rng.choice(pool, n)
    t = np.where(rng.random(n) < 0.3, rng.uniform(pool.min(), pool.max(), n), t)
    g = np.arange(n) % r.G
    if flags == "gene":
        f = np.ones(n)
    elif flags == "latent":
        f = np.zeros(n)
    else:
        f = (rng.random(n) < 0.7).astype(np.float64)
    g = np.where(f == 1, g, -1)
    return np.stack([t, g.astype(np.float64), f], axis=1)


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_covariance_entry_points_match_oracle(cuda, name):
    """ops.cross_covariance (square, rectangular, mixed flags), ops.gram and ops.h_terms, entry by entry."""
    from dis_project_b200 import ops
    r = BY_NAME[name]
    p = r.params()
    th = p.pack()
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    worst = 0.0
    shapes = [(m, m) for m in SIZES] + [(1, 257), (257, 1), (31, 129), (65, 33), (128, 63)]
    for m, n in shapes:
        a = _rows(r, m, rng, "gene" if m == 1 else "mixed")
        b = _rows(r, n, rng, "latent" if n == 1 else "mixed")
        ref = o.cross_covariance(p, a, b)
        got = ops.cross_covariance(a, b, th, r.G).cpu().numpy()
        sa = np.sqrt(np.diag(sigma_scale(p, a)))
        sb = np.sqrt(np.diag(sigma_scale(p, b)))
        err = np.max(np.abs(got - ref) / np.outer(sa, sb))
        worst = max(worst, err)
        assert err <= ENTRY_TOL, (name, m, n, err)
    x = r.x()
    sc = sigma_scale(p, x)
    err = np.max(np.abs(ops.gram(x, th, r.G).cpu().numpy() - o.gram(p, x)) / sc)
    assert err <= ENTRY_TOL, (name, err)
    _report(name, "cross_covariance / gram", max(worst, err))
    # h itself: every (j, k, t1, t2) of the design, on the scale E0 (A1 + A2) of its two terms (|R1|, |R2| <= 2)
    n = x.shape[0]
    J, K = np.meshgrid(x[:, 1], x[:, 1], indexing="ij")
    T1, T2 = np.meshgrid(x[:, 0], x[:, 0], indexing="ij")
    J, K, T1, T2 = (a.reshape(-1) for a in (J, K, T1, T2))
    got = ops.h_terms(J, K, T1, T2, th, r.G).cpu().numpy()
    ji, ki = J.astype(int), K.astype(int)
    ref = o.h(p, ji, ki, T1, T2)
    gk = p.d[ki] * p.l / 2
    hs = np.exp(gk * gk) / (p.d[ji] + p.d[ki]) * (np.exp(-p.d[ki] * (T2 - T1)) + np.exp(-(p.d[ki] * T2 + p.d[ji] * T1)))
    err = np.max(np.abs(got - ref) / hs)
    _report(name, "h_terms", err)
    assert got.shape == (n * n,) and err <= ENTRY_TOL, (name, err)


def _unc(p):
    return o.unconstrain(p.pack())


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_nlml_and_gradients_match_oracle(cuda, name):
    """ops.nlml / nlml_grad / nlml_grad_unc on the direct path (time_grid = 0) and on the time-grid tables, and
    NlmlGradPlan (constrained and unconstrained): the value to 1e-12, the gradient component by component."""
    from dis_project_b200 import ops
    r = BY_NAME[name]
    p, x, y, _ = problem(r, seed=11)
    th, u = p.pack(), _unc(p)
    v_ref, g_ref = o.nlml_and_grad(p, x, y)
    vu_ref, gu_ref = o.nlml_and_grad_unc(u, x, y, JITTER)
    worst = 0.0
    for tg in (0, None):
        out, info = ops.nlml(x, y, th, JITTER, r.G, time_grid=tg)
        assert int(info.item()) == 0 and abs(out.item() - v_ref) <= VAL_RTOL * abs(v_ref), (name, tg)
        out, info = ops.nlml_grad(x, y, th, JITTER, r.G, time_grid=tg)
        out = out.cpu().numpy()
        assert int(info.item()) == 0 and abs(out[0] - v_ref) <= VAL_RTOL * abs(v_ref), (name, tg)
        worst = max(worst, grad_close(out[1:], g_ref))
        out, info = ops.nlml_grad_unc(x, y, u, JITTER, r.G, time_grid=tg)
        out = out.cpu().numpy()
        assert int(info.item()) == 0 and abs(out[0] - vu_ref) <= VAL_RTOL * abs(vu_ref), (name, tg)
        worst = max(worst, grad_close(out[1:], gu_ref))
        for unc, arg, gr in ((False, th, g_ref), (True, u, gu_ref)):
            plan = ops.NlmlGradPlan(x, y, r.G, JITTER, unconstrained=unc, time_grid=tg)
            out, info = plan(arg)
            out = out.cpu().numpy().copy()
            plan.close()
            assert int(info.item()) == 0 and abs(out[0] - v_ref) <= VAL_RTOL * abs(v_ref), (name, tg, unc)
            worst = max(worst, grad_close(out[1:], gr))
    _report(name, "nlml_grad (direct, grid, plan)", worst)
    assert worst <= 1.0, (name, worst)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["gamma7.0_l3.499", "offset"])
def test_heteroscedastic_nlml_gradients_match_oracle(cuda, name):
    from dis_project_b200 import ops
    r = BY_NAME[name]
    p, x, y, var = problem(r, seed=12)
    var = var * 20
    u = _unc(p)
    vu_ref, gu_ref = o.nlml_and_grad_unc(u, x, y, JITTER, variances=var)
    worst = 0.0
    for tg in (0, None):
        out, info = ops.nlml_grad_unc(x, y, u, JITTER, r.G, time_grid=tg, variances=var)
        out = out.cpu().numpy()
        assert int(info.item()) == 0 and abs(out[0] - vu_ref) <= VAL_RTOL * abs(vu_ref)
        worst = max(worst, grad_close(out[1:], gu_ref))
        plan = ops.NlmlGradPlan(x, y, r.G, JITTER, unconstrained=True, time_grid=tg, variances=var)
        out, info = plan(u)
        out = out.cpu().numpy().copy()
        plan.close()
        assert int(info.item()) == 0 and abs(out[0] - vu_ref) <= VAL_RTOL * abs(vu_ref)
        worst = max(worst, grad_close(out[1:], gu_ref))
    U = u[None, :].repeat(2, 0)
    val, grad, info = ops.batched_nlml_grad_unc(x, y, U, JITTER, r.G, variances=var)
    assert not info.cpu().numpy().any() and abs(val[0].item() - vu_ref) <= VAL_RTOL * abs(vu_ref)
    worst = max(worst, grad_close(grad[1].cpu().numpy(), gu_ref))
    _report(name, "nlml_grad heteroscedastic", worst)
    assert worst <= 1.0, (name, worst)


# batched kernels: one warp (1), teams of four and eight warps, one CTA per LFM (0)
TEAMS = [1, 4, 8, 0]
# regimes that share the time axis [0, 12]: one batch, every LFM in a different regime
SHARED_AXIS = [n for n in NAMES if BY_NAME[n].times == P53_T]


def _use_team(monkeypatch, team):
    if team:
        monkeypatch.setenv("LFM_BATCHED_TEAM", str(team))
    else:
        monkeypatch.delenv("LFM_BATCHED_TEAM", raising=False)
    return 0 if team == 0 else None


def _batch_cases():
    """(X, y, [(label, constrained theta)]) per time axis: the [0, 12] regimes in one batch; the offset axis with the
    slow-path LFM between two that stay below the threshold; and one batch per remaining axis."""
    cases = []
    x = BY_NAME["p53"].x()
    y = problem(BY_NAME["p53"], seed=21)[2]
    cases.append((x, y, [(n, BY_NAME[n].params().pack()) for n in SHARED_AXIS]))
    off, ctl = BY_NAME["offset"], BY_NAME["offset_control"]
    cases.append((off.x(), problem(off, seed=22)[2],
                  [("offset_control", ctl.params().pack()), ("offset", off.params().pack()),
                   ("offset_control", ctl.params().pack())]))
    for n in ("long", "negative", "logspaced", "disjoint"):
        r = BY_NAME[n]
        cases.append((r.x(), problem(r, seed=23)[2], [(n, r.params().pack())]))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("team", TEAMS)
def test_batched_regimes_match_oracle_and_run_alone(cuda, team, monkeypatch):
    """ops.batched_nlml_grad_unc against the oracle per LFM, and every LFM's outputs equal, bit for bit, the same LFM
    run alone: the slow path and the erf / erfc choices are per LFM and must not leak to the neighbours."""
    from dis_project_b200 import ops
    tg = _use_team(monkeypatch, team)
    for x, y, lfms in _batch_cases():
        U = np.stack([o.unconstrain(th) for _, th in lfms])
        val, grad, info = ops.batched_nlml_grad_unc(x, y, U, JITTER, 3, time_grid=tg)
        assert not info.cpu().numpy().any()
        val, grad = val.cpu().numpy(), grad.cpu().numpy()
        for b, (label, _) in enumerate(lfms):
            v, g = o.nlml_and_grad_unc(U[b], x, y, JITTER)
            w = grad_close(grad[b], g)
            _report(label, f"batched_nlml_grad_unc team={team}", max(w * GRAD_FLOOR, abs(val[b] - v) / abs(v)))
            assert abs(val[b] - v) <= VAL_RTOL * abs(v) and w <= 1.0, (label, team, w)
            v1, g1, i1 = ops.batched_nlml_grad_unc(x, y, U[b:b + 1], JITTER, 3, time_grid=tg)
            assert not i1.cpu().numpy().any()
            assert v1.cpu().numpy()[0] == val[b] and np.array_equal(g1.cpu().numpy()[0], grad[b]), (label, team)


@pytest.mark.gpu
@pytest.mark.parametrize("team", TEAMS)
def test_batched_fit_regimes_match_oracle_fit(cuda, team, monkeypatch):
    """30 Adam steps of batched_fit_steps per regime against o.fit (loss history and final theta)."""
    from dis_project_b200 import ops
    tg = _use_team(monkeypatch, team)
    for x, y, lfms in _batch_cases():
        if lfms[0][0] == "long":
            continue   # Adam moves D past 709 / 650, where the formula itself overflows (the reference returns NaN too)
        TH = np.stack([th for _, th in lfms])
        st = ops.BatchedFitState(TH, 3, 30)
        if tg is not None:
            st.time_grid = tg
        ops.batched_fit_steps(st, x, y, JITTER, 30)
        theta, hist, info = st.theta.cpu().numpy(), st.hist.cpu().numpy(), st.info.cpu().numpy()
        assert not info.any()
        for b, (label, _) in enumerate(lfms):
            th_ref, h_ref = o.fit(TH[b], x, y, JITTER, num_iters=30)
            eh = np.max(np.abs(hist[b] - h_ref) / np.abs(h_ref))
            et = np.max(np.abs(theta[b] - th_ref) / np.abs(th_ref))
            _report(label, f"batched_fit_steps team={team}", max(eh, et))
            assert eh <= 1e-10 and et <= 1e-9, (label, team, eh, et)


def _edge_case(kind, big):
    """(X, y, G, regime label) on either side of a dispatch limit of the warp / team kernels (batched_warp.cu)."""
    rng = np.random.default_rng(31 + big)
    if kind == "U":          # unique rows: 36 / 37 (one gene, 36 / 37 times)
        T = 37 if big else 36
        r = Regime("gamma7.0_l2.5/U", (2 * 7.0 / 2.5,), 2.5, (tuple(np.linspace(0.0, 12.0, T)),), (1.0,), (0.05,))
    elif kind == "GT2":      # G Tu^2: 2048 (2 x 32^2) / 2178 (2 x 33^2), two genes on disjoint time sets
        t0 = tuple(np.linspace(0.0, 12.0, 16 + big))
        t1 = tuple(np.linspace(0.37, 11.63, 16 + big))
        if big:
            t1 = t1[:-1] + (t0[5],)        # one shared time: 17 + 17 rows over 33 distinct times
        r = Regime("disjoint/GT2", (0.4, 3.0), 2.8, (t0, t1), (0.7, 1.3), (0.05, 0.08))
    else:                    # parameters: P = 62 (G = 20) / 65 (G = 21), two replicates of one time per gene
        G = 21 if big else 20
        ts = np.linspace(0.0, 12.0, 9)
        d = tuple(np.linspace(0.2, 4.0, G))
        r = Regime("gamma5.6/P", d, 2.8, tuple((float(ts[g % 9]),) for g in range(G)), tuple(np.linspace(0.5, 1.5, G)),
                   tuple(np.linspace(0.01, 0.1, G)))
    p = r.params()
    x = r.x()
    if kind == "P":
        x = np.concatenate([x, x])
    S = o.sigma_matrix(p, x)
    y = o.mean_function(p, x) + np.linalg.cholesky(S) @ rng.standard_normal(x.shape[0])
    return x, y, r.G, r.name, p


@pytest.mark.gpu
@pytest.mark.parametrize("kind,expect", [("U", (1, 0)), ("GT2", (1, 0)), ("P", (1, 0))])
def test_batched_dispatch_edges_match_oracle(cuda, kind, expect, monkeypatch):
    """Either side of each limit of the warp / team kernels (U <= 36, G Tu^2 <= 2048, P <= 64): lfm_batched_team_size
    says which kernel runs, and each result is compared with the oracle."""
    from dis_project_b200 import _lib, ops
    monkeypatch.setenv("LFM_BATCHED_TEAM", "1")
    lib = _lib.lib()
    for big, team in zip((0, 1), expect):
        x, y, G, label, p = _edge_case(kind, big)
        B = 2
        hint, tg = ops.unique_rows(x), ops.distinct_times(x)
        assert lib.lfm_batched_team_size(B, x.shape[0], G, hint, tg) == team, (kind, big, hint, tg)
        u = o.unconstrain(p.pack())
        U = np.stack([u, u + 0.05])
        val, grad, info = ops.batched_nlml_grad_unc(x, y, U, JITTER, G)
        assert not info.cpu().numpy().any()
        for b in range(B):
            v, g = o.nlml_and_grad_unc(U[b], x, y, JITTER)
            w = grad_close(grad[b].cpu().numpy(), g)
            _report(label, f"batched edge {kind} big={big} team={team}", w * GRAD_FLOOR)
            assert abs(val[b].item() - v) <= VAL_RTOL * abs(v) and w <= 1.0, (kind, big, w)


POSTERIOR_REGIMES = ["p53", "gamma5.25_l3.499", "gamma7.0_l2.5", "gamma8.75_l3.499", "offset", "offset_control"]
POST_TOL = 1e-11


def _post_inputs(r):
    p, x, y, var = problem(r, seed=41)
    lat = r.latent()
    gene = np.concatenate([np.stack([lat[:, 0], np.full(lat.shape[0], g), np.ones(lat.shape[0])], 1)
                           for g in range(r.G)])
    return p, x, y, var, lat, gene


def _prior_var(p, rows):
    return np.array([o.cross_covariance(p, rows[i:i + 1], rows[i:i + 1])[0, 0] for i in range(rows.shape[0])]) + p.jitter


@pytest.mark.gpu
@pytest.mark.parametrize("name", POSTERIOR_REGIMES)
def test_posteriors_match_oracle(cuda, name):
    """ops.latent_posterior / gene_posterior and their batched forms: the variance (and covariance) entry by entry on
    the scale of the prior variance at that entry, the mean on the scale of its prior standard deviation times |y - mu|."""
    from dis_project_b200 import ops
    r = BY_NAME[name]
    p, x, y, var, lat, gene = _post_inputs(r)
    th = p.pack()
    zs = np.max(np.abs(y - o.mean_function(p, x)))
    m_ref, v_ref = o.latent_predict(p, lat, x, y, var)
    gm_ref, gc_ref = o.multi_gene_predict(p, gene, x, y, var)
    lv, gv = _prior_var(p, lat), _prior_var(p, gene)
    gsc = np.sqrt(np.outer(gv, gv))

    def check(path, m, v, gm=None, gc=None, gvar=None):
        em = np.max(np.abs(m - m_ref) / (np.sqrt(lv) * zs)) if gm is None else np.max(np.abs(gm - gm_ref) / (np.sqrt(gv) * zs))
        ev = np.max(np.abs(v - v_ref) / lv) if gm is None else np.max(np.abs(gvar - np.diag(gc_ref)) / gv)
        ec = 0.0 if gc is None else np.max(np.abs(gc - gc_ref) / gsc)
        _report(name, path, max(em, ev, ec))
        assert max(em, ev, ec) <= POST_TOL, (name, path, em, ev, ec)

    m, v, info = ops.latent_posterior(x, y, var, th, JITTER, lat, r.G)
    assert int(info.item()) == 0
    check("latent_posterior", m.cpu().numpy(), v.cpu().numpy())
    m, c, v, info = ops.gene_posterior(x, y, var, th, JITTER, gene, r.G)
    assert int(info.item()) == 0
    check("gene_posterior", None, None, m.cpu().numpy(), c.cpu().numpy(), v.cpu().numpy())
    TH = np.stack([th, th])
    m, v, info = ops.batched_latent_posterior(x, y, var, TH, JITTER, lat, r.G)
    assert not info.cpu().numpy().any()
    check("batched_latent_posterior", m.cpu().numpy()[1], v.cpu().numpy()[1])
    m, c, v, info = ops.batched_gene_posterior(x, y, var, TH, JITTER, gene, r.G, full_cov=True)
    assert not info.cpu().numpy().any()
    check("batched_gene_posterior", None, None, m.cpu().numpy()[1], c.cpu().numpy()[1], v.cpu().numpy()[1])
