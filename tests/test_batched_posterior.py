"""Batched posteriors: latent_predict / multi_gene_predict of B fitted LFMs in one launch (include/lfm_b200.h,
lfm_batched_latent_posterior / lfm_batched_gene_posterior; ops.batched_latent_posterior / batched_gene_posterior).

CPU: a numpy restatement of the duplicate-row-compressed posterior against the dense oracle.  GPU: the kernels against
the oracle, the reference-executed goldens and the single-LFM path; independence of the batch, failure isolation and a
candidate-TF screen end to end."""
import ctypes as C
import json
import os

import numpy as np
import pytest
from scipy.linalg import cholesky, solve_triangular

from oracle import lfm_oracle as o

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RTOL = 1e-9
LITERAL_NOISE_TOL = 1e-8   # latent mean at the goldens' 'random' point and fit: the reference's own erf-sum noise
JIT = 1e-4


def relerr(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def het_problem(G, T, R, seed):
    """synthetic_problem with its variances scaled by U(0.5, 20), so that the variance term matters."""
    x, y, var, _ = o.synthetic_problem(G, T, R, seed=seed)
    return x, y, var * np.random.default_rng(seed + 1).uniform(0.5, 20.0, var.shape)


def non_uniform_design(seed):
    """Two replicates with four measurements of the second one missing: N = 36 rows that are not compressed."""
    x, y, var = het_problem(4, 5, 2, seed)
    keep = np.ones(x.shape[0], dtype=bool)
    keep[[27, 33, 36, 39]] = False
    return np.ascontiguousarray(x[keep]), np.ascontiguousarray(y[keep]), np.ascontiguousarray(var[keep])


def start_points(G, B, seed, scale=0.3):
    th0 = o.Params.reference_init(G).pack()
    TH = o.constrain(o.unconstrain(th0)[None, :] + scale * np.random.default_rng(seed).standard_normal((B, th0.shape[0])))
    TH[0] = th0
    return TH


def _compression(x):
    """(U x N incidence P^T, R) under the kernels' rule: compress only a uniform multiplicity R > 1, else U = N."""
    keys = [tuple(r) for r in x]
    first = {}
    cls = np.array([first.setdefault(k, len(first)) for k in keys])
    counts = np.bincount(cls)
    if counts.min() != counts.max() or counts[0] == 1:
        return np.eye(x.shape[0]), 1
    Pt = np.zeros((len(first), x.shape[0]))
    Pt[cls, np.arange(x.shape[0])] = 1.0
    return Pt, int(counts[0])


# ---- CPU: the compressed mathematics ---------------------------------------------------------------------------------
def compressed_posterior(p, x, y, var, xs, gene):
    """The kernels' formulas: latent (mean, var) or gene (mean, cov) from the U x U system M = diag(cbar) + R K_u."""
    Pt, R = _compression(x)
    xu = x[np.argmax(Pt, axis=1)]
    z = y - o.mean_function(p, x)
    c = var + (p.sigma**2 if gene else p.jitter)
    cbar = R / (Pt @ (1.0 / c))
    q = cbar * (Pt @ (z / c))
    L = cholesky(np.diag(cbar) + R * o.gram(p, xu), lower=True)
    beta = solve_triangular(L, solve_triangular(L, q, lower=True), lower=True, trans="T")
    kxu = o.cross_covariance(p, xu, xs)
    V = solve_triangular(L, kxu, lower=True)
    mean = o.mean_function(p, xs) + kxu.T @ beta
    if gene:
        cov = o.gram(p, xs) - R * V.T @ V
        cov[np.diag_indices_from(cov)] += p.jitter
        return mean, cov
    kdiag = np.array([o.cross_covariance(p, xs[i:i + 1], xs[i:i + 1])[0, 0] for i in range(xs.shape[0])])
    return mean, kdiag + p.jitter - R * np.sum(V * V, axis=0) + p.jitter


@pytest.mark.parametrize("design", ["R1", "R3", "non_uniform", "zero_variances"])
def test_compressed_posterior_matches_the_dense_oracle(design):
    if design == "non_uniform":
        x, y, var = non_uniform_design(71)
    else:
        x, y, var = het_problem(5, 7, 1 if design == "R1" else 3, 71)
        if design == "zero_variances":   # cbar_u = jitter (latent) or sigma^2 (gene) exactly
            var = np.zeros_like(var)
    G = int(x[:, 1].max()) + 1
    assert (_compression(x)[1] > 1) == (design in ("R3", "zero_variances"))
    p = o.Params.unpack(o.Params.reference_init(G).pack() * np.random.default_rng(72).uniform(0.8, 1.2, 3 * G + 2), JIT)
    xs, xg = o.generate_test_times(100), o.generate_test_times_pred(100, G)
    m, v = compressed_posterior(p, x, y, var, xs, False)
    m_ref, v_ref = o.latent_predict(p, xs, x, y, var)
    # without variances the latent covariance is K + 1e-4 I: two rearrangements of the same solve agree to kappa * eps
    # (3.7e-10 here), not to 1e-12; every other case has kappa * eps < 1e-12
    kappa = np.linalg.cond(o.gram(p, x) + np.diag(var) + p.jitter * np.eye(x.shape[0]))
    tol = max(1e-12, kappa * np.finfo(np.float64).eps)
    assert relerr(m, m_ref) < tol and relerr(v, v_ref) < tol
    gm, gc = compressed_posterior(p, x, y, var, xg, True)
    gm_ref, gc_ref = o.multi_gene_predict(p, xg, x, y, var)
    assert relerr(gm, gm_ref) < 1e-12 and relerr(gc, gc_ref) < 1e-12


def test_batched_posterior_argument_errors():
    """Shapes are checked before anything reaches the device."""
    from dis_project_b200 import ops
    x, y, var = het_problem(5, 7, 3, 5)
    TH = start_points(5, 3, 6)
    xs, xg = o.generate_test_times(10), o.generate_test_times_pred(4, 5)
    with pytest.raises(ValueError):
        ops.batched_latent_posterior(x, y, var, TH[:, :-1], JIT, xs, 5)          # theta is not (B, P)
    with pytest.raises(ValueError):
        ops.batched_latent_posterior(x, y, var, TH[0], JIT, xs, 5)               # one flat theta
    with pytest.raises(ValueError):
        ops.batched_latent_posterior(x, y[:-1], var, TH, JIT, xs, 5)             # y
    with pytest.raises(ValueError):
        ops.batched_latent_posterior(x, y, np.stack([var] * 2), TH, JIT, xs, 5)  # variances (2, N) for B = 3
    with pytest.raises(ValueError):
        ops.batched_latent_posterior(x, y, None, TH, JIT, xs, 5)                 # variances are required
    with pytest.raises(ValueError):
        ops.batched_gene_posterior(x, y, var, TH, JIT, xg[:-1], 5)               # T* % G
    bad = x.copy()
    bad[0, 2] = 0.0
    with pytest.raises(ValueError):
        ops.batched_latent_posterior(bad, y, var, TH, JIT, xs, 5)                # training flags


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _host(*ts):
    return [None if t is None else t.cpu().numpy() for t in ts]


def _problem(design, per_lfm, B):
    if design == "non_uniform":
        x, y, var = non_uniform_design(201)
        G = 4
    else:
        G, T, R = design
        x, y, var = het_problem(G, T, R, 201 + G * T * R)
    TH = start_points(G, B, 202)
    if per_lfm:
        rng = np.random.default_rng(203)
        y = y[None, :] + 0.1 * rng.standard_normal((B, y.shape[0]))
        var = var[None, :] * rng.uniform(0.5, 2.0, (B, var.shape[0]))
    return G, x, y, var, TH


PARITY = [   # design (G, T, R) or "non_uniform", B, per-LFM y and variances, latent T*, gene T* (full covariance up to 500)
    ((5, 7, 3), 1, False, 1, 5),
    ((5, 7, 3), 7, True, 100, 500),
    ((5, 7, 1), 300, False, 100, 100),
    ((4, 32, 1), 7, True, 5000, 500),      # N = 128; 5000 test rows span many chunks
    ((3, 12, 2), 7, False, 100, 99),
    ("non_uniform", 7, True, 100, 100),
]


@pytest.mark.gpu
@pytest.mark.parametrize("design,B,per_lfm,Tl,Tg", PARITY)
def test_batched_posteriors_match_the_oracle(cuda, design, B, per_lfm, Tl, Tg):
    from dis_project_b200 import ops
    G, x, y, var, TH = _problem(design, per_lfm, B)
    xs, xg = o.generate_test_times(Tl), o.generate_test_times_pred(Tg // G, G)
    mean, lvar, info = _host(*ops.batched_latent_posterior(x, y, var, TH, JIT, xs, G))
    assert mean.shape == (B, Tl) and not info.any()
    gm, gc, gv, ginfo = _host(*ops.batched_gene_posterior(x, y, var, TH, JIT, xg, G, full_cov=True))
    assert gc.shape == (B, Tg, Tg) and not ginfo.any()
    gm2, none, gv2, _ = ops.batched_gene_posterior(x, y, var, TH, JIT, xg, G)
    assert none is None and relerr(gm2.cpu().numpy(), gm) == 0.0 and relerr(gv2.cpu().numpy(), gv) < 1e-12
    assert np.array_equal(gv, np.diagonal(gc, axis1=1, axis2=2))                  # var is the diagonal of cov
    for b in range(B):
        yb, vb = (y[b], var[b]) if per_lfm else (y, var)
        p = o.Params.unpack(TH[b], JIT)
        # the oracle's mean_function wants T* % G == 0; latent rows carry flag 0 (mean_t = 0 in every positional block),
        # so the first T* rows of G stacked copies are the posterior at xs
        m_ref, v_ref = (a[:Tl] for a in o.latent_predict(p, np.tile(xs, (G, 1)), x, yb, vb))
        assert relerr(mean[b], m_ref) < RTOL and relerr(lvar[b], v_ref) < RTOL, b
        gm_ref, gc_ref = o.multi_gene_predict(p, xg, x, yb, vb)
        assert relerr(gm[b], gm_ref) < RTOL and relerr(gc[b], gc_ref) < RTOL, b
        assert relerr(gv[b], np.diag(gc_ref)) < RTOL


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["p53_rep0", "p53_all", "p53_sub3"])
def test_batched_posteriors_reproduce_the_reference_goldens(cuda, name):
    """Every executed point and the reference's own fitted parameters as the rows of one batch, against the moments the
    reference computed (tolerances of tests/test_ref_parity.py)."""
    from dis_project_b200 import ops
    with open(os.path.join(GOLD, f"ref_{name}.json")) as fh:
        c = json.load(fh)
    X, y, var, xs, xg = (np.array(c[k]) for k in ("X", "y", "variances", "Xstar", "Xgene"))
    G, jit = c["G"], c["jitter"]
    rows = c["points"] + [dict(c["fit"], label="fit")]
    TH = np.stack([np.array(r["theta"]) for r in rows])
    mean, lvar, info = _host(*ops.batched_latent_posterior(X, y, var, TH, jit, xs, G))
    gm, gc, gv, ginfo = _host(*ops.batched_gene_posterior(X, y, var, TH, jit, xg, G, full_cov=True))
    assert not info.any() and not ginfo.any()
    for b, r in enumerate(rows):
        assert relerr(mean[b], r["latent_mean"]) < (RTOL if r["label"] == "init" else LITERAL_NOISE_TOL)
        assert relerr(np.sqrt(lvar[b]), r["latent_std"]) < RTOL
        assert relerr(gm[b], r["gene_mean"]) < RTOL and relerr(np.sqrt(gv[b]), r["gene_std"]) < RTOL
        if "gene_cov_row0" in r:
            assert relerr(gc[b, 0], r["gene_cov_row0"]) < RTOL


@pytest.mark.gpu
@pytest.mark.parametrize("design,per_lfm", [((5, 7, 3), True), ((4, 32, 1), False), ("non_uniform", False)])
def test_batched_posteriors_equal_the_single_lfm_path(cuda, design, per_lfm):
    from dis_project_b200 import ops
    B = 9
    G, x, y, var, TH = _problem(design, per_lfm, B)
    xs, xg = o.generate_test_times(300), o.generate_test_times_pred(60, G)
    mean, lvar, _ = _host(*ops.batched_latent_posterior(x, y, var, TH, JIT, xs, G))
    gm, gc, gv, _ = _host(*ops.batched_gene_posterior(x, y, var, TH, JIT, xg, G, full_cov=True))
    for b in range(B):
        yb, vb = (y[b], var[b]) if per_lfm else (y, var)
        m1, v1, i1 = _host(*ops.latent_posterior(x, yb, vb, TH[b], JIT, xs, G))
        g1, c1, w1, j1 = _host(*ops.gene_posterior(x, yb, vb, TH[b], JIT, xg, G))
        assert i1[0] == 0 and j1[0] == 0
        assert relerr(mean[b], m1) < RTOL and relerr(lvar[b], v1) < RTOL
        assert relerr(gm[b], g1) < RTOL and relerr(gc[b], c1) < RTOL and relerr(gv[b], w1) < RTOL


@pytest.mark.gpu
def test_batched_posterior_rows_do_not_depend_on_the_batch(cuda):
    """Row b is bit-identical alone, inside a larger batch at any position, and across repeated calls."""
    import torch
    from dis_project_b200 import ops
    B = 40
    G, x, y, var, TH = _problem((5, 7, 3), True, B)
    xs, xg = o.generate_test_times(150), o.generate_test_times_pred(30, G)
    lat = ops.batched_latent_posterior(x, y, var, TH, JIT, xs, G)
    gen = ops.batched_gene_posterior(x, y, var, TH, JIT, xg, G, full_cov=True)
    assert all(torch.equal(a, b) for a, b in zip(lat, ops.batched_latent_posterior(x, y, var, TH, JIT, xs, G)))
    assert all(torch.equal(a, b) for a, b in zip(gen, ops.batched_gene_posterior(x, y, var, TH, JIT, xg, G, full_cov=True)))
    perm = np.random.default_rng(5).permutation(B)
    lp = ops.batched_latent_posterior(x, y[perm], var[perm], TH[perm], JIT, xs, G)
    gp = ops.batched_gene_posterior(x, y[perm], var[perm], TH[perm], JIT, xg, G, full_cov=True)
    for k, b in enumerate(perm):
        assert all(torch.equal(a[b], c[k]) for a, c in zip(lat, lp))
        assert all(torch.equal(a[b], c[k]) for a, c in zip(gen, gp))
    for b in (0, 17, B - 1):
        one = ops.batched_latent_posterior(x, y[b:b + 1], var[b:b + 1], TH[b:b + 1], JIT, xs, G)
        assert all(torch.equal(a[b], c[0]) for a, c in zip(lat, one))
        one = ops.batched_gene_posterior(x, y[b:b + 1], var[b:b + 1], TH[b:b + 1], JIT, xg, G, full_cov=True)
        assert all(torch.equal(a[b], c[0]) for a, c in zip(gen, one))
    # shared y and variances are the same as every LFM carrying copies of them
    s = ops.batched_latent_posterior(x, y[3], var[3], TH, JIT, xs, G)
    r = ops.batched_latent_posterior(x, np.repeat(y[3:4], B, 0), np.repeat(var[3:4], B, 0), TH, JIT, xs, G)
    assert all(torch.equal(a, c) for a, c in zip(s, r))
    s1 = ops.batched_latent_posterior(x, y[3], var[3].reshape(-1, 1), TH, JIT, xs, G)
    assert all(torch.equal(a, c) for a, c in zip(s, s1))


@pytest.mark.gpu
def test_batched_posterior_failures_are_isolated(cuda):
    """A negative variance of one LFM gives info = 1 and NaN for that LFM only; the other rows are bit-identical to a
    batch without it.  A too-small unique-row hint gives info = -1; N = 129 is refused."""
    import torch
    from dis_project_b200 import _lib, ops
    B = 6
    G, x, y, var, TH = _problem((5, 7, 3), True, B)
    xs, xg = o.generate_test_times(50), o.generate_test_times_pred(10, G)
    bad = var.copy()
    bad[2, ::4] = -50.0
    keep = [b for b in range(B) if b != 2]
    for fn, kw, xt in ((ops.batched_latent_posterior, {}, xs), (ops.batched_gene_posterior, dict(full_cov=True), xg)):
        out = fn(x, y, bad, TH, JIT, xt, G, **kw)
        ref = fn(x, y[keep], var[keep], TH[keep], JIT, xt, G, **kw)
        info = out[-1].cpu().numpy()
        assert info[2] == 1 and np.all(info[keep] == 0)
        for a, r in zip(out[:-1], ref[:-1]):
            if a is None:
                continue
            assert torch.isnan(a[2]).all()
            assert torch.equal(a[keep], r)
    # unique_rows_hint below the U the kernel finds
    l = _lib.lib()
    X, Y, V = (torch.as_tensor(np.ascontiguousarray(a), device="cuda") for a in (x, y, var))
    T = torch.as_tensor(TH, device="cuda")
    Xs = torch.as_tensor(xs, device="cuda")
    N = x.shape[0]
    assert ops.unique_rows(x) == 35
    ws = torch.empty(int(l.lfm_batched_posterior_workspace_bytes(B, N, G, 50, 20, 0)), dtype=torch.uint8, device="cuda")
    mean, lv = torch.empty((B, 50), dtype=torch.float64, device="cuda"), torch.empty((B, 50), dtype=torch.float64, device="cuda")
    info = torch.zeros(B, dtype=torch.int32, device="cuda")
    _lib.check(l.lfm_batched_latent_posterior(ops._stream(), B, N, G, X.data_ptr(), Y.data_ptr(), N, V.data_ptr(), N,
                                              T.data_ptr(), JIT, 50, Xs.data_ptr(), 20, ws.data_ptr(), ws.numel(),
                                              mean.data_ptr(), lv.data_ptr(), info.data_ptr()), "latent")
    assert np.all(info.cpu().numpy() == -1) and torch.isnan(mean).all() and torch.isnan(lv).all()
    # workspace too small for the full covariance; N > 128
    assert l.lfm_batched_gene_posterior(ops._stream(), B, N, G, X.data_ptr(), Y.data_ptr(), N, V.data_ptr(), N,
                                        T.data_ptr(), JIT, 50, Xs.data_ptr(), 35, ws.data_ptr(), ws.numel(), mean.data_ptr(),
                                        mean.data_ptr(), None, info.data_ptr()) == -4
    x9, y9, v9 = het_problem(3, 43, 1, 7)
    assert x9.shape[0] == 129
    with pytest.raises(_lib.LfmError):
        ops.batched_latent_posterior(x9, y9, v9, start_points(3, 2, 8), JIT, xs, 3)
    assert l.lfm_batched_posterior_workspace_bytes(B, 129, 3, 50, 0, 1) == 0


@pytest.mark.gpu
def test_candidate_tf_screen_then_batched_posteriors(cuda):
    """multi_start_fit with one row of observations per LFM (candidate TFs), then both posteriors of every fitted LFM
    from MultiStartResult.theta in one launch each, equal to the single-LFM path."""
    from dis_project_b200 import ops
    from dis_project_b200.batched import multi_start_fit
    G, T, R, B = 5, 7, 3, 12
    x, y, var = het_problem(G, T, R, 301)
    Y = y[None, :] + 0.2 * np.random.default_rng(302).standard_normal((B, y.shape[0]))
    TH0 = start_points(G, B, 303)
    res = multi_start_fit(x, Y, TH0, JIT, num_iters=60, chunk=None, variances=var)
    assert not np.any(res.info) and res.theta.shape == (B, 3 * G + 2)
    xs, xg = o.generate_test_times(100), o.generate_test_times_pred(20, G)
    mean, lvar, info = _host(*ops.batched_latent_posterior(x, Y, var, res.theta, JIT, xs, G))
    gm, _, gv, ginfo = _host(*ops.batched_gene_posterior(x, Y, var, res.theta, JIT, xg, G))
    assert not info.any() and not ginfo.any()
    for b in range(B):
        m1, v1, _ = _host(*ops.latent_posterior(x, Y[b], var, res.theta[b], JIT, xs, G))
        g1, _, w1, _ = _host(*ops.gene_posterior(x, Y[b], var, res.theta[b], JIT, xg, G, full_cov=False))
        assert relerr(mean[b], m1) < RTOL and relerr(lvar[b], v1) < RTOL
        assert relerr(gm[b], g1) < RTOL and relerr(gv[b], w1) < RTOL
