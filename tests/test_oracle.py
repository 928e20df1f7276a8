"""Pins the CPU oracle (no GPU needed).  The reference has no tests or golden vectors of its own
(SURVEY.md 8c: "parity unpinned"), so the oracle is anchored on
  (1) a 50-digit mpmath evaluation of the reference's formulas (src/model.py:197-365), written
      independently from the numpy code,
  (2) the GPyTorch twin's formulas (src/gpytorch_alfi/model_alfi.py:302-382, 414-476) restated,
  (3) autograd versus closed-form gradients,
  (4) the constants the reference hard-codes, and the committed golden vectors."""
import glob
import json
import os

import mpmath as mp
import numpy as np
import pytest

from oracle import lfm_oracle as o

mp.mp.dps = 50
# oracle-generated vectors (make_golden.py); the reference-executed ref_*.json are consumed by test_ref_parity.py
GOLDEN = sorted(g for g in glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.json"))
                if not os.path.basename(g).startswith("ref_"))


def mp_h(d, l, j, k, t1, t2):
    """model.py:343-362, literally, in 50-digit arithmetic."""
    d = [mp.mpf(float(v)) for v in d]
    l, t1, t2 = mp.mpf(float(l)), mp.mpf(float(t1)), mp.mpf(float(t2))
    t_dist = t2 - t1
    gk = d[k] * l / 2
    multiplier = mp.e ** (gk**2) / (d[j] + d[k])
    first = mp.e ** (-d[k] * t_dist) * (mp.erf(t_dist / l - gk) + mp.erf(t1 / l + gk))
    second = mp.e ** (-(d[k] * t2 + d[j] * t1)) * (mp.erf(t2 / l - gk) + mp.erf(gk))
    return multiplier * (first - second)


def mp_kxx(p, t, j, tp, k):
    mult = mp.mpf(float(p.s[j])) * mp.mpf(float(p.s[k])) * mp.mpf(float(p.l)) * mp.sqrt(mp.pi) / 2
    return mult * (mp_h(p.d, p.l, k, j, tp, t) + mp_h(p.d, p.l, j, k, t, tp))


def mp_kxf(p, tg, j, tl):
    d, l, s = mp.mpf(float(p.d[j])), mp.mpf(float(p.l)), mp.mpf(float(p.s[j]))
    tg, tl = mp.mpf(float(tg)), mp.mpf(float(tl))
    td = tg - tl
    g = d * l / 2
    return l * mp.sqrt(mp.pi) / 2 * s * mp.e ** (g**2) * mp.e ** (-d * td) * (mp.erf(td / l - g) + mp.erf(tl / l + g))


def rand_params(G, seed):
    rng = np.random.default_rng(seed)
    return o.Params(d=rng.uniform(0.2, 1.0, G), s=rng.uniform(0.5, 1.5, G), b=rng.uniform(0.01, 0.1, G),
                    l=float(rng.uniform(0.8, 3.2)), sigma=1.0, jitter=1e-4)


def test_kernel_entries_against_mpmath():
    p = rand_params(5, 0)
    rng = np.random.default_rng(1)
    worst_xx = worst_xf = 0.0
    for _ in range(150):
        t, tp = rng.uniform(0, 12, 2)
        j, k = rng.integers(0, 5, 2)
        a = np.array([[t, j, 1.0]]); b = np.array([[tp, k, 1.0]]); f = np.array([[tp, -1.0, 0.0]])
        ref = mp_kxx(p, t, j, tp, k)
        got = o.cross_covariance(p, a, b)[0, 0]
        worst_xx = max(worst_xx, abs(float((mp.mpf(float(got)) - ref))) / max(1e-3, abs(float(ref))))
        ref = mp_kxf(p, t, j, tp)
        got = o.cross_covariance(p, a, f)[0, 0]
        got_t = o.cross_covariance(p, f, a)[0, 0]
        assert got == got_t  # k_xf and its transpose branch agree (model.py:191-192)
        worst_xf = max(worst_xf, abs(float(mp.mpf(float(got)) - ref)) / max(1e-3, abs(float(ref))))
    assert worst_xx < 5e-13 and worst_xf < 5e-13
    # k_ff with the reference's 2*l denominator (SURVEY Q1)
    f1 = np.array([[1.0, -1, 0]]); f2 = np.array([[3.5, -1, 0]])
    assert o.cross_covariance(p, f1, f2)[0, 0] == pytest.approx(np.exp(-(2.5**2) / (2 * p.l)), rel=1e-15)


def test_literal_erf_sum_noise_is_bounded():
    """The cancellation-free erf sums (oracle.erfsum) and the reference's literal sums agree to the
    literal form's own rounding noise: <= 1e-16 * exp(D |dt|) absolute (SURVEY Q7)."""
    p = rand_params(6, 8)
    x = o.make_inputs(6, 25)
    xs = o.generate_test_times(300)
    acc = o.cross_covariance(p, x, xs)
    try:
        o.LITERAL_ERF_SUMS = True
        lit = o.cross_covariance(p, x, xs)
        litg = o.gram(p, x)
    finally:
        o.LITERAL_ERF_SUMS = False
    accg = o.gram(p, x)
    assert np.max(np.abs(acc - lit)) < 2e-16 * np.exp(1.0 * 13.0)
    assert np.max(np.abs(accg - litg)) < 2e-16 * np.exp(1.0 * 12.0) * 10
    # and the accurate form is the one closer to the exact value
    i, jx = np.unravel_index(np.argmax(np.abs(acc - lit)), acc.shape)
    exact = float(mp_kxf(p, x[i, 0], int(x[i, 1]), xs[jx, 0]))
    assert abs(acc[i, jx] - exact) <= abs(lit[i, jx] - exact)


def test_twin_block_formulas_agree():
    """GPyTorch/ALFI twin (model_alfi.py:302-382): k_xx(j,k,t1,t2) block = S_j S_k l sqrt(pi)/2 (h_kj(t2,t1)^T + h_jk(t1,t2))."""
    p = rand_params(4, 3)
    times = np.linspace(0, 12, 9)
    from scipy.special import erf

    def twin_h(k, j, t2, t1):  # model_alfi.py:343-378 restated: h_kj with decays D_k, D_j and gamma_k
        l = p.l
        tp, t = np.meshgrid(t1, t2, indexing="ij")   # tprime_mat (rows), t_mat (cols)
        dist = tp - t
        gk = p.d[k] * l / 2
        m = np.exp(gk**2) / (p.d[j] + p.d[k])
        a = np.exp(-p.d[k] * dist) * (erf(dist / l - gk) + erf(t / l + gk))
        b = np.exp(-(p.d[k] * tp + p.d[j] * t)) * (erf(tp / l - gk) + erf(gk))
        return m * (a - b)

    for j in range(4):
        for k in range(4):
            blk = p.s[j] * p.s[k] * p.l * np.sqrt(np.pi) / 2 * (twin_h(k, j, times, times).T + twin_h(j, k, times, times))
            xa = np.stack((times, np.full(9, j), np.ones(9)), axis=-1)
            xb = np.stack((times, np.full(9, k), np.ones(9)), axis=-1)
            ours = o.cross_covariance(p, xa, xb)
            assert np.max(np.abs(ours - blk)) < 1e-10 * max(1.0, np.max(np.abs(blk)))


def test_gram_symmetry_and_structure():
    p = rand_params(5, 4)
    x = o.make_inputs(5, 7, 3)
    K = o.gram(p, x)
    assert np.max(np.abs(K - K.T)) < 1e-13  # k_xx is the sum of the two transposed h terms (model.py:231)
    assert np.array_equal(K[:35, :35], K[35:70, 70:105])  # replicates share the time grid
    assert np.allclose(o.gram_xx_fast(p, x), K, rtol=0, atol=1e-15)


def test_mean_function_is_positional():
    """model.py:143-149: blocks of N // G rows, not the gene column (SURVEY Q3)."""
    p = rand_params(5, 5)
    x = o.make_inputs(5, 7, 3)
    m = o.mean_function(p, x)
    assert np.array_equal(m, np.repeat(p.b / p.d, 21))
    xs = o.generate_test_times(100)
    assert np.all(o.mean_function(p, xs) == 0)
    with pytest.raises(ValueError):
        o.mean_function(p, x[:33])


def test_gradients_two_derivations():
    for (G, T, R, seed) in ((5, 7, 1, 0), (5, 7, 3, 1), (3, 6, 1, 2)):
        x, y, _, _ = o.synthetic_problem(G, T, R, seed=seed)
        u = o.unconstrain(rand_params(G, seed + 10).pack())
        v1, g1 = o.nlml_and_grad_unc(u, x, y, 1e-4)
        v2, g2 = o.nlml_and_grad_unc_autograd(u, x, y, 1e-4)
        assert abs(v1 - v2) < 1e-11 * abs(v2)
        assert np.max(np.abs(g1 - g2)) < 1e-10 * np.max(np.abs(g2))
        assert abs(v1 - o.nlml(o.Params.unpack(o.constrain(u), 1e-4), x, y)) < 1e-11 * abs(v1)


def test_gradient_magnitudes_against_dense_derivatives():
    """nlml_and_grad(magnitudes=True): M_k against the same sums taken over the dense derivative matrices dK/dtheta_k
    (torch autograd of the kernel, entry by entry) and dmu/dtheta_k; M_k >= |grad_k|; the value and the gradient are
    the default call's, bit for bit.  Replicates put equal genes at different times, so entries whose row and column
    are the same gene (one term for the two decay paths) are covered."""
    import torch
    for (G, T, R, seed) in ((3, 5, 2, 0), (4, 6, 1, 1)):
        x, y, var, _ = o.synthetic_problem(G, T, R, seed=seed)
        p = rand_params(G, seed + 30)
        p.sigma = 0.8
        v0, g0 = o.nlml_and_grad(p, x, y, chunk=7)
        v, g, M = o.nlml_and_grad(p, x, y, chunk=7, magnitudes=True)
        assert v == v0 and np.array_equal(g, g0)
        n, P = x.shape[0], 3 * G + 2
        t = torch.as_tensor(x[:, 0])
        gi = torch.as_tensor(x[:, 1].astype(np.int64))

        def kern(th):
            d, s, l = th[:G], th[G:2 * G], th[3 * G]

            def hh(j, k, t1, t2):
                g_ = d[k] * l / 2
                return torch.exp(g_ ** 2) / (d[j] + d[k]) * (
                    torch.exp(-d[k] * (t2 - t1)) * (torch.erf((t2 - t1) / l - g_) + torch.erf(t1 / l + g_))
                    - torch.exp(-(d[k] * t2 + d[j] * t1)) * (torch.erf(t2 / l - g_) + torch.erf(g_)))
            j, k, tt, tp = gi[:, None], gi[None, :], t[:, None], t[None, :]
            return s[j] * s[k] * l * np.sqrt(np.pi) / 2 * (hh(k, j, tp, tt) + hh(j, k, tt, tp))

        def mean(th):
            return torch.repeat_interleave(th[2 * G:3 * G] / th[:G], n // G)

        th = torch.as_tensor(p.pack())
        dK = torch.autograd.functional.jacobian(kern, th).numpy()      # (n, n, P)
        dmu = torch.autograd.functional.jacobian(mean, th).numpy()     # (n, P)
        S = o.sigma_matrix(p, x)
        Sinv = np.linalg.inv(S)
        alpha = np.linalg.solve(S, y - o.mean_function(p, x))
        Kbar = 0.5 * (Sinv - np.outer(alpha, alpha))
        ref = np.abs(Kbar[:, :, None] * dK).sum(axis=(0, 1)) + np.abs(alpha[:, None] * dmu).sum(axis=0)
        ref[P - 1] = p.sigma * (np.abs(np.diag(Sinv)).sum() + alpha @ alpha)
        gref = (Kbar[:, :, None] * dK).sum(axis=(0, 1)) - alpha @ dmu
        gref[P - 1] = 2 * p.sigma * np.trace(Kbar)
        # the closed-form partials and autograd round each entry's derivative differently: 1.2e-12 of M_k measured
        assert np.max(np.abs(g - gref) / ref) < 1e-10           # the brute force computes the same gradient
        assert np.max(np.abs(M - ref) / ref) < 1e-10, (M, ref)
        assert np.all(M >= np.abs(g))
        assert np.min(M / np.abs(g)) < 10.0                      # a scale of the component, not of the whole gradient
        # unconstrained: the chain rule scales each term by the bijector's derivative
        u = o.unconstrain(p.pack())
        vu, gu = o.nlml_and_grad_unc(u, x, y, p.jitter)
        _, gc, Mc = o.nlml_and_grad(o.Params.unpack(o.constrain(u), p.jitter), x, y, magnitudes=True)
        assert np.array_equal(gu, gc * o.constrain_jac(u)) and np.all(Mc * np.abs(o.constrain_jac(u)) >= np.abs(gu))


def test_heteroscedastic_objective_two_derivations():
    """sigma_matrix(variances=...): the GPyTorch twin's training convention (measurement variances on the diagonal,
    src/gpytorch_alfi/model_alfi.py:294-299).  Closed-form gradient against torch autograd of the literal expressions;
    the variances are constants, so only Sigma changes; zero variances reproduce the GPJax objective bit for bit."""
    for (G, T, R, seed) in ((5, 7, 3, 3), (3, 6, 1, 4)):
        x, y, var, _ = o.synthetic_problem(G, T, R, seed=seed)
        u = o.unconstrain(rand_params(G, seed + 20).pack())
        v0, g0 = o.nlml_and_grad_unc(u, x, y, 1e-4)
        vz, gz = o.nlml_and_grad_unc(u, x, y, 1e-4, variances=np.zeros_like(var))
        assert vz == v0 and np.array_equal(gz, g0)
        v1, g1 = o.nlml_and_grad_unc(u, x, y, 1e-4, variances=var)
        v2, g2 = o.nlml_and_grad_unc_autograd(u, x, y, 1e-4, variances=var)
        assert abs(v1 - v2) < 1e-11 * abs(v2)
        assert np.max(np.abs(g1 - g2)) < 1e-10 * np.max(np.abs(g2))
        assert abs(v1 - o.nlml(o.Params.unpack(o.constrain(u), 1e-4), x, y, variances=var)) < 1e-11 * abs(v1)
        assert abs(v1 - v0) > 1e-6 * abs(v0)   # the term is not a no-op
        S = o.sigma_matrix(o.Params.unpack(o.constrain(u), 1e-4), x, var)
        S0 = o.sigma_matrix(o.Params.unpack(o.constrain(u), 1e-4), x)
        assert np.allclose(np.diag(S) - np.diag(S0), var.reshape(-1), rtol=0, atol=1e-15)
        assert np.array_equal(S - np.diag(np.diag(S)), S0 - np.diag(np.diag(S0)))


def test_reference_constants_and_bijectors():
    p = o.Params.reference_init(5)
    assert np.all(p.d == 0.4) and np.all(p.s == 1.0) and np.all(p.b == 0.05) and p.l == 2.5 and p.sigma == 1.0
    th = p.pack()
    u = o.unconstrain(th)
    assert np.allclose(o.constrain(u), th, rtol=1e-15, atol=0)
    assert u[15] == pytest.approx(np.log((2.5 - 0.5) / (3.5 - 2.5)))  # logit of the Sigmoid(0.5, 3.5) bijector
    assert u[0] == pytest.approx(np.log(np.expm1(0.4)))
    h = 1e-6
    jac = o.constrain_jac(u)
    fd = (o.constrain(u + h) - o.constrain(u - h)) / (2 * h)
    assert np.allclose(jac, fd, rtol=1e-8)


def test_trainer_hook_semantics():
    """Q5: the p21 hook fires after step 0 in unconstrained space, and again in constrained space."""
    x, y, _, _ = o.synthetic_problem(5, 7, 1, seed=3)
    th0 = o.Params.reference_init(5).pack()
    th, hist = o.fit(th0, x, y, 1e-4, num_iters=3)
    assert th[3] == 0.8 and th[8] == 1.0
    th1, _ = o.fit(th0, x, y, 1e-4, num_iters=1)
    # after one step: raw values 0.8 / 1.0 were written in unconstrained space, then overwritten again
    th1n, _ = o.fit(th0, x, y, 1e-4, num_iters=1, fix_params=False)
    assert th1n[3] != 0.8
    assert hist[0] == pytest.approx(o.nlml(o.Params.unpack(th0, 1e-4), x, y), rel=1e-13)
    th3, _ = o.fit(o.Params.reference_init(3).pack(), *o.synthetic_problem(3, 6, 1, seed=1)[:2], 1e-4, num_iters=2)
    assert th3.shape == (11,)  # index 3 out of range: hook silently dropped


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(g) for g in GOLDEN])
def test_oracle_reproduces_golden(path):
    g = json.load(open(path))
    G = g["G"]
    p = o.Params.unpack(np.array(g["theta"]), g["jitter"])
    x, y, var = np.array(g["X"]), np.array(g["y"]), np.array(g["variances"])
    rows = np.array(g["K_rows"])
    assert np.allclose(o.cross_covariance(p, rows, rows), np.array(g["K_block"]), rtol=1e-13, atol=1e-15)
    v, gr = o.nlml_and_grad(p, x, y)
    assert v == pytest.approx(g["nlml"], rel=1e-12)
    assert np.allclose(gr, g["grad_constrained"], rtol=1e-9, atol=1e-11 * np.max(np.abs(gr)))
    m, pv = o.latent_predict(p, np.array(g["Xstar"]), x, y, var)
    assert np.allclose(m, g["posterior_mean"], rtol=1e-10, atol=1e-12)
    assert np.allclose(pv, g["posterior_var"], rtol=1e-10, atol=1e-12)
    assert G == p.num_genes


# ---- whole-path anchor in 50-digit arithmetic (independent of numpy / LAPACK) ------------------------------------
def _mp_nlml(theta, x, y, jitter, G):
    """objectives.py:64-78 over model.py:124-149,197-235 literally: mean, Sigma = K + (jitter + sigma^2) I, mpmath
    Cholesky, -log N(y; mu, Sigma)."""
    th = [mp.mpf(v) for v in theta]
    d, s, b, l, sigma = th[:G], th[G:2 * G], th[2 * G:3 * G], th[3 * G], th[3 * G + 1]

    class P:  # the attributes mp_kxx reads
        pass
    P.d, P.s, P.l = d, s, l
    N = x.shape[0]
    block = N // G
    mu = [b[min(i // block, G - 1)] / d[min(i // block, G - 1)] * int(x[i, 2]) for i in range(N)]
    K = mp.matrix(N, N)
    for i in range(N):
        for j in range(i + 1):
            v = mp_kxx_mp(P, mp.mpf(float(x[i, 0])), int(x[i, 1]), mp.mpf(float(x[j, 0])), int(x[j, 1]))
            K[i, j] = v
            K[j, i] = v
        K[i, i] += mp.mpf(jitter) + sigma**2
    L = mp.cholesky(K)
    z = mp.matrix([mp.mpf(float(y[i])) - mu[i] for i in range(N)])
    w = mp.lu_solve(L, z)  # exact triangular solve at 50 digits
    logdet = 2 * sum(mp.log(L[i, i]) for i in range(N))
    return (N * mp.log(2 * mp.pi) + logdet + sum(w[i] ** 2 for i in range(N))) / 2


def mp_h_mp(d, l, j, k, t1, t2):
    t_dist = t2 - t1
    gk = d[k] * l / 2
    multiplier = mp.e ** (gk**2) / (d[j] + d[k])
    first = mp.e ** (-d[k] * t_dist) * (mp.erf(t_dist / l - gk) + mp.erf(t1 / l + gk))
    second = mp.e ** (-(d[k] * t2 + d[j] * t1)) * (mp.erf(t2 / l - gk) + mp.erf(gk))
    return multiplier * (first - second)


def mp_kxx_mp(P, t, j, tp, k):
    mult = P.s[j] * P.s[k] * P.l * mp.sqrt(mp.pi) / 2
    return mult * (mp_h_mp(P.d, P.l, k, j, tp, t) + mp_h_mp(P.d, P.l, j, k, t, tp))


def test_nlml_and_gradient_against_mpmath_end_to_end():
    """NLML and its gradient (central differences at 50 digits, h = 1e-20) for a 3-gene x 4-time problem: pins the
    oracle's composition -- positional mean, jitter + sigma^2 on the diagonal, Cholesky log-det, quadratic form and
    every closed-form derivative -- on arithmetic that shares no code with it."""
    G, T = 3, 4
    x, y, var, _ = o.synthetic_problem(G, T, 1, seed=61)
    p = rand_params(G, 62)
    p.sigma = 0.8
    theta = p.pack()
    v, g = o.nlml_and_grad(p, x, y)
    ref = _mp_nlml([float(t) for t in theta], x, y, p.jitter, G)
    assert abs(float(mp.mpf(float(v)) - ref)) <= 1e-12 * abs(float(ref))
    h = mp.mpf(10) ** -20
    for idx in range(theta.shape[0]):
        tp = [mp.mpf(float(t)) for t in theta]; tm = list(tp)
        tp[idx] += h; tm[idx] -= h
        gref = (_mp_nlml(tp, x, y, p.jitter, G) - _mp_nlml(tm, x, y, p.jitter, G)) / (2 * h)
        assert abs(float(mp.mpf(float(g[idx])) - gref)) <= 1e-10 * max(1.0, abs(float(gref))), (idx, g[idx], gref)


def test_latent_posterior_against_mpmath_end_to_end():
    """model.py:420-463 at 50 digits: Sigma_p = K + diag(variances) + jitter I, mean = K_fx Sigma_p^-1 (y - mu),
    var = k_ff(t*, t*) + 2 jitter - k^T Sigma_p^-1 k (jitter enters twice, SURVEY Q4)."""
    G, T = 3, 4
    x, y, var, _ = o.synthetic_problem(G, T, 1, seed=63)
    p = rand_params(G, 64)
    ts = np.array([[0.7, -1.0, 0.0], [5.2, -1.0, 0.0], [11.0, -1.0, 0.0]])
    m, v = o.latent_predict(p, ts, x, y, var)

    class P:
        pass
    P.d = [mp.mpf(float(t)) for t in p.d]; P.s = [mp.mpf(float(t)) for t in p.s]; P.l = mp.mpf(float(p.l))
    b = [mp.mpf(float(t)) for t in p.b]
    N = x.shape[0]
    block = N // G
    K = mp.matrix(N, N)
    for i in range(N):
        for j in range(N):
            K[i, j] = mp_kxx_mp(P, mp.mpf(float(x[i, 0])), int(x[i, 1]), mp.mpf(float(x[j, 0])), int(x[j, 1]))
        K[i, i] += mp.mpf(float(var[i])) + mp.mpf(p.jitter)
    z = mp.matrix([mp.mpf(float(y[i])) - b[min(i // block, G - 1)] / P.d[min(i // block, G - 1)] for i in range(N)])
    Kinv = K ** -1
    for q in range(ts.shape[0]):
        k = mp.matrix([mp_kxf(p, x[i, 0], int(x[i, 1]), ts[q, 0]) for i in range(N)])
        mean = (k.T * Kinv * z)[0]
        vv = 1 + 2 * mp.mpf(p.jitter) - (k.T * Kinv * k)[0]
        assert abs(float(mp.mpf(float(m[q])) - mean)) <= 1e-11 * max(1.0, abs(float(mean)))
        assert abs(float(mp.mpf(float(v[q])) - vv)) <= 1e-11 * max(1.0, abs(float(vv)))


# ---- the extended-precision linear algebra the dense factorisation is tested against (oracle/ld_linalg.py) ----------
def _mp_cholesky(S):
    """Textbook Cholesky in mpmath (40 digits) with LAPACK's info."""
    n = len(S)
    A = [[mp.mpf(float(S[i][j])) for j in range(n)] for i in range(n)]
    L = [[mp.mpf(0)] * n for _ in range(n)]
    for j in range(n):
        d = A[j][j] - mp.fsum(L[j][k] ** 2 for k in range(j))
        if not d > 0:
            return L, j + 1
        L[j][j] = mp.sqrt(d)
        for i in range(j + 1, n):
            L[i][j] = (A[i][j] - mp.fsum(L[i][k] * L[j][k] for k in range(j))) / L[j][j]
    return L, 0


def _mp_ld(M):
    """mpmath matrix -> longdouble array, through decimal strings (no fp64 rounding on the way)."""
    from oracle import ld_linalg as ld
    return np.array([[ld.LD(mp.nstr(M[i, j], 30)) for j in range(M.cols)] for i in range(M.rows)])


@pytest.mark.parametrize("n", [1, 2, 7, 24])
def test_ld_linalg_matches_mpmath(n):
    """Cholesky, triangular inverse, W^T W, log-determinant, solves and the residual helpers of oracle/ld_linalg.py
    against a 40-digit mpmath evaluation, on an ill-conditioned (cond 1e10) and a graded matrix (rows 2^+-40).  Each
    longdouble result must be at least 100x closer to the 40-digit value than the fp64 LAPACK / numpy result of the same
    quantity (or within 1e-17 of its scale): what makes it a reference for fp64 kernels."""
    from scipy.linalg import lapack, solve_triangular
    from oracle import ld_linalg as ld

    assert ld.EPS_LD < 1e-18, "np.longdouble is not the 80-bit extended format on this host"
    rng = np.random.default_rng(n)
    Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    lam = np.logspace(0, -10, n)
    d = 2.0 ** rng.integers(-40, 40, n)
    for S in ((Q * lam) @ Q.T, d[:, None] * (np.eye(n) + 0.1 * np.ones((n, n))) * d[None, :]):
        S = 0.5 * (S + S.T)
        with mp.workdps(40):
            Lm, info_m = _mp_cholesky(S)
            assert info_m == 0
            Wm = mp.matrix(Lm) ** -1
            b = rng.standard_normal(n)
            bm = mp.matrix([mp.mpf(float(v)) for v in b])
            refs = {"L": _mp_ld(mp.matrix(Lm)), "W": _mp_ld(Wm), "Sinv": _mp_ld(Wm.T * Wm), "x": _mp_ld(Wm * bm),
                    "xt": _mp_ld(Wm.T * bm)}
            logdet_ref = ld.LD(mp.nstr(2 * mp.fsum(mp.log(Lm[i][i]) for i in range(n)), 30))

        L, info = ld.cholesky(S, nb=5)   # a block size that does not divide n: every branch of the blocking
        assert info == 0
        W = ld.tri_inv(L, nb=5)
        c, _ = lapack.dpotrf(S, lower=1, clean=1)
        Wf, _ = lapack.dtrtri(c, lower=1)
        Sf, _ = lapack.dpotri(c, lower=1)
        Sf = np.tril(Sf) + np.tril(Sf, -1).T
        got = {"L": L, "W": W, "Sinv": ld.wtw(W, nb=5), "x": ld.tri_solve(L, b)[:, None],
               "xt": ld.tri_solve(L, b, trans=True)[:, None]}
        fp64 = {"L": c, "W": Wf, "Sinv": Sf, "x": solve_triangular(c, b, lower=True)[:, None],
                "xt": solve_triangular(c, b, lower=True, trans=1)[:, None]}
        for k, ref in refs.items():
            rs = np.abs(ref).max(axis=1, keepdims=True)   # per row: graded rows differ by 2^80
            rs[rs == 0] = 1
            e_ld = float(np.max(np.abs(got[k] - ref) / rs))
            e_64 = float(np.max(np.abs(fp64[k].astype(ld.LD) - ref) / rs))
            assert e_ld <= max(1e-17, 1e-2 * e_64), (k, e_ld, e_64)
        e_64 = abs(ld.LD(2 * np.sum(np.log(np.diag(c)))) - logdet_ref)
        assert abs(ld.logdet(L) - logdet_ref) <= max(1e-17 * abs(float(logdet_ref)), 1e-2 * e_64)
        # residual helpers: the longdouble factor rounded to fp64 has residuals at the fp64 level
        Lf = np.tril(np.asarray(L, dtype=np.float64))
        assert ld.componentwise_backward_error(Lf, S, rows=5) < (n + 1) * 2.0 ** -53
        assert ld.normwise_backward_error(Lf, S, rows=5) < (n + 1) * 2.0 ** -53
        v = rng.standard_normal((n, 2))
        assert ld.chol_probe_residual(Lf, S, v, rows=5) < (n + 1) * 2.0 ** -53
    if n > 1:
        # exact residuals: L = I against S = I + E e_n e_n^T
        E = 2.0 ** -30
        Se = np.eye(n)
        Se[-1, -1] += E
        assert ld.componentwise_backward_error(np.eye(n), Se) == E
        assert ld.normwise_backward_error(np.eye(n), Se) == E / (1 + E)
        v = np.zeros((n, 1))
        v[-1] = 1.0
        assert ld.chol_probe_residual(np.eye(n), Se, v) == E / (1 + E)
        assert ld.sinv_probe_residual(np.eye(n), Se, v) == E
    # LAPACK's info: 1-based failing pivot (against mpmath), rows before it final
    for p in range(n):
        A = rng.standard_normal((n, n))
        S = A @ A.T + n * np.eye(n)
        Lc, info = ld.cholesky(S, nb=5)
        S[p, p] -= 1.5 * float(Lc[p, p]) ** 2
        with mp.workdps(40):
            info_m = _mp_cholesky(S)[1]
        L, info = ld.cholesky(S, nb=5)
        assert info == info_m == p + 1
        assert np.array_equal(L[:p], Lc[:p])
    Sn = np.eye(n)
    Sn[n - 1, 0] = np.nan
    assert ld.cholesky(Sn)[1] == n
