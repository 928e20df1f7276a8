"""CPU oracle: fp64 numpy/scipy restatement of the reference LFM hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``dis_project_b200/`` may import this
module; only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs use it, and only as the checker
(or as the timed CPU arm), never as the product path.

PARITY PINNED TO REFERENCE SOURCE EXECUTED HERE.  The reference (wejpurvis/DIS_project) ships no
tests, no golden vectors and no fixtures for this path, and its stack (jax 0.4.28, gpjax 0.8.2,
cola-ml 0.0.5, optax 0.1.9, tfp 0.22.1 -- environment.yml:48-119) is not installable in this
container.  Its own source files are nevertheless executable: ``tests/refshim`` provides torch-fp64
stand-ins for those packages, under which the UNMODIFIED ``src/{dataset,model,objectives,trainer,
utils}.py`` run end to end (CSV loader, kernels, objective, jax.value_and_grad, the 150-step
trainer.fit, both posteriors).  ``tests/golden/make_ref_golden.py`` writes what they return to
``tests/golden/ref_*.json``; ``tests/test_ref_parity.py`` asserts this oracle against those files
(NLML 1e-12, gradients 1e-10, covariance entries 1e-11, posteriors 1e-9, fit history 1e-9; with
``LITERAL_ERF_SUMS`` the covariance entries agree to 1e-14), and the CUDA path against the same
files.  What remains restated rather than executed is the third-party arithmetic listed below.
Independent anchors kept from round 1 (tests/test_oracle.py):
  * an arbitrary-precision (mpmath, 50 digits) evaluation of single kernel entries and of the
    whole path (NLML, gradient, latent posterior) written from the formulas in src/model.py:197-365,
  * a second restatement of the GPyTorch twin's block formulas
    (src/gpytorch_alfi/model_alfi.py:302-382,414-476),
  * torch-fp64 autograd of the same expressions versus the closed-form
    gradient (two independent derivations),
  * the hard-coded reference constants (initial state model.py:100-114,
    Barenco profile dataset.py:111-113, kinetics dataset.py:201-203).

Third-party semantics restated from the pinned versions' published behaviour:
  * tfp ``Softplus`` / ``Sigmoid(low, high)`` bijectors (model.py:66,79,86,93,111)
  * gpjax ``Module.constrain/unconstrain`` = bijector forward/inverse per leaf
  * gpjax ``GaussianDistribution.log_prob`` = dense Cholesky form
    -1/2 [ n log 2pi + log det S + z^T S^-1 z ]      (objectives.py:76-78)
  * optax ``adam(lr)`` defaults b1=.9 b2=.999 eps=1e-8 eps_root=0, bias
    corrected, update = -lr * mhat / (sqrt(vhat) + eps)   (main.py:45)
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field, replace

import numpy as np
from scipy.special import erf, erfc
from scipy.linalg import cho_solve, cholesky, solve_triangular
from scipy.linalg.lapack import dpotrf, dpotri

from . import ld_linalg

SQRT_PI = math.sqrt(math.pi)
L_LOW, L_HIGH = 0.5, 3.5  # model.py:111


# --------------------------------------------------------------------------- #
# parameters + bijectors
# --------------------------------------------------------------------------- #
@dataclass
class Params:
    """Constrained hyper-parameters (model.py:64-121)."""

    d: np.ndarray  # true_d  (G,)
    s: np.ndarray  # true_s  (G,)
    b: np.ndarray  # true_b  (G,)
    l: float  # lengthscale, in [0.5, 3.5]
    sigma: float  # obs_stddev
    jitter: float = 1e-6  # static (model.py:64); main.py:41 uses 1e-4

    @property
    def num_genes(self) -> int:
        return int(np.asarray(self.d).shape[0])

    @staticmethod
    def reference_init(num_genes: int = 5, jitter: float = 1e-4) -> "Params":
        """model.py:99-108 (d=.4, s=1, b=.05), :114 (l=2.5), :65 (sigma=1)."""
        return Params(
            d=np.full(num_genes, 0.4),
            s=np.full(num_genes, 1.0),
            b=np.full(num_genes, 0.05),
            l=2.5,
            sigma=1.0,
            jitter=jitter,
        )

    def pack(self) -> np.ndarray:
        """theta layout used by the C-ABI: [d(G), s(G), b(G), l, sigma]."""
        return np.concatenate([self.d, self.s, self.b, [self.l, self.sigma]]).astype(np.float64)

    @staticmethod
    def unpack(theta: np.ndarray, jitter: float) -> "Params":
        theta = np.asarray(theta, dtype=np.float64)
        G = (theta.shape[0] - 2) // 3
        return Params(theta[:G].copy(), theta[G : 2 * G].copy(), theta[2 * G : 3 * G].copy(),
                      float(theta[3 * G]), float(theta[3 * G + 1]), jitter)


def softplus(x):
    x = np.asarray(x, dtype=np.float64)
    return np.logaddexp(0.0, x)


def softplus_inv(y):
    y = np.asarray(y, dtype=np.float64)
    return y + np.log(-np.expm1(-y))


def sigmoid(x):
    x = np.asarray(x, dtype=np.float64)
    return 0.5 * (1.0 + np.tanh(0.5 * x))


def l_forward(x):
    return L_LOW + (L_HIGH - L_LOW) * sigmoid(x)


def l_inverse(y):
    u = (np.asarray(y, dtype=np.float64) - L_LOW) / (L_HIGH - L_LOW)
    return np.log(u) - np.log1p(-u)


def unconstrain(theta: np.ndarray) -> np.ndarray:
    """Module.unconstrain (trainer.py:75): softplus^-1 on d,s,b,sigma; logit on l."""
    theta = np.asarray(theta, dtype=np.float64)
    G = (theta.shape[-1] - 2) // 3
    out = softplus_inv(theta)
    out[..., 3 * G] = l_inverse(theta[..., 3 * G])
    return out


def constrain(theta_unc: np.ndarray) -> np.ndarray:
    """Module.constrain (trainer.py:103,218)."""
    theta_unc = np.asarray(theta_unc, dtype=np.float64)
    G = (theta_unc.shape[-1] - 2) // 3
    out = softplus(theta_unc)
    out[..., 3 * G] = l_forward(theta_unc[..., 3 * G])
    return out


def constrain_jac(theta_unc: np.ndarray) -> np.ndarray:
    """d constrained / d unconstrained (diagonal)."""
    theta_unc = np.asarray(theta_unc, dtype=np.float64)
    G = (theta_unc.shape[-1] - 2) // 3
    sg = sigmoid(theta_unc)
    out = sg.copy()  # softplus' = sigmoid
    out[..., 3 * G] = (L_HIGH - L_LOW) * sg[..., 3 * G] * (1.0 - sg[..., 3 * G])
    return out


# --------------------------------------------------------------------------- #
# kernels (model.py:152-369) -- broadcasting numpy versions
# --------------------------------------------------------------------------- #
LITERAL_ERF_SUMS = False  # True: evaluate erf(a)+erf(b) exactly as written in the reference


def erfsum(a, b):
    """erf(a) + erf(b).

    The reference writes both erf sums of h, and the one of k_xf, literally (model.py:276-278,
    349-351, 355-357).  The first, R1 = erf(dt/l - gamma) + erf(t1/l + gamma), multiplies exp(-D dt)
    with dt << 0 where erf(a) ~ -1 and erf(b) ~ +1 cancel: the literal form carries ~1e-16 * e^(D |dt|)
    absolute rounding noise (SURVEY Q7; ~2e-11 on O(1) entries in the p53 regime, which a posterior
    mean amplifies to ~1e-9 relative).  The second, R2 = erf(t2/l - gamma) + erf(gamma), cancels for
    t2/l < gamma and is multiplied by exp(gamma^2): ~1e-16 * exp(gamma^2) absolute noise, harmless in
    the p53 regime (gamma <= 1.6) but 5e-11 of the covariance scale at gamma = 4.4 and 4e-2 at
    gamma = 7, which a fit's restarts reach (D is unbounded).  The checker evaluates both with the
    mathematically identical, cancellation-free erfc(-n) - erfc(p) for opposite-sign arguments beyond
    0.5.  `LITERAL_ERF_SUMS = True` restores the reference's literal arithmetic for both sums;
    tests/test_oracle.py bounds the difference between the two in the p53 regime and
    tests/test_sim_regimes.py checks the cancellation-free form against mpmath beyond it.
    """
    a, b = np.broadcast_arrays(np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64))
    lit = erf(a) + erf(b)
    if LITERAL_ERF_SUMS:
        return lit
    opp = (a * b < 0.0) & (np.minimum(np.abs(a), np.abs(b)) > 0.5)
    acc = erfc(-np.minimum(a, b)) - erfc(np.maximum(a, b))
    return np.where(opp, acc, lit)


def gamma(p: Params, k):
    """model.py:367-369."""
    return p.d[k] * p.l / 2.0


def h(p: Params, j, k, t1, t2):
    """model.py:315-365.  j,k integer arrays; t1,t2 float arrays (broadcast)."""
    t_dist = t2 - t1
    g = gamma(p, k)
    multiplier = np.exp(g**2) / (p.d[j] + p.d[k])
    first_multiplier = np.exp(-p.d[k] * t_dist)
    first_erf_terms = erfsum(t_dist / p.l - g, t1 / p.l + g)
    second_multiplier = np.exp(-(p.d[k] * t2 + p.d[j] * t1))
    second_erf_terms = erfsum(t2 / p.l - g, g)
    return multiplier * (first_multiplier * first_erf_terms - second_multiplier * second_erf_terms)


def kernel_xx(p: Params, t, j, tp, k):
    """model.py:197-235 (gene j at t versus gene k at t')."""
    mult = p.s[j] * p.s[k] * p.l * SQRT_PI * 0.5
    return mult * (h(p, k, j, tp, t) + h(p, j, k, t, tp))


def kernel_xf(p: Params, t_gene, j, t_latent):
    """model.py:237-282 after the flag-based argument resolution (:262-263)."""
    t_dist = t_gene - t_latent
    g = gamma(p, j)
    return (0.5 * p.l * SQRT_PI * p.s[j]) * np.exp(g**2) * np.exp(-p.d[j] * t_dist) * erfsum(
        t_dist / p.l - g, t_latent / p.l + g)


def kernel_ff(p: Params, t, tp):
    """model.py:284-312.  NB divides by 2*l, not 2*l^2 (SURVEY Q1)."""
    return np.exp(-np.square(t - tp) / (2.0 * p.l))


_CLAMP_G = None  # set by cross_covariance: jnp clamps out-of-range indices (SURVEY Q6)


def _gene_index(col, G=None):
    # .astype(int) on the float gene column (model.py:223-224); jnp indexing: negatives wrap, then clamp
    g = np.asarray(col, dtype=np.float64).astype(np.int64)
    if G is not None:
        g = np.where(g < 0, g + G, g)
        g = np.clip(g, 0, G - 1)
    return g


def cross_covariance(p: Params, x: np.ndarray, y: np.ndarray) -> np.ndarray:
    """model.py:372-394 with model.kernel (:152-195): all four branches are
    evaluated for every pair and blended by the 0/1 flag switches."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    t = x[:, 0][:, None]
    tp = y[:, 0][None, :]
    j = _gene_index(x[:, 1], p.num_genes)[:, None]
    k = _gene_index(y[:, 1], p.num_genes)[None, :]
    f1 = x[:, 2].astype(np.int64)[:, None]
    f2 = y[:, 2].astype(np.int64)[None, :]
    kxx_sw = f1 * f2
    kff_sw = (1 - f1) * (1 - f2)
    kxf_sw = f1 * (1 - f2)
    kxf_t_sw = (1 - f1) * f2
    with np.errstate(over="ignore", invalid="ignore"):
        kxx = kernel_xx(p, t, j, tp, k)
        kff = kernel_ff(p, t, tp)
        # kernel_xf(t, t'): gene = (t if t.flag != 0 else t')  (model.py:262-263)
        # branch 3: kernel_xf(t, t_prime)
        a_is_latent = f1 == 0
        gene_t = np.where(a_is_latent, tp, t)
        gene_j = np.where(a_is_latent, k, j)
        lat_t = np.where(a_is_latent, t, tp)
        kxf = kernel_xf(p, gene_t, gene_j, lat_t)
        # branch 4: kernel_xf(t_prime, t): "t" is now the column point
        b_is_latent = f2 == 0
        gene_t2 = np.where(b_is_latent, t, tp)
        gene_j2 = np.where(b_is_latent, j, k)
        lat_t2 = np.where(b_is_latent, tp, t)
        kxf_t = kernel_xf(p, gene_t2, gene_j2, lat_t2)
        return kxx_sw * kxx + kff_sw * kff + kxf_sw * kxf + kxf_t_sw * kxf_t


def gram(p: Params, x: np.ndarray) -> np.ndarray:
    """model.py:396-414."""
    return cross_covariance(p, x, x)


def gram_xx_fast(p: Params, x: np.ndarray) -> np.ndarray:
    """k_xx only (all flags 1): what `gram` reduces to on training rows."""
    t = x[:, 0]
    j = _gene_index(x[:, 1])
    return kernel_xx(p, t[:, None], j[:, None], t[None, :], j[None, :])


def mean_function(p: Params, x: np.ndarray) -> np.ndarray:
    """model.py:124-149: positional blocks of N // G rows, times the flag (Q3)."""
    x = np.asarray(x, dtype=np.float64)
    f = x[:, 2].astype(np.int64)
    G = p.num_genes
    block = x.shape[0] // G
    mean = np.repeat(p.b / p.d, block)
    if mean.shape[0] != x.shape[0]:
        raise ValueError(
            f"mean_function: {x.shape[0]} rows is not divisible by num_genes={G} (model.py:145-149)")
    return mean * f


# --------------------------------------------------------------------------- #
# objective (objectives.py:64-78) and its gradient
# --------------------------------------------------------------------------- #
def sigma_matrix(p: Params, x: np.ndarray, variances=None) -> np.ndarray:
    """K + jitter I + sigma^2 I (objectives.py:70-73).  `variances` (N,) adds diag(variances): the heteroscedastic
    convention of the GPyTorch twin, which puts the measurement variances inside the kernel when it trains
    (src/gpytorch_alfi/model_alfi.py:294-299); None = the GPJax objective."""
    K = gram(p, x)
    n = K.shape[0]
    K[np.diag_indices(n)] += p.jitter
    K[np.diag_indices(n)] += p.sigma**2
    if variances is not None:
        K[np.diag_indices(n)] += np.asarray(variances, dtype=np.float64).reshape(-1)
    return K


def nlml(p: Params, x: np.ndarray, y: np.ndarray, variances=None) -> float:
    """CustomConjMLL(negative=True) (objectives.py:21-78)."""
    y = np.asarray(y, dtype=np.float64).reshape(-1)
    S = sigma_matrix(p, x, variances)
    z = y - mean_function(p, x)
    L = cholesky(S, lower=True)
    a = solve_triangular(L, z, lower=True)
    n = z.shape[0]
    return 0.5 * (n * math.log(2.0 * math.pi) + 2.0 * np.sum(np.log(np.diag(L))) + a @ a)


def _h_partials(p: Params, a, b, u, v):
    """H(a,b,u,v)=h(j=a,k=b,t1=u,t2=v) with dH/dd_a, dH/dd_b, dH/dl (SURVEY 7.3)."""
    l = p.l
    da, db = p.d[a], p.d[b]
    g = db * l / 2.0
    delta = v - u
    inv = 1.0 / (da + db)
    E0 = np.exp(g * g) * inv
    A1 = np.exp(-db * delta)
    x1, x2, x3 = delta / l - g, u / l + g, v / l - g
    R1 = erfsum(x1, x2)
    A2 = np.exp(-(db * v + da * u))
    R2 = erfsum(x3, g)
    c = 2.0 / SQRT_PI
    g1, g2, g3, g4 = c * np.exp(-x1 * x1), c * np.exp(-x2 * x2), c * np.exp(-x3 * x3), c * np.exp(-g * g)
    H = E0 * (A1 * R1 - A2 * R2)
    dH_da = -H * inv + E0 * u * A2 * R2
    dH_db = H * (g * l - inv) + E0 * (
        -delta * A1 * R1 + A1 * (l / 2.0) * (-g1 + g2) + v * A2 * R2 - A2 * (l / 2.0) * (-g3 + g4))
    dH_dl = H * g * db + E0 * (
        A1 * (g1 * (-delta / l**2 - db / 2.0) + g2 * (-u / l**2 + db / 2.0))
        - A2 * (g3 * (-v / l**2 - db / 2.0) + g4 * db / 2.0))
    return H, dH_da, dH_db, dH_dl


def nlml_and_grad(p: Params, x: np.ndarray, y: np.ndarray, *, chunk: int = 256, threads: int | None = None,
                  variances=None, linalg: str = "fp64"):
    """Closed-form NLML and gradient w.r.t. the CONSTRAINED theta=[d,s,b,l,sigma].

    K_bar = 1/2 (S^-1 - a a^T); dNLML/dtheta = sum_ij K_bar_ij dK_ij/dtheta (+ mean terms).
    Training rows only (all flags 1).  Row-chunked (so N=32768 fits in RAM) and the chunks are
    spread over `threads` host threads (numpy ufuncs and LAPACK release the GIL).
    linalg="ld": the Cholesky, the solve, the log-determinant and S^-1 run in extended precision
    (oracle.ld_linalg, n <= ~1024) and are rounded to fp64 before the same contraction -- the reference
    where cond(S) makes LAPACK's fp64 answer itself inaccurate.
    """
    import os
    from concurrent.futures import ThreadPoolExecutor

    threads = threads or os.cpu_count() or 1
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64).reshape(-1)
    if not np.all(x[:, 2] == 1):
        raise ValueError("nlml_and_grad expects training rows (flag 1)")
    n = x.shape[0]
    G = p.num_genes
    t = x[:, 0]
    gi = _gene_index(x[:, 1])
    S = np.empty((n, n))
    bounds = [(r0, min(n, r0 + chunk)) for r0 in range(0, n, chunk)]

    def build(b):
        r0, r1 = b
        S[r0:r1] = kernel_xx(p, t[r0:r1, None], gi[r0:r1, None], t[None, :], gi[None, :])

    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(build, bounds))
        S[np.diag_indices(n)] += p.jitter
        S[np.diag_indices(n)] += p.sigma**2
        if variances is not None:   # heteroscedastic convention (see sigma_matrix): constant in theta, the gradient
            S[np.diag_indices(n)] += np.asarray(variances, dtype=np.float64).reshape(-1)   # formulas are unchanged
        mu = mean_function(p, x)
        z = y - mu
        if linalg == "ld":
            Lx, info = ld_linalg.cholesky(S)
            if info != 0:
                raise np.linalg.LinAlgError(f"Sigma not positive definite at pivot {info}")
            logdet = float(ld_linalg.logdet(Lx))
            Wx = ld_linalg.tri_inv(Lx)
            alpha = (Wx.T @ (Wx @ z.astype(ld_linalg.LD))).astype(np.float64)
            Sinv = ld_linalg.wtw(Wx).astype(np.float64)
            del Lx, Wx
        elif linalg == "fp64":
            c, info = dpotrf(S, lower=1, overwrite_a=1, clean=0)
            if info != 0:
                raise np.linalg.LinAlgError(f"Sigma not positive definite at pivot {info}")
            logdet = 2.0 * np.sum(np.log(np.diag(c)))
            alpha = cho_solve((c, True), z)
            Sinv, info = dpotri(c, lower=1, overwrite_c=1)  # valid in the lower triangle
        else:
            raise ValueError(f"linalg must be 'fp64' or 'ld', got {linalg!r}")
        val = 0.5 * (n * math.log(2.0 * math.pi) + logdet + z @ alpha)
        mult0 = p.l * SQRT_PI * 0.5

        def contract(b):
            r0, r1 = b
            rows = slice(r0, r1)
            Kb = Sinv[rows, :].copy()  # symmetric completion of this row block
            Kb[:, r1:] = Sinv[r1:, rows].T
            blk = Sinv[rows, rows]
            Kb[:, rows] = np.tril(blk) + np.tril(blk, -1).T
            tr = np.trace(Kb[:, rows])
            Kb = 0.5 * (Kb - np.outer(alpha[rows], alpha))
            j = gi[rows, None]
            k = gi[None, :]
            tt = t[rows, None]
            tp = t[None, :]
            # k_xx = S_j S_k mult0 [ H(k,j,t',t) + H(j,k,t,t') ]
            H1, dH1_da, dH1_db, dH1_dl = _h_partials(p, k, j, tp, tt)  # a=k (col gene), b=j (row gene)
            H2, dH2_da, dH2_db, dH2_dl = _h_partials(p, j, k, tt, tp)  # a=j (row gene), b=k (col gene)
            ss = p.s[j] * p.s[k]
            kxx = ss * mult0 * (H1 + H2)
            w = Kb * ss * mult0
            gd = np.zeros(G)
            gs = np.zeros(G)
            np.add.at(gd, gi[rows], (w * (dH1_db + dH2_da)).sum(axis=1))  # through the ROW gene's decay
            np.add.at(gd, gi, (w * (dH1_da + dH2_db)).sum(axis=0))        # through the COLUMN gene's decay
            kk = Kb * kxx
            np.add.at(gs, gi[rows], kk.sum(axis=1) / p.s[gi[rows]])
            np.add.at(gs, gi, kk.sum(axis=0) / p.s[gi])
            gl = np.sum(w * (dH1_dl + dH2_dl)) + np.sum(kk) / p.l
            return gd, gs, gl, tr

        parts = list(ex.map(contract, bounds))
    gd = np.sum([q[0] for q in parts], axis=0)
    gs = np.sum([q[1] for q in parts], axis=0)
    gl = float(np.sum([q[2] for q in parts]))
    trK = float(np.sum([q[3] for q in parts]))
    trKbar = 0.5 * (trK - alpha @ alpha)
    gsig = 2.0 * p.sigma * trKbar
    # mean terms: d/dB_m = -sum_{i in block m} alpha_i / D_m ; d/dD_m += sum alpha_i B_m / D_m^2
    block = n // G
    asum = alpha.reshape(G, block).sum(axis=1)
    gb = -asum / p.d
    gd = gd + asum * p.b / p.d**2
    grad = np.concatenate([gd, gs, gb, [gl, gsig]])
    return float(val), grad


def nlml_and_grad_unc(theta_unc: np.ndarray, x, y, jitter: float, variances=None):
    """value_and_grad of JaxTrainer.loss w.r.t. the UNCONSTRAINED leaves (trainer.py:86-131)."""
    theta = constrain(theta_unc)
    val, g = nlml_and_grad(Params.unpack(theta, jitter), x, y, variances=variances)
    return val, g * constrain_jac(theta_unc)


# --------------------------------------------------------------------------- #
# torch-fp64 autograd of the same expressions (independent gradient derivation)
# --------------------------------------------------------------------------- #
def nlml_and_grad_unc_autograd(theta_unc: np.ndarray, x, y, jitter: float, variances=None):
    import torch

    x = np.asarray(x, dtype=np.float64)
    yv = torch.as_tensor(np.asarray(y, dtype=np.float64).reshape(-1))
    n = x.shape[0]
    G = (len(theta_unc) - 2) // 3
    th = torch.tensor(np.asarray(theta_unc, dtype=np.float64), requires_grad=True)
    sp = torch.nn.functional.softplus
    d, s, b = sp(th[:G]), sp(th[G:2 * G]), sp(th[2 * G:3 * G])
    l = L_LOW + (L_HIGH - L_LOW) * torch.sigmoid(th[3 * G])
    sigma = sp(th[3 * G + 1])
    t = torch.as_tensor(x[:, 0])
    gi = torch.as_tensor(_gene_index(x[:, 1]))
    flag = torch.as_tensor(x[:, 2])
    terf, terfc = torch.special.erf, torch.special.erfc

    def tsum(a, b):   # erfsum in torch (both branches have finite derivatives, so torch.where is safe)
        a, b = torch.broadcast_tensors(a, b)
        lit = terf(a) + terf(b)
        if LITERAL_ERF_SUMS:
            return lit
        opp = (a * b < 0.0) & (torch.minimum(a.abs(), b.abs()) > 0.5)
        return torch.where(opp, terfc(-torch.minimum(a, b)) - terfc(torch.maximum(a, b)), lit)

    def hh(j, k, t1, t2):
        td = t2 - t1
        g = d[k] * l / 2
        return torch.exp(g**2) / (d[j] + d[k]) * (
            torch.exp(-d[k] * td) * tsum(td / l - g, t1 / l + g)
            - torch.exp(-(d[k] * t2 + d[j] * t1)) * tsum(t2 / l - g, g))

    j, k = gi[:, None], gi[None, :]
    tt, tp = t[:, None], t[None, :]
    K = s[j] * s[k] * l * SQRT_PI * 0.5 * (hh(k, j, tp, tt) + hh(j, k, tt, tp))
    S = K + (jitter + sigma**2) * torch.eye(n, dtype=torch.float64)
    if variances is not None:
        S = S + torch.diag(torch.as_tensor(np.asarray(variances, dtype=np.float64).reshape(-1)))
    mu = torch.repeat_interleave(b / d, n // G) * flag
    z = yv - mu
    Lc = torch.linalg.cholesky(S)
    a = torch.linalg.solve_triangular(Lc, z[:, None], upper=False)[:, 0]
    val = 0.5 * (n * math.log(2 * math.pi) + 2 * torch.log(torch.diagonal(Lc)).sum() + a @ a)
    val.backward()
    return float(val.detach()), th.grad.numpy().copy()


# --------------------------------------------------------------------------- #
# latent posterior (model.py:420-463)
# --------------------------------------------------------------------------- #
def latent_predict(p: Params, test_inputs: np.ndarray, x: np.ndarray, y: np.ndarray,
                   variances: np.ndarray):
    """Returns (mean (T*,), var_diag (T*,)).  Noise model Q2, double jitter Q4."""
    x = np.asarray(x, dtype=np.float64)
    t = np.asarray(test_inputs, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64).reshape(-1)
    variances = np.asarray(variances, dtype=np.float64).reshape(-1)
    mean_x = mean_function(p, x)
    mean_t = mean_function(p, t)
    Kxx = gram(p, x)
    Kxx[np.diag_indices_from(Kxx)] += variances
    Kxx[np.diag_indices_from(Kxx)] += p.jitter
    Kxf = cross_covariance(p, x, t)
    L = cholesky(Kxx, lower=True)
    alpha = cho_solve((L, True), y - mean_x)
    mean = mean_t + Kxf.T @ alpha
    V = solve_triangular(L, Kxf, lower=True)
    # diag(gram(t)) (model.py:456): kernel_ff(t,t)=1 on latent rows; general rows via the blend
    if np.all(t[:, 2] == 0):
        kdiag = np.ones(t.shape[0])
    else:
        kdiag = np.array([float(cross_covariance(p, t[i:i + 1], t[i:i + 1])[0, 0]) for i in range(t.shape[0])])
    var = kdiag + p.jitter - np.sum(V * V, axis=0) + p.jitter
    return mean, var


def multi_gene_predict(p: Params, test_inputs: np.ndarray, x: np.ndarray, y: np.ndarray, variances: np.ndarray):
    """model.py:465-514: returns (mean (T*,), cov (T*,T*)).  Noise model K + diag(var) + sigma^2 I (Q2)."""
    x = np.asarray(x, dtype=np.float64)
    t = np.asarray(test_inputs, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64).reshape(-1)
    variances = np.asarray(variances, dtype=np.float64).reshape(-1)
    mean_x = mean_function(p, x)
    Sigma = gram(p, x)
    Sigma[np.diag_indices_from(Sigma)] += variances
    Sigma[np.diag_indices_from(Sigma)] += p.sigma**2
    mean_t = mean_function(p, t)
    Ktt = gram(p, t)
    Kxt = cross_covariance(p, x, t)
    L = cholesky(Sigma, lower=True)
    Sinv_Kxt = cho_solve((L, True), Kxt)
    mean = mean_t + Sinv_Kxt.T @ (y - mean_x)
    cov = Ktt - Kxt.T @ Sinv_Kxt
    cov[np.diag_indices_from(cov)] += p.jitter
    return mean, cov


def generate_test_times_pred(t: int = 100, num_genes: int = 5) -> np.ndarray:
    """utils.py:290-314 / :81-99: gene indices 1..G (one past the end; jnp clamps, SURVEY Q6), flag 1."""
    times = np.tile(np.linspace(0, 13, t), num_genes)
    genes = np.repeat(np.arange(1, num_genes + 1), t).astype(np.float64)
    return np.stack((times, genes, np.ones(times.shape[0])), axis=1)


def generate_test_times(t: int = 100) -> np.ndarray:
    """utils.py:268-287."""
    times = np.linspace(0, 13, t)
    return np.stack((times, np.repeat(-1.0, t), np.repeat(0.0, t)), axis=-1)


# --------------------------------------------------------------------------- #
# trainer (trainer.py:36-228) with optax.adam restated
# --------------------------------------------------------------------------- #
def fit(theta0: np.ndarray, x, y, jitter: float, *, num_iters: int = 150, lr: float = 0.01,
        fix_params: bool = True, num_steps_per_epoch: int = 1000, b1: float = 0.9,
        b2: float = 0.999, eps: float = 1e-8, grad_fn=None, variances=None):
    """JaxTrainer(...).fit (trainer.py:162-228).  theta0 is CONSTRAINED; returns
    (final constrained theta, loss history (num_iters,))."""
    grad_fn = grad_fn or nlml_and_grad_unc
    G = (len(theta0) - 2) // 3
    u = unconstrain(np.asarray(theta0, dtype=np.float64))  # trainer.py:75
    m = np.zeros_like(u)
    v = np.zeros_like(u)
    hist = np.empty(num_iters)
    for step in range(num_iters):
        val, g = grad_fn(u, x, y, jitter) if variances is None else grad_fn(u, x, y, jitter, variances=variances)
        hist[step] = val
        m = b1 * m + (1 - b1) * g
        v = b2 * v + (1 - b2) * g * g
        mhat = m / (1 - b1 ** (step + 1))
        vhat = v / (1 - b2 ** (step + 1))
        u = u - lr * mhat / (np.sqrt(vhat) + eps)
        # trainer.py:205-210: hook fires when step % num_steps_per_epoch == 0, in UNCONSTRAINED space (Q5)
        if fix_params and step % num_steps_per_epoch == 0 and G > 3:
            u[G + 3] = 1.0  # true_s[3]
            u[3] = 0.8  # true_d[3]
    theta = constrain(u)  # trainer.py:218
    if fix_params and G > 3:  # trainer.py:219-220, constrained space
        theta[G + 3] = 1.0
        theta[3] = 0.8
    return theta, hist


# --------------------------------------------------------------------------- #
# synthetic inputs (SURVEY 8d) -- reference layout dataset.py:358-399
# --------------------------------------------------------------------------- #
def make_inputs(G: int, T: int, R: int = 1, t_max: float = 12.0) -> np.ndarray:
    times = np.linspace(0.0, t_max, T)
    tcol = np.tile(times, G * R)
    gcol = np.tile(np.repeat(np.arange(G), T), R)
    return np.stack((tcol, gcol.astype(np.float64), np.ones(G * T * R)), axis=-1)


def synthetic_problem(G: int, T: int, R: int = 1, seed: int = 42, jitter: float = 1e-4):
    """X (N,3), y (N,), measurement variances (N,), theta_true; y drawn from the model prior."""
    rng = np.random.default_rng(seed)
    x = make_inputs(G, T, R)
    p_true = Params(d=rng.uniform(0.2, 1.0, G), s=rng.uniform(0.5, 1.5, G), b=rng.uniform(0.01, 0.1, G),
                    l=2.5, sigma=1.0, jitter=jitter)
    n = x.shape[0]
    zz = rng.standard_normal(n)
    variances = rng.uniform(0.01, 0.1, n)
    if n <= 8192:
        S = gram_xx_fast(p_true, x)
        S[np.diag_indices(n)] += jitter + p_true.sigma**2
        y = mean_function(p_true, x) + cholesky(S, lower=True) @ zz
    else:
        # large N: y = mu + K^(1/2)-free surrogate (low-rank latent draw + noise), same moments' scale
        tl = np.linspace(0.0, 12.0, 512)
        xl = np.stack((tl, -np.ones_like(tl), np.zeros_like(tl)), axis=-1)
        Kff = cross_covariance(p_true, xl, xl) + 1e-8 * np.eye(512)
        Kxf = cross_covariance(p_true, x, xl)
        f = cholesky(Kff, lower=True) @ rng.standard_normal(512)
        y = mean_function(p_true, x) + Kxf @ np.linalg.solve(Kff, f) + p_true.sigma * zz
    return x, y, variances, p_true
