"""The assembled dense path -- NLML, gradient, latent and gene posteriors -- against the oracle at the sizes where its
structure changes, through the public ops entry points.

    G x T     N     Np    what changes there
    8 x 125   1000  1024  smallest two-launch Sigma build (columns [0, 256) first; the second launch writes 24 identity
                          rows); 16 row tiles of 64 in the gradient contraction
    9 x 128   1152  1152  9 blocks of 128: the sweep, then the recursive inverse; no padding; posterior row chunks of
                          PR_ROWS = 1024: a full one and one of 128 rows
    25 x 80   2000  2048  two-launch Sigma with the early S11' of the sweep, 48 padded rows
    33 x 128  4224  4224  smallest recursive factorisation (33 blocks)
    64 x 128  8192  8192  last size whose gradient work items span 2 column tiles (ntile = 128)
    43 x 192  8256  8320  first size with 16-tile work items: ntile = 129, 9 chunks, the last one of a single tile;
                          64 padded rows
    43 x 210  9030  9088  ntile = 142: the last tile has 6 rows, the last chunk 14 tiles

The gradient is compared component by component on the scale of that component's own terms:
|g_k - r_k| <= RTOL |r_k| + FLOOR M_k, with M_k = sum |K_bar_ij dK_ij/dtheta_k| (+ the mean and sigma terms) from
oracle.nlml_and_grad(magnitudes=True).  A bound normalised by the largest component lets the smallest one (2e-4 of the
largest at N = 9030) be wrong by several parts in a million.

Decays are drawn from [0.3, 1] so that Sigma stays well conditioned (the ill-conditioned case is the strict xfail of
test_dense_factor.py).  Every oracle result is computed once per module; GPU memory stays below 2 GB."""
import numpy as np
import pytest
import torch

from oracle import lfm_oracle as o

pytestmark = pytest.mark.gpu

JITTER = 1e-4
RTOL = 1e-9          # north_star, per component and for the NLML value
# |g_k - r_k| / M_k measured on a B200 (1000 W): <= 3.0e-13 over every size, path and objective here (N = 8192, unconstrained);
# 1.1e-13 .. 1.5e-13 from N = 4224 up, 2e-14 .. 5e-14 below.  The factor 10 leaves room for a reordered sum.
FLOOR = 3e-12
# Posterior entries on the scale of the prior (see _post_check), measured on a B200: latent mean <= 5.5e-12 (N = 8256),
# latent variance <= 3.3e-14, gene mean / covariance / variance <= 8.6e-13 (N = 1152, T* = 513).  A 1e-9 bound would let
# the latent variance lose one training row per row chunk after the first (3e-10 at N = 1152).
POST_TOL = 5e-11
SIZES = {1000: (8, 125), 1152: (9, 128), 2000: (25, 80), 4224: (33, 128), 8192: (64, 128), 8256: (43, 192),
         9030: (43, 210)}
HET_SIZES = [1000, 2000, 8256]
LATENT_SIZES = [1000, 1152, 8256]
LATENT_TS = [1, 2048, 2049, 4224]      # PC_COLS = 2048 test points per chunk
GENE_CASES = [(1152, 135), (1152, 513), (8256, 129)]


def _report(N, what, err):
    print(f"DENSE N={N:5d} {what:44s} {err:.2e}")


class _Refs:
    """Problems and oracle results, each computed on first use."""

    def __init__(self):
        self._c = {}

    def _get(self, key, fn):
        if key not in self._c:
            self._c[key] = fn()
        return self._c[key]

    def problem(self, N):
        """(G, T, x, y, variances, p, u): theta = constrain(u) exactly, so that the constrained and the unconstrained
        entry points evaluate the same point and one oracle run serves both."""
        def make():
            G, T = SIZES[N]
            x, y, var, _ = o.synthetic_problem(G, T, 1, seed=N)
            rng = np.random.default_rng(N + 1)
            p = o.Params(d=rng.uniform(0.3, 1.0, G), s=rng.uniform(0.5, 1.5, G), b=rng.uniform(0.01, 0.1, G),
                         l=float(rng.uniform(0.8, 3.2)), sigma=float(rng.uniform(0.6, 1.4)), jitter=JITTER)
            u = o.unconstrain(p.pack())
            return G, T, x, y, var, o.Params.unpack(o.constrain(u), JITTER), u
        return self._get(("problem", N), make)

    def grad(self, N, het=False):
        """(value, gradient, M) of the constrained objective; o.nlml_and_grad_unc(u) is by definition this value and
        this gradient times constrain_jac(u)."""
        G, T, x, y, var, p, u = self.problem(N)
        return self._get(("grad", N, het),
                         lambda: o.nlml_and_grad(p, x, y, variances=var if het else None, magnitudes=True))

    def latent(self, N):
        """(test rows, mean, var, prior var) at max(LATENT_TS) latent test points rounded up to a multiple of G (the
        reference's mean_function reshape).  Latent rows have prior mean 0 and the reference's posterior is column by
        column, so a prefix of the rows is the reference of a problem of its own."""
        def make():
            G, T, x, y, var, p, u = self.problem(N)
            ts = np.random.default_rng(N + 2).uniform(-1.0, 13.0, -(-max(LATENT_TS) // G) * G)
            xs = np.stack([ts, -np.ones_like(ts), np.zeros_like(ts)], axis=1)
            m, v = o.latent_predict(p, xs, x, y, var)
            return xs, m, v, _prior_var(p, xs)
        return self._get(("latent", N), make)

    def gene(self, N, Ts):
        def make():
            G, T, x, y, var, p, u = self.problem(N)
            k = Ts // G
            xs = np.stack([np.tile(np.linspace(-0.5, 12.5, k), G), np.repeat(np.arange(G), k).astype(np.float64),
                           np.ones(Ts)], axis=1)
            m, c = o.multi_gene_predict(p, xs, x, y, var)
            return xs, m, c, _prior_var(p, xs)
        return self._get(("gene", N, Ts), make)


@pytest.fixture(scope="module")
def refs():
    return _Refs()


def grad_ratio(got, ref, M):
    """Worst |got_k - ref_k| / (RTOL |ref_k| + FLOOR M_k): <= 1 passes."""
    got = np.asarray(got, dtype=np.float64)
    return float(np.max(np.abs(got - ref) / (RTOL * np.abs(ref) + FLOOR * M)))


def _free():
    from dis_project_b200 import ops
    ops.release_workspaces()
    torch.cuda.empty_cache()


def _check_eval(N, label, out, info, v_ref, g_ref, M):
    out = out.cpu().numpy().copy()
    assert int(info.item()) == 0, (N, label, int(info.item()))
    ev = abs(out[0] - v_ref) / abs(v_ref)
    w = grad_ratio(out[1:], g_ref, M)
    wm = float(np.max(np.abs(out[1:] - g_ref) / M))
    _report(N, f"{label} value", ev)
    _report(N, f"{label} grad: worst err / bound", w)
    _report(N, f"{label} grad: worst err / M", wm)
    assert ev <= RTOL, (N, label, ev)
    assert w <= 1.0, (N, label, w, int(np.argmax(np.abs(out[1:] - g_ref) / (RTOL * np.abs(g_ref) + FLOOR * M))))
    return out


@pytest.mark.parametrize("N", list(SIZES), ids=[f"N{n}" for n in SIZES])
def test_nlml_grad_per_component(cuda, refs, N):
    """nlml_grad and nlml_grad_unc on the time-grid tables and by direct evaluation, per component against the oracle;
    a too-small time-grid bound falls back to direct evaluation with the same bits; ops.nlml (TRSV path) against the
    oracle and against nlml_grad's value; NlmlGradPlan replays the eager bits."""
    from dis_project_b200 import ops
    G, T, x, y, var, p, u = refs.problem(N)
    v_ref, g_ref, M = refs.grad(N)
    jac = o.constrain_jac(u)
    th = p.pack()
    xd, yd = torch.as_tensor(x).cuda(), torch.as_tensor(y).cuda()
    eager = {}
    for tg in (None, 0):
        out, info = ops.nlml_grad(xd, yd, th, JITTER, G, time_grid=tg)
        eager[(False, tg)] = _check_eval(N, f"nlml_grad tg={tg}", out, info, v_ref, g_ref, M)
        out, info = ops.nlml_grad_unc(xd, yd, u, JITTER, G, time_grid=tg)
        eager[(True, tg)] = _check_eval(N, f"nlml_grad_unc tg={tg}", out, info, v_ref, g_ref * jac, M * np.abs(jac))
        v, info = ops.nlml(xd, yd, th, JITTER, G, time_grid=tg)
        v = v.item()
        assert int(info.item()) == 0
        _report(N, f"nlml tg={tg} value", abs(v - v_ref) / abs(v_ref))
        assert abs(v - v_ref) <= RTOL * abs(v_ref), (N, tg)
        assert abs(v - eager[(False, tg)][0]) <= 1e-10 * abs(v), (N, tg)
    # a bound below the T distinct times: the tables do not apply and the direct evaluation runs, bit for bit
    for unc, arg, fn in ((False, th, ops.nlml_grad), (True, u, ops.nlml_grad_unc)):
        out, info = fn(xd, yd, arg, JITTER, G, time_grid=T - 1)
        assert int(info.item()) == 0 and np.array_equal(out.cpu().numpy(), eager[(unc, 0)]), (N, unc)
    _free()
    for unc, arg in ((False, th), (True, u)):
        plan = ops.NlmlGradPlan(xd, yd, G, JITTER, unconstrained=unc)
        for _ in range(2):
            out, info = plan(arg)
            assert int(info.item()) == 0 and np.array_equal(out.cpu().numpy(), eager[(unc, None)]), (N, unc)
        plan.close()
        del plan
        _free()


@pytest.mark.parametrize("N", HET_SIZES, ids=[f"N{n}" for n in HET_SIZES])
def test_heteroscedastic_per_component(cuda, refs, N):
    """Sigma = K + diag(variances) + (jitter + sigma^2) I: the variances reach the second launch of the two-launch Sigma
    build (N = 1000, 2000) and the padded tail (2000, 8256).  Eager (tables and direct) and plan."""
    from dis_project_b200 import ops
    G, T, x, y, var, p, u = refs.problem(N)
    v_ref, g_ref, M = refs.grad(N, het=True)
    v_hom = refs.grad(N)[0]
    assert abs(v_ref - v_hom) > 1e-6 * abs(v_hom)        # the variances are not a no-op at this size
    jac = o.constrain_jac(u)
    th = p.pack()
    xd, yd, vd = (torch.as_tensor(a).cuda() for a in (x, y, var))
    for tg in (None, 0):
        out, info = ops.nlml_grad(xd, yd, th, JITTER, G, time_grid=tg, variances=vd)
        _check_eval(N, f"het nlml_grad tg={tg}", out, info, v_ref, g_ref, M)
        v, info = ops.nlml(xd, yd, th, JITTER, G, time_grid=tg, variances=vd)
        assert int(info.item()) == 0 and abs(v.item() - v_ref) <= RTOL * abs(v_ref), (N, tg)
    out, info = ops.nlml_grad_unc(xd, yd, u, JITTER, G, variances=vd)
    eager = _check_eval(N, "het nlml_grad_unc", out, info, v_ref, g_ref * jac, M * np.abs(jac))
    _free()
    plan = ops.NlmlGradPlan(xd, yd, G, JITTER, unconstrained=True, variances=vd)
    out, info = plan(u)
    out = out.cpu().numpy().copy()
    plan.close()
    del plan
    _free()
    assert int(info.item()) == 0 and np.array_equal(out, eager), N


def _prior_var(p, rows):
    return np.array([o.cross_covariance(p, rows[i:i + 1], rows[i:i + 1])[0, 0] for i in range(rows.shape[0])]) + p.jitter


def _post_check(N, label, p, x, y, got_m, ref_m, got_v, ref_v, pv):
    """Variance on the prior variance of the entry, mean on sqrt(prior variance) max|y - mu|
    (test_sim_regimes.py::test_posteriors_match_oracle)."""
    zs = np.max(np.abs(y - o.mean_function(p, x)))
    em = float(np.max(np.abs(got_m - ref_m) / (np.sqrt(pv) * zs)))
    ev = float(np.max(np.abs(got_v - ref_v) / pv))
    _report(N, f"{label} mean", em)
    _report(N, f"{label} var", ev)
    assert em <= POST_TOL and ev <= POST_TOL, (N, label, em, ev)


@pytest.mark.parametrize("N", LATENT_SIZES, ids=[f"N{n}" for n in LATENT_SIZES])
def test_latent_posterior_chunks(cuda, refs, N):
    """Every T* in LATENT_TS against the oracle, and the test points of every chunk after the first evaluated in a call
    of their own give the same bits: the N = 1152, T* = 2049 call runs a full chunk without the pad memset, then a
    one-column chunk with it."""
    from dis_project_b200 import ops
    G, T, x, y, var, p, u = refs.problem(N)
    xs, m_ref, v_ref, pv = refs.latent(N)
    th = p.pack()
    xd, yd, vd = (torch.as_tensor(a).cuda() for a in (x, y, var))
    for ts in LATENT_TS:
        m, v, info = ops.latent_posterior(xd, yd, vd, th, JITTER, xs[:ts], G)
        assert int(info.item()) == 0
        m, v = m.cpu().numpy(), v.cpu().numpy()
        _post_check(N, f"latent T*={ts}", p, x, y, m, m_ref[:ts], v, v_ref[:ts], pv[:ts])
        for c0 in range(2048, ts, 2048):
            c1 = min(ts, c0 + 2048)
            m1, v1, info = ops.latent_posterior(xd, yd, vd, th, JITTER, xs[c0:c1], G)
            assert int(info.item()) == 0
            assert np.array_equal(m1.cpu().numpy(), m[c0:c1]) and np.array_equal(v1.cpu().numpy(), v[c0:c1]), (N, ts, c0)
    _free()


@pytest.mark.parametrize("N,Ts", GENE_CASES, ids=[f"N{n}-T{t}" for n, t in GENE_CASES])
def test_gene_posterior_sizes(cuda, refs, N, Ts):
    """Mean and covariance against multi_gene_predict with Tp = 256 / 640 padded test columns and 2 or 9 row chunks; the
    covariance is exactly symmetric (mirrored from the lower tiles) and var is its diagonal, bit for bit; full_cov=False
    returns the same mean and its own variance (the kdiag path) within the same bound."""
    from dis_project_b200 import ops
    G, T, x, y, var, p, u = refs.problem(N)
    xs, m_ref, c_ref, pv = refs.gene(N, Ts)
    th = p.pack()
    xd, yd, vd = (torch.as_tensor(a).cuda() for a in (x, y, var))
    m, c, v, info = ops.gene_posterior(xd, yd, vd, th, JITTER, xs, G, full_cov=True)
    assert int(info.item()) == 0
    m, c, v = m.cpu().numpy(), c.cpu().numpy(), v.cpu().numpy()
    assert np.array_equal(c, c.T), (N, Ts, float(np.max(np.abs(c - c.T))))
    assert np.array_equal(v, np.diag(c)), (N, Ts)
    _post_check(N, f"gene T*={Ts} full_cov", p, x, y, m, m_ref, v, np.diag(c_ref), pv)
    ec = float(np.max(np.abs(c - c_ref) / np.sqrt(np.outer(pv, pv))))
    _report(N, f"gene T*={Ts} cov", ec)
    assert ec <= POST_TOL, (N, Ts, ec)
    m2, c2, v2, info = ops.gene_posterior(xd, yd, vd, th, JITTER, xs, G, full_cov=False)
    assert int(info.item()) == 0 and c2 is None
    m2, v2 = m2.cpu().numpy(), v2.cpu().numpy()
    assert np.array_equal(m2, m), (N, Ts)
    _post_check(N, f"gene T*={Ts} diag", p, x, y, m2, m_ref, v2, np.diag(c_ref), pv)
    _free()
