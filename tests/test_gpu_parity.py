"""Parity of the CUDA path (through the C-ABI) against the CPU oracle.  Tolerance: 1e-9 relative
(north_star), stated per assertion; matrix entries are compared to 1e-11 of the matrix scale."""
import numpy as np
import pytest
import torch

from oracle import lfm_oracle as o

pytestmark = pytest.mark.gpu
RTOL = 1e-9


def relerr(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def rand_params(G, seed, jitter=1e-4):
    rng = np.random.default_rng(seed)
    return o.Params(d=rng.uniform(0.2, 1.0, G), s=rng.uniform(0.5, 1.5, G), b=rng.uniform(0.01, 0.1, G),
                    l=float(rng.uniform(0.8, 3.2)), sigma=float(rng.uniform(0.6, 1.4)), jitter=jitter)


CASES = [(5, 7, 1), (5, 7, 3), (3, 6, 1), (6, 50, 1), (16, 40, 1)]


@pytest.mark.parametrize("G,T,R", CASES)
def test_cross_covariance_blocks(cuda, G, T, R):
    from dis_project_b200 import ops
    x, y, var, _ = o.synthetic_problem(G, T, R, seed=1)
    p = rand_params(G, 2)
    xs = o.generate_test_times(37)
    both = np.concatenate([x, xs], axis=0)  # mixed flags: exercises k_xx, k_xf, k_xf^T and k_ff
    ref = o.cross_covariance(p, both, both)
    got = ops.cross_covariance(both, both, p.pack(), G).cpu().numpy()
    assert relerr(got, ref) < 1e-11
    # rectangular, odd sizes (scalar-store path)
    ref2 = o.cross_covariance(p, x[:11], xs[:7])
    got2 = ops.cross_covariance(x[:11], xs[:7], p.pack(), G).cpu().numpy()
    assert relerr(got2, ref2) < 1e-11
    m = ops.mean_function(x, p.pack(), G).cpu().numpy().reshape(-1)
    assert relerr(m, o.mean_function(p, x)) < 1e-15


def test_empty_and_ragged(cuda):
    from dis_project_b200 import ops
    p = rand_params(5, 3)
    x, *_ = o.synthetic_problem(5, 7, 1)
    e = np.zeros((0, 3))
    assert ops.cross_covariance(e, x, p.pack(), 5).shape == (0, 35)
    assert ops.cross_covariance(x, e, p.pack(), 5).shape == (35, 0)
    with pytest.raises(ValueError):
        ops.mean_function(x[:33], p.pack(), 5)
    with pytest.raises(ValueError):
        ops.cross_covariance(x[:, :2], x, p.pack(), 5)
    # out-of-range gene indices follow jnp indexing: -1 wraps, >= G clamps (SURVEY Q6)
    xq = x.copy()
    xq[:7, 1] = -1
    xq[7:14, 1] = 9
    xr = x.copy()
    xr[:7, 1] = 4
    xr[7:14, 1] = 4
    a = ops.gram(xq, p.pack(), 5).cpu().numpy()
    b = ops.gram(xr, p.pack(), 5).cpu().numpy()
    assert np.array_equal(a, b)


@pytest.mark.parametrize("G,T,R", CASES)
def test_nlml_and_grad(cuda, G, T, R):
    from dis_project_b200 import ops
    x, y, var, _ = o.synthetic_problem(G, T, R, seed=4)
    p = rand_params(G, 5)
    val_ref, g_ref = o.nlml_and_grad(p, x, y)
    v, info = ops.nlml(x, y, p.pack(), p.jitter, G)
    assert int(info.item()) == 0
    assert abs(v.item() - val_ref) <= RTOL * abs(val_ref)
    out, info = ops.nlml_grad(x, y, p.pack(), p.jitter, G)
    out = out.cpu().numpy()
    assert int(info.item()) == 0
    assert abs(out[0] - val_ref) <= RTOL * abs(val_ref)
    assert relerr(out[1:], g_ref) < RTOL
    # unconstrained coordinates (what the optimiser sees)
    u = o.unconstrain(p.pack())
    v2, g2 = o.nlml_and_grad_unc(u, x, y, p.jitter)
    out2, _ = ops.nlml_grad_unc(x, y, u, p.jitter, G)
    out2 = out2.cpu().numpy()
    assert abs(out2[0] - v2) <= RTOL * abs(v2)
    assert relerr(out2[1:], g2) < RTOL


def test_nlml_grad_half_sweep_sizes(cuda):
    """N = 2048 (16 blocks of 128) is the smallest problem whose factorisation starts Sigma^-1 = W^T W early (W11^T W11 into
    the dead L11 block half-way through the sweep, diag(L11) copied out first; chol.cu); N = 1920 (15 blocks) and N = 3200
    (25 blocks) take the plain recursion.  Value (log-determinant from the copied diagonal) and gradient (the whole of
    Sigma^-1) against the oracle."""
    from dis_project_b200 import ops
    for G, T in ((16, 128), (15, 128), (25, 128)):
        x, y, var, _ = o.synthetic_problem(G, T, 1, seed=8)
        p = rand_params(G, 9)
        val_ref, g_ref = o.nlml_and_grad(p, x, y)
        out, info = ops.nlml_grad(x, y, p.pack(), p.jitter, G)
        out = out.cpu().numpy()
        assert int(info.item()) == 0
        assert abs(out[0] - val_ref) <= RTOL * abs(val_ref), (G, T)
        assert relerr(out[1:], g_ref) < RTOL, (G, T)
        plan = ops.NlmlGradPlan(torch.as_tensor(x).cuda(), torch.as_tensor(y).cuda(), G, p.jitter)
        out2, info2 = plan(torch.as_tensor(p.pack()).cuda())
        assert np.array_equal(out2.cpu().numpy(), out)   # the captured graph replays the same arithmetic


def test_nlml_grad_vs_autograd(cuda):
    from dis_project_b200 import ops
    x, y, var, _ = o.synthetic_problem(5, 7, 3, seed=6)
    p = o.Params.reference_init(5)
    u = o.unconstrain(p.pack())
    v, g = o.nlml_and_grad_unc_autograd(u, x, y, p.jitter)
    out, _ = ops.nlml_grad_unc(x, y, u, p.jitter, 5)
    out = out.cpu().numpy()
    assert abs(out[0] - v) <= RTOL * abs(v)
    assert relerr(out[1:], g) < RTOL


def test_not_positive_definite_reports_info_and_nan(cuda):
    from dis_project_b200 import ops
    x, y, var, _ = o.synthetic_problem(5, 7, 1)
    p = o.Params.reference_init(5)
    p.sigma = 1e-30
    out, info = ops.nlml_grad(x, y, p.pack(), -1.0, 5)  # negative jitter -> Sigma indefinite
    assert int(info.item()) > 0
    assert np.all(np.isnan(out.cpu().numpy()))


@pytest.mark.parametrize("G,T,R,Ts", [(5, 7, 1, 100), (5, 7, 3, 100), (6, 50, 1, 2400)])
def test_latent_posterior(cuda, G, T, R, Ts):
    from dis_project_b200 import ops
    x, y, var, _ = o.synthetic_problem(G, T, R, seed=7)
    p = rand_params(G, 8)
    xs = o.generate_test_times(Ts)
    m_ref, v_ref = o.latent_predict(p, xs, x, y, var)
    m, v, info = ops.latent_posterior(x, y, var, p.pack(), p.jitter, xs, G)
    assert int(info.item()) == 0
    assert relerr(m.cpu().numpy(), m_ref) < RTOL
    assert relerr(v.cpu().numpy(), v_ref) < RTOL


def test_dense_factor_inverse(cuda):
    from dis_project_b200 import ops
    rng = np.random.default_rng(0)
    for n in (128, 384, 640):
        A = rng.standard_normal((n, n))
        S = A @ A.T + n * np.eye(n)
        L, Sinv, info = ops.debug_potrf_potri(torch.as_tensor(S.copy()).cuda())
        assert int(info.item()) == 0
        Lr = np.linalg.cholesky(S)
        assert relerr(np.tril(L.cpu().numpy()), Lr) < 1e-12
        Si = np.tril(Sinv.cpu().numpy())
        assert relerr(Si, np.tril(np.linalg.inv(S))) < 1e-11
    A = rng.standard_normal((256, 48))
    B = rng.standard_normal((384, 48))
    Cm = ops.debug_dgemm_nt(torch.as_tensor(A).cuda(), torch.as_tensor(B).cuda()).cpu().numpy()
    assert relerr(Cm, A @ B.T) < 1e-14


@pytest.mark.parametrize("n", [512, 1024, 1536, 2048, 4096, 4608, 8192])
def test_dense_driver_paths(cuda, n):
    """Every driver of the blocked factorisation / inverse: look-ahead right-looking sweep with the triangular
    inverse interleaved (power-of-two block counts up to 4096), the same sweep followed by the recursive inverse
    (1536, 4608 blocks are not a power of two), and the recursive factorisation above 4096 -- against cuSOLVER /
    cuBLAS through torch on the same device, and L L^T = S, S^-1 S = I on probe vectors."""
    from dis_project_b200 import ops
    g = torch.Generator(device="cuda")
    g.manual_seed(n)
    A = torch.randn(n, 192, dtype=torch.float64, device="cuda", generator=g)
    S = A @ A.T
    S.diagonal().add_(torch.linspace(1.0, 3.0, n, dtype=torch.float64, device="cuda"))
    Lref = torch.linalg.cholesky(S)
    probe = torch.randn(n, 3, dtype=torch.float64, device="cuda", generator=g)
    Sp = S @ probe
    L, Sinv, info = ops.debug_potrf_potri(S.clone())
    assert int(info.item()) == 0
    Lt = torch.tril(L)
    assert float((Lt - Lref).abs().max() / Lref.abs().max()) < 1e-12
    Si = torch.tril(Sinv) + torch.tril(Sinv, -1).T
    assert float((Si @ Sp - probe).abs().max() / probe.abs().max()) < 1e-10
    L2, none, info2 = ops.debug_potrf_potri(S.clone(), want_inverse=False)   # factorisation alone (value-only path)
    assert none is None and int(info2.item()) == 0
    assert torch.equal(torch.tril(L2), Lt)                                     # same arithmetic with / without the inverse


@pytest.mark.parametrize("G,T,R", [(5, 7, 1), (5, 7, 3), (4, 32, 1)])
def test_batched_eval(cuda, G, T, R):
    from dis_project_b200 import ops
    x, y, var, _ = o.synthetic_problem(G, T, R, seed=9)
    rng = np.random.default_rng(10)
    B = 7
    u0 = o.unconstrain(o.Params.reference_init(G).pack())
    U = u0[None, :] + 0.5 * rng.standard_normal((B, u0.shape[0]))
    val, grad, info = ops.batched_nlml_grad_unc(x, y, U, 1e-4, G)
    val, grad = val.cpu().numpy(), grad.cpu().numpy()
    assert not info.cpu().numpy().any()
    for b in range(B):
        v, g = o.nlml_and_grad_unc(U[b], x, y, 1e-4)
        assert abs(val[b] - v) <= RTOL * abs(v)
        assert relerr(grad[b], g) < RTOL


@pytest.mark.parametrize("team", [1, 4])
@pytest.mark.parametrize("R,fix", [(1, True), (3, True), (1, False), (3, False)])   # (3, False) = notebook.py:36,73-75
def test_batched_fit_matches_trainer(cuda, R, fix, team, monkeypatch):
    """150 Adam steps with the p21 hook (trainer.py:162-228), B restarts, split into chunks; warp-per-LFM kernel
    (register Cholesky) and four-warp team kernel (symmetric sweep)."""
    from dis_project_b200 import ops
    monkeypatch.setenv("LFM_BATCHED_TEAM", str(team))
    G, T = 5, 7
    x, y, var, _ = o.synthetic_problem(G, T, R, seed=11)
    rng = np.random.default_rng(12)
    B, steps = 3, 150
    th0 = o.Params.reference_init(G).pack()
    TH = o.constrain(o.unconstrain(th0)[None, :] + 0.3 * rng.standard_normal((B, th0.shape[0])))
    TH[0] = th0
    st = ops.BatchedFitState(TH, G, steps)
    for chunk in (1, 49, 100):
        ops.batched_fit_steps(st, x, y, 1e-4, chunk, fix_params=fix)
    theta, hist = st.theta.cpu().numpy(), st.hist.cpu().numpy()
    for b in range(B):
        th_ref, h_ref = o.fit(TH[b], x, y, 1e-4, num_iters=steps, fix_params=fix)
        # 150 chained optimiser steps amplify rounding differences; 1e-7 on the trajectory end point
        assert relerr(hist[b], h_ref) < 1e-8
        assert relerr(theta[b], th_ref) < 1e-7


@pytest.mark.parametrize("team", [1, 4, 8])
@pytest.mark.parametrize("G,T,R", [(5, 7, 1), (5, 7, 3), (3, 12, 2), (8, 8, 1), (2, 20, 3), (4, 8, 2), (2, 9, 1), (3, 11, 1), (3, 12, 1), (2, 17, 1)])
def test_batched_warp_kernel_matches_cta_kernel(cuda, G, T, R, team, monkeypatch):
    """Warp- / team-per-LFM kernel (time-grid tables in shared memory; team = warps per LFM) against the
    one-CTA-per-LFM kernel (time_grid=0) and the oracle: evaluation and a 40-step fit, unique rows 16..64
    (both lane mappings of the warp kernel, partial tile rows of the team sweep)."""
    from dis_project_b200 import ops
    monkeypatch.setenv("LFM_BATCHED_TEAM", str(team))
    x, y, var, _ = o.synthetic_problem(G, T, R, seed=41)
    rng = np.random.default_rng(42)
    B = 5
    u0 = o.unconstrain(o.Params.reference_init(G).pack())
    U = u0[None, :] + 0.4 * rng.standard_normal((B, u0.shape[0]))
    v1, g1, i1 = ops.batched_nlml_grad_unc(x, y, U, 1e-4, G)
    v0, g0, i0 = ops.batched_nlml_grad_unc(x, y, U, 1e-4, G, time_grid=0)
    assert not i1.cpu().numpy().any() and not i0.cpu().numpy().any()
    v1, g1, v0, g0 = (t.cpu().numpy() for t in (v1, g1, v0, g0))
    for b in range(B):
        v, g = o.nlml_and_grad_unc(U[b], x, y, 1e-4)
        assert abs(v1[b] - v) <= RTOL * abs(v) and relerr(g1[b], g) < RTOL
        assert abs(v1[b] - v0[b]) <= 1e-11 * abs(v0[b]) and relerr(g1[b], g0[b]) < 1e-10
    TH = o.constrain(U)
    sa = ops.BatchedFitState(TH, G, 40)
    sb = ops.BatchedFitState(TH, G, 40)
    sb.time_grid = 0
    for chunk in (7, 33):
        ops.batched_fit_steps(sa, x, y, 1e-4, chunk)
        ops.batched_fit_steps(sb, x, y, 1e-4, chunk)
    assert relerr(sa.hist.cpu().numpy(), sb.hist.cpu().numpy()) < 1e-9
    assert relerr(sa.theta.cpu().numpy(), sb.theta.cpu().numpy()) < 1e-8
    # a time-grid bound that is too small is refused, not silently wrong (warp kernel: unique rows <= 36)
    if G * T <= 36:
        vv, gg, ii = ops.batched_nlml_grad_unc(x, y, U, 1e-4, G, time_grid=T - 1)
        assert np.all(ii.cpu().numpy() == -2) and np.all(np.isnan(vv.cpu().numpy()))


@pytest.mark.parametrize("team", [1, 4, 8])
def test_batched_not_positive_definite_is_reported(cuda, team, monkeypatch):
    """A negative jitter that makes Sigma indefinite: info > 0 and NaN objective from every team size, and the
    team size chosen from the batch size (no override) agrees with the forced ones on a healthy problem."""
    from dis_project_b200 import ops
    monkeypatch.setenv("LFM_BATCHED_TEAM", str(team))
    G, T = 5, 7
    x, y, var, _ = o.synthetic_problem(G, T, 1, seed=5)
    u0 = o.unconstrain(o.Params.reference_init(G).pack())
    U = np.tile(u0, (3, 1))
    val, grad, info = ops.batched_nlml_grad_unc(x, y, U, -5.0, G)
    assert np.all(info.cpu().numpy() > 0) and np.all(np.isnan(val.cpu().numpy()))
    v1, g1, i1 = ops.batched_nlml_grad_unc(x, y, U, 1e-4, G)
    monkeypatch.delenv("LFM_BATCHED_TEAM")
    v0, g0, i0 = ops.batched_nlml_grad_unc(x, y, U, 1e-4, G)
    assert not i1.cpu().numpy().any() and not i0.cpu().numpy().any()
    assert relerr(v1.cpu().numpy(), v0.cpu().numpy()) < 1e-12 and relerr(g1.cpu().numpy(), g0.cpu().numpy()) < 1e-10


@pytest.mark.parametrize("team,time_grid", [(1, None), (4, None), (1, 0)])
def test_batched_per_lfm_observations(cuda, team, time_grid, monkeypatch):
    """One row of observations per LFM on a shared design X (north_star: replicas / candidate TFs): evaluation and
    a 30-step fit of every LFM against the oracle on its own data -- warp kernel, team kernel, CTA kernel."""
    from dis_project_b200 import ops
    from dis_project_b200.batched import multi_start_fit
    monkeypatch.setenv("LFM_BATCHED_TEAM", str(team))
    G, T, R, B = 5, 7, 3, 6
    x, y0, var, _ = o.synthetic_problem(G, T, R, seed=21)
    rng = np.random.default_rng(22)
    Y = np.stack([o.synthetic_problem(G, T, R, seed=30 + b)[1].reshape(-1) for b in range(B)])
    u0 = o.unconstrain(o.Params.reference_init(G).pack())
    U = u0[None, :] + 0.3 * rng.standard_normal((B, u0.shape[0]))
    val, grad, info = ops.batched_nlml_grad_unc(x, Y, U, 1e-4, G, time_grid=time_grid)
    val, grad = val.cpu().numpy(), grad.cpu().numpy()
    assert not info.cpu().numpy().any()
    for b in range(B):
        v, g = o.nlml_and_grad_unc(U[b], x, Y[b], 1e-4)
        assert abs(val[b] - v) <= RTOL * abs(v) and relerr(grad[b], g) < RTOL
    TH = o.constrain(U)
    st = ops.BatchedFitState(TH, G, 30)
    if time_grid is not None:
        st.time_grid = time_grid
    for chunk in (11, 19):
        ops.batched_fit_steps(st, x, Y, 1e-4, chunk)
    hist, theta = st.hist.cpu().numpy(), st.theta.cpu().numpy()
    for b in range(B):
        th_ref, h_ref = o.fit(TH[b], x, Y[b], 1e-4, num_iters=30)
        assert relerr(hist[b], h_ref) < 1e-9 and relerr(theta[b], th_ref) < 1e-8
    if time_grid is None:
        res = multi_start_fit(x, Y, TH, 1e-4, num_iters=30, chunk=10)
        assert relerr(res.history, hist) < 1e-12 and res.best_id == int(np.argmin(hist[:, -1]))
    with pytest.raises(ValueError):
        ops.batched_nlml_grad_unc(x, Y[:, :-1], U, 1e-4, G)


@pytest.mark.parametrize("team", [0, 1, 4])
def test_batched_non_uniform_duplicate_rows(cuda, team, monkeypatch):
    """ADVICE r1: a design with NON-uniformly duplicated rows (three replicates, one measurement missing) is not
    compressed; the batched kernels must fit it at full size instead of refusing (info = -1, NaN)."""
    from dis_project_b200 import ops
    if team:
        monkeypatch.setenv("LFM_BATCHED_TEAM", str(team))
    G, T = 4, 5
    x, y, var, _ = o.synthetic_problem(G, T, 2, seed=21)          # N = 40, every row twice
    keep = np.ones(x.shape[0], dtype=bool); keep[[27, 33, 36, 39]] = False   # drop 4 rows of the second replicate
    x, y = np.ascontiguousarray(x[keep]), np.ascontiguousarray(y[keep])      # N = 36, divisible by G
    assert ops.unique_rows(x) == 36
    th0 = o.Params.reference_init(G).pack()
    TH = np.stack([th0, th0 * 1.1])
    val, grad, info = ops.batched_nlml_grad_unc(x, y, o.unconstrain(TH), 1e-4, G, time_grid=0 if team == 0 else None)
    assert np.all(info.cpu().numpy() == 0)
    for b in range(2):
        v_ref, g_ref = o.nlml_and_grad_unc(o.unconstrain(TH[b]), x, y, 1e-4)
        assert abs(val[b].item() - v_ref) <= RTOL * abs(v_ref) and relerr(grad[b].cpu().numpy(), g_ref) < RTOL
    st = ops.BatchedFitState(TH, G, 20)
    if team == 0:
        st.time_grid = 0
    ops.batched_fit_steps(st, x, y, 1e-4, 20, fix_params=False)
    theta, hist, info, _ = ops.batched_to_host(st)
    assert np.all(info == 0)
    for b in range(2):
        th_ref, h_ref = o.fit(TH[b], x, y, 1e-4, num_iters=20, fix_params=False)
        assert relerr(hist[b], h_ref) < 1e-9 and relerr(theta[b], th_ref) < 1e-8


@pytest.mark.parametrize("G,T,R", [(5, 7, 1), (5, 7, 3), (6, 50, 1)])
def test_heteroscedastic_objective(cuda, G, T, R):
    """Sigma = K + diag(variances) + jitter I + sigma^2 I (src/gpytorch_alfi/model_alfi.py:294-299) on the device:
    value, constrained and unconstrained gradient against the oracle's closed form AND against torch autograd of the
    literal expressions; eager, time-grid and direct paths, the evaluation plan and the host-buffer entry point."""
    import ctypes as C
    from dis_project_b200 import _lib, ops
    x, y, var, _ = o.synthetic_problem(G, T, R, seed=31)
    var = var * np.random.default_rng(32).uniform(0.5, 20.0, var.shape)     # make the term matter
    p = rand_params(G, 33)
    v_ref, g_ref = o.nlml_and_grad(p, x, y, variances=var)
    v_hom, _ = o.nlml_and_grad(p, x, y)
    assert abs(v_ref - v_hom) > 1e-3 * abs(v_hom)
    for tg in (None, 0):
        v, info = ops.nlml(x, y, p.pack(), p.jitter, G, time_grid=tg, variances=var)
        assert int(info.item()) == 0 and abs(v.item() - v_ref) <= RTOL * abs(v_ref)
        out, info = ops.nlml_grad(x, y, p.pack(), p.jitter, G, time_grid=tg, variances=var)
        out = out.cpu().numpy()
        assert abs(out[0] - v_ref) <= RTOL * abs(v_ref) and relerr(out[1:], g_ref) < RTOL
    u = o.unconstrain(p.pack())
    vu_ref, gu_ref = o.nlml_and_grad_unc(u, x, y, p.jitter, variances=var)
    va, ga = o.nlml_and_grad_unc_autograd(u, x, y, p.jitter, variances=var)
    out, info = ops.nlml_grad_unc(x, y, u, p.jitter, G, variances=var)
    out = out.cpu().numpy()
    assert abs(out[0] - vu_ref) <= RTOL * abs(vu_ref) and relerr(out[1:], gu_ref) < RTOL
    assert abs(out[0] - va) <= RTOL * abs(va) and relerr(out[1:], ga) < RTOL
    plan = ops.NlmlGradPlan(x, y, G, p.jitter, unconstrained=True, variances=var)
    pout, pinfo = plan(u)
    assert np.array_equal(pout.cpu().numpy(), out)                              # replay == eager, bit for bit
    plan.close()
    lib = _lib.lib()
    h = C.c_void_p()
    assert lib.lfm_handle_create(C.byref(h)) == 0
    hout = np.empty(3 * G + 3); hinfo = C.c_int(-1)
    th = p.pack()
    for _ in range(2):   # second call reuses the cached plan and the cached structure of X
        assert lib.lfm_nlml_grad_het_host(h, x.shape[0], G, x.ctypes.data, y.ctypes.data, var.ctypes.data, th.ctypes.data,
                                          p.jitter, 0, hout.ctypes.data, C.byref(hinfo)) == 0
        assert hinfo.value == 0 and abs(hout[0] - v_ref) <= RTOL * abs(v_ref) and relerr(hout[1:], g_ref) < RTOL
    assert lib.lfm_nlml_grad_het_host(h, x.shape[0], G, x.ctypes.data, y.ctypes.data, None, th.ctypes.data, p.jitter, 0,
                                      hout.ctypes.data, C.byref(hinfo)) == 0
    assert abs(hout[0] - v_hom) <= RTOL * abs(v_hom)                           # NULL variances == the plain objective
    xbad = x.copy(); xbad[1, 2] = 0.0
    assert lib.lfm_nlml_grad_host(h, x.shape[0], G, xbad.ctypes.data, y.ctypes.data, th.ctypes.data, p.jitter, 0,
                                  hout.ctypes.data, C.byref(hinfo)) == -3        # flag-0 training row: refused
    assert lib.lfm_handle_destroy(h) == 0


def test_heteroscedastic_trainer_and_plan_cache(cuda):
    """CustomConjMLL(variances=...) through JaxTrainer (host loop: the batched kernels have no variance term) against
    the oracle's fit with the same objective; and the plan cache follows the CONTENTS of the data set (ADVICE r1)."""
    from dis_project_b200.gpx_compat import Dataset, adam
    from dis_project_b200.model import ExactLFM
    from dis_project_b200.objectives import CustomConjMLL
    from dis_project_b200.trainer import JaxTrainer
    x, y, var, _ = o.synthetic_problem(5, 7, 1, seed=41)
    var = var * 10.0
    model = ExactLFM(jitter=1e-4, num_genes=5)
    loss = CustomConjMLL(negative=True, variances=var)
    tr = JaxTrainer(model=model, objective=loss, training_data=Dataset(x, y.reshape(-1, 1)), optim=adam(0.01), key=None,
                    num_iters=25)
    trained, hist = tr.fit(fix_params=True)
    th_ref, h_ref = o.fit(model.pack(), x, y, 1e-4, num_iters=25, fix_params=True, variances=var)
    assert relerr(hist, h_ref) < 1e-9 and relerr(trained.pack(), th_ref) < 1e-8
    # plan cache: same objective object, a second Dataset with other observations, then an in-place edit
    plain = CustomConjMLL(negative=True)
    u = model.unconstrain()
    d1 = Dataset(x, y.reshape(-1, 1))
    v1, _ = plain.value_and_grad(u, d1)
    y2 = y * 1.5
    d2 = Dataset(x, y2.reshape(-1, 1))
    v2, _ = plain.value_and_grad(u, d2)
    assert abs(v1 - o.nlml_and_grad_unc(o.unconstrain(model.pack()), x, y, 1e-4)[0]) <= RTOL * abs(v1)
    assert abs(v2 - o.nlml_and_grad_unc(o.unconstrain(model.pack()), x, y2, 1e-4)[0]) <= RTOL * abs(v2)
    d2.y[...] = y.reshape(-1, 1)            # in-place edit of the cached data set
    v3, _ = plain.value_and_grad(u, d2)
    assert abs(v3 - v1) <= 1e-12 * abs(v1)


def test_bijector_kernels(cuda):
    """lfm_constrain / lfm_unconstrain (tfp Softplus and Sigmoid(0.5, 3.5), model.py:66-111) against the oracle, B
    vectors at once, including the tails where softplus is the identity to rounding."""
    from dis_project_b200 import ops
    G = 5
    rng = np.random.default_rng(51)
    U = rng.normal(0.0, 3.0, (7, 3 * G + 2))
    U[0] = 0.0; U[1] = -30.0; U[2] = 30.0; U[2, 3 * G] = 12.0; U[1, 3 * G] = -12.0
    th = ops.constrain(U, G).cpu().numpy()
    ref = np.stack([o.constrain(u) for u in U])
    assert relerr(th, ref) < 1e-14
    assert np.all(th[:, 3 * G] >= 0.5) and np.all(th[:, 3 * G] <= 3.5)
    back = ops.unconstrain(ref[3:], G).cpu().numpy()
    assert relerr(back, np.stack([o.unconstrain(t) for t in ref[3:]])) < 1e-13
    assert relerr(back, U[3:]) < 1e-9


@pytest.mark.parametrize("team,B", [(4, 20), (1, 9), (4, 333)])
def test_batched_queue_mode_matches_chunked_launches(cuda, team, B, monkeypatch):
    """lfm_batched_fit_het with a queue workspace: persistent workers + device-side task queue (an LFM changes SM after every chunk).  Forced
    on here (LFM_BATCHED_QUEUE=1; the library otherwise only uses it where the static assignment is unbalanced): the fit
    must equal the same fit run as separate launches of the same chunk length, bit for bit -- same arithmetic, only the
    placement differs -- including per-LFM observations and the per-step best-objective keys."""
    from dis_project_b200 import ops
    monkeypatch.setenv("LFM_BATCHED_TEAM", str(team))
    G, T, R = 5, 7, 3
    x, y, var, _ = o.synthetic_problem(G, T, R, seed=61)
    rng = np.random.default_rng(62)
    th0 = o.Params.reference_init(G).pack()
    TH = o.constrain(o.unconstrain(th0)[None, :] + 0.3 * rng.standard_normal((B, th0.shape[0])))
    Y = y[None, :] + 0.05 * rng.standard_normal((B, y.shape[0]))
    steps, chunk = 23, 5
    for yy in (y, Y):
        ref = ops.BatchedFitState(TH, G, steps)
        kref = torch.full((steps,), torch.iinfo(torch.int64).max, dtype=torch.int64, device="cuda")
        for c0 in range(0, steps, chunk):
            ops.batched_fit_steps(ref, x, yy, 1e-4, min(chunk, steps - c0), step_keys=kref)
        monkeypatch.setenv("LFM_BATCHED_QUEUE", "1")
        st = ops.BatchedFitState(TH, G, steps)
        keys = torch.full((steps,), torch.iinfo(torch.int64).max, dtype=torch.int64, device="cuda")
        ops.batched_fit_steps(st, x, yy, 1e-4, steps, step_keys=keys, queue_chunk=chunk)
        monkeypatch.delenv("LFM_BATCHED_QUEUE")
        assert st.queue_ws is not None and st.step == steps
        assert torch.equal(st.hist, ref.hist) and torch.equal(st.theta, ref.theta) and torch.equal(st.u, ref.u)
        assert torch.equal(st.adam, ref.adam) and torch.equal(st.info, ref.info) and torch.equal(keys, kref)
    th_ref, h_ref = o.fit(TH[1], x, Y[1], 1e-4, num_iters=steps)
    assert relerr(st.hist[1].cpu().numpy(), h_ref) < 1e-9
