"""Batched fits with measurement variances: the heteroscedastic objective Sigma = K + diag(v) + (jitter + sigma^2) I in
the duplicate-row-compressed batched kernels (include/lfm_b200.h, lfm_batched_nlml_grad_unc_het / lfm_batched_fit_het).

CPU: a numpy restatement of the compressed formulas against the dense oracle.  GPU: every batched kernel (one warp per
LFM, teams of four and eight warps, one CTA per LFM) against the oracle, per-LFM variances, the queue mode, the
multi-start driver, the host-buffer entry point and the executed GPyTorch twin."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from oracle import lfm_oracle as o

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RTOL = 1e-9


def relerr(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def het_problem(G, T, R, seed):
    """synthetic_problem with its variances scaled by U(0.5, 20), so that the variance term matters."""
    x, y, var, _ = o.synthetic_problem(G, T, R, seed=seed)
    return x, y, var * np.random.default_rng(seed + 1).uniform(0.5, 20.0, var.shape)


def non_uniform_design(seed):
    """Two replicates with four measurements of the second one missing: N = 36 rows that the kernels do not
    compress (non-uniform multiplicities)."""
    x, y, var = het_problem(4, 5, 2, seed)
    keep = np.ones(x.shape[0], dtype=bool)
    keep[[27, 33, 36, 39]] = False
    return np.ascontiguousarray(x[keep]), np.ascontiguousarray(y[keep]), np.ascontiguousarray(var[keep])


def start_points(G, B, seed, scale=0.3):
    th0 = o.Params.reference_init(G).pack()
    TH = o.constrain(o.unconstrain(th0)[None, :] + scale * np.random.default_rng(seed).standard_normal((B, th0.shape[0])))
    TH[0] = th0
    return TH


# ---- CPU: the compressed mathematics ---------------------------------------------------------------------------------
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


def compressed_het(p, x, y, var):
    """NLML, gradient (constrained theta) and the intermediates of the U x U formulation, restating the kernels."""
    G, N = p.num_genes, x.shape[0]
    Pt, R = _compression(x)
    first_row = np.argmax(Pt, axis=1)
    xu = x[first_row]
    z = y - o.mean_function(p, x)
    c = var + p.jitter + p.sigma**2
    om, om2 = Pt @ (1.0 / c), Pt @ (1.0 / c**2)
    cbar = R / om
    q = cbar * (Pt @ (z / c))
    Ku = o.gram(p, xu)
    M = np.diag(cbar) + R * Ku
    Minv = np.linalg.inv(M)
    beta = Minv @ q
    kb = (q - cbar * beta) / R
    logdet = np.sum(np.log(c)) - np.sum(np.log(cbar)) + np.linalg.slogdet(M)[1]
    quad = np.sum(z * z / c) - np.sum(q / cbar * kb)
    val = 0.5 * (N * np.log(2.0 * np.pi) + logdet + quad)
    W = 0.5 * (R * Minv - np.outer(beta, beta))                               # P^T Kbar P
    sens = 0.5 * (1.0 - cbar * np.diag(Minv) - beta * kb)                      # diag(P^T Kbar P K_u)
    alpha = (z - Pt.T @ kb) / c
    trS = np.sum(1.0 / c) - np.sum(om2 / om) + R * np.sum(om2 * np.diag(Minv) / om**2)
    # kernel-parameter terms contracted over the unique pairs, as the oracle contracts over all pairs
    t, gi = xu[:, 0], o._gene_index(xu[:, 1])
    j, k = gi[:, None], gi[None, :]
    H1, dH1_da, dH1_db, dH1_dl = o._h_partials(p, k, j, t[None, :], t[:, None])
    H2, dH2_da, dH2_db, dH2_dl = o._h_partials(p, j, k, t[:, None], t[None, :])
    mult0 = p.l * np.sqrt(np.pi) * 0.5
    w = W * p.s[j] * p.s[k] * mult0
    gd, gs = np.zeros(G), np.zeros(G)
    np.add.at(gd, gi, (w * (dH1_db + dH2_da)).sum(axis=1))
    np.add.at(gd, gi, (w * (dH1_da + dH2_db)).sum(axis=0))
    np.add.at(gs, gi, 2.0 * sens / p.s[gi])
    gl = np.sum(w * (dH1_dl + dH2_dl)) + np.sum(W * Ku) / p.l
    asum = alpha.reshape(G, N // G).sum(axis=1)
    grad = np.concatenate([gd + asum * p.b / p.d**2, gs, -asum / p.d, [gl, p.sigma * (trS - alpha @ alpha)]])
    return val, grad, dict(Pt=Pt, beta=beta, W=W, sens=sens, Ku=Ku, alpha=alpha, trS=trS, M=M, q=q, cbar=cbar, R=R)


@pytest.mark.parametrize("design", ["R1", "R3", "non_uniform", "zero_variances"])
def test_compressed_formulas_match_the_dense_oracle(design):
    if design == "non_uniform":
        x, y, var = non_uniform_design(71)
    else:
        x, y, var = het_problem(5, 7, 3 if design == "R3" else 1, 71)
        if design == "zero_variances":
            var = np.zeros_like(var)
    G = int(x[:, 1].max()) + 1
    p = o.Params.unpack(o.Params.reference_init(G).pack() * np.random.default_rng(72).uniform(0.8, 1.2, 3 * G + 2), 1e-4)
    v_ref, g_ref = o.nlml_and_grad(p, x, y, variances=var)
    val, grad, m = compressed_het(p, x, y, var)
    assert abs(val - v_ref) <= 1e-12 * abs(v_ref)
    assert relerr(grad, g_ref) < 1e-12
    # the intermediates against their dense definitions
    S = o.sigma_matrix(p, x, variances=var)
    Sinv = np.linalg.inv(S)
    alpha = Sinv @ (y - o.mean_function(p, x))
    Kbar = 0.5 * (Sinv - np.outer(alpha, alpha))
    Pt = m["Pt"]
    assert relerr(m["alpha"], alpha) < 1e-12 and relerr(m["beta"], Pt @ alpha) < 1e-12
    assert relerr(m["W"], Pt @ Kbar @ Pt.T) < 1e-12
    assert relerr(m["sens"], np.diag(Pt @ Kbar @ Pt.T @ m["Ku"])) < 1e-12
    assert abs(m["trS"] - np.trace(Sinv)) <= 1e-12 * np.trace(Sinv)


def test_variance_shapes():
    from dis_project_b200 import ops
    B, N = 4, 35
    assert ops._variance_layout((B, N), B, N) is True
    assert ops._variance_layout((N,), B, N) is False
    assert ops._variance_layout((N, 1), B, N) is False
    assert ops._variance_layout((1, N), 1, N) is False
    for bad in ((N - 1,), (B, N - 1), (B + 1, N), (N, 2), (1, N), (B, N, 1)):
        with pytest.raises(ValueError):
            ops._variance_layout(bad, B, N)


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _use(monkeypatch, team):
    """team 1 / 4 / 8: warps per LFM of the time-grid kernels; 0: the CTA-per-LFM kernel (time_grid = 0)."""
    if team:
        monkeypatch.setenv("LFM_BATCHED_TEAM", str(team))
    return 0 if team == 0 else None


TEAMS = [1, 4, 8, 0]


@pytest.mark.gpu
@pytest.mark.parametrize("team", TEAMS)
@pytest.mark.parametrize("G,T,R", [(5, 7, 1), (5, 7, 3), (3, 12, 2), (4, 32, 1)])
def test_batched_het_evaluation_matches_oracle(cuda, G, T, R, team, monkeypatch):
    from dis_project_b200 import ops
    tg = _use(monkeypatch, team)
    x, y, var = het_problem(G, T, R, 81)
    U = o.unconstrain(start_points(G, 5, 82, 0.4))
    val, grad, info = ops.batched_nlml_grad_unc(x, y, U, 1e-4, G, time_grid=tg, variances=var)
    assert not info.cpu().numpy().any()
    val, grad = val.cpu().numpy(), grad.cpu().numpy()
    for b in range(U.shape[0]):
        v, g = o.nlml_and_grad_unc(U[b], x, y, 1e-4, variances=var)
        assert abs(val[b] - v) <= RTOL * abs(v) and relerr(grad[b], g) < RTOL
    v_hom = o.nlml_and_grad_unc(U[0], x, y, 1e-4)[0]
    assert abs(val[0] - v_hom) > 1e-3 * abs(v_hom)                             # the variance term matters


@pytest.mark.gpu
@pytest.mark.parametrize("team", TEAMS)
@pytest.mark.parametrize("R,fix", [(1, True), (3, True), (1, False), (3, False)])
def test_batched_het_fit_matches_oracle(cuda, R, fix, team, monkeypatch):
    """150 Adam steps in chunks of 1, 49 and 100 against the oracle's fit with the same objective."""
    from dis_project_b200 import ops
    tg = _use(monkeypatch, team)
    G, T, B, steps = 5, 7, 3, 150
    x, y, var = het_problem(G, T, R, 91)
    TH = start_points(G, B, 92)
    st = ops.BatchedFitState(TH, G, steps)
    if tg is not None:
        st.time_grid = tg
    for chunk in (1, 49, 100):
        ops.batched_fit_steps(st, x, y, 1e-4, chunk, fix_params=fix, variances=var)
    theta, hist, info = st.theta.cpu().numpy(), st.hist.cpu().numpy(), st.info.cpu().numpy()
    assert not info.any()
    for b in range(B):
        th_ref, h_ref = o.fit(TH[b], x, y, 1e-4, num_iters=steps, fix_params=fix, variances=var)
        assert relerr(hist[b], h_ref) < 1e-8
        assert relerr(theta[b], th_ref) < 1e-7


@pytest.mark.gpu
@pytest.mark.parametrize("team", [1, 4, 0])
def test_batched_het_per_lfm_variances(cuda, team, monkeypatch):
    """One row of observations AND one row of variances per LFM (candidate gene sets with their own measurement errors):
    evaluation and a 30-step fit against the oracle on each LFM's own data; multi_start_fit on host arrays and on device
    tensors equals batched_fit_steps."""
    import torch
    from dis_project_b200 import ops
    from dis_project_b200.batched import multi_start_fit
    tg = _use(monkeypatch, team)
    G, T, R, B = 5, 7, 3, 6
    x = het_problem(G, T, R, 101)[0]
    Y = np.stack([het_problem(G, T, R, 110 + b)[1] for b in range(B)])
    V = np.stack([het_problem(G, T, R, 120 + b)[2] for b in range(B)])
    TH = start_points(G, B, 102)
    U = o.unconstrain(TH)
    val, grad, info = ops.batched_nlml_grad_unc(x, Y, U, 1e-4, G, time_grid=tg, variances=V)
    assert not info.cpu().numpy().any()
    val, grad = val.cpu().numpy(), grad.cpu().numpy()
    for b in range(B):
        v, g = o.nlml_and_grad_unc(U[b], x, Y[b], 1e-4, variances=V[b])
        assert abs(val[b] - v) <= RTOL * abs(v) and relerr(grad[b], g) < RTOL
    st = ops.BatchedFitState(TH, G, 30)
    if tg is not None:
        st.time_grid = tg
    for chunk in (11, 19):
        ops.batched_fit_steps(st, x, Y, 1e-4, chunk, variances=V)
    hist, theta = st.hist.cpu().numpy(), st.theta.cpu().numpy()
    for b in range(B):
        th_ref, h_ref = o.fit(TH[b], x, Y[b], 1e-4, num_iters=30, variances=V[b])
        assert relerr(hist[b], h_ref) < 1e-8 and relerr(theta[b], th_ref) < 1e-8
    if tg is None:
        for inputs in ((x, Y, V), tuple(torch.as_tensor(a, device="cuda") for a in (x, Y, V))):
            res = multi_start_fit(inputs[0], inputs[1], TH, 1e-4, num_iters=30, chunk=10, variances=inputs[2])
            assert relerr(res.history, hist) < 1e-12 and res.best_id == int(np.argmin(hist[:, -1]))
        # shared variances: (N,) and (N, 1) are the same fit
        r1 = multi_start_fit(x, Y, TH, 1e-4, num_iters=30, chunk=None, trace=True, variances=V[2])
        r2 = multi_start_fit(x, Y, TH, 1e-4, num_iters=30, chunk=None, trace=True, variances=V[2].reshape(-1, 1))
        assert np.array_equal(r1.history, r2.history)
        assert relerr(r1.history[4], o.fit(TH[4], x, Y[4], 1e-4, num_iters=30, variances=V[2])[1]) < 1e-8
    with pytest.raises(ValueError):
        ops.batched_nlml_grad_unc(x, Y, U, 1e-4, G, variances=V[:, :-1])


@pytest.mark.gpu
@pytest.mark.parametrize("team,B", [(4, 20), (1, 9)])
def test_batched_het_queue_mode_matches_chunked_launches(cuda, team, B, monkeypatch):
    """The persistent-queue launch with variances (shared and one row per LFM, reloaded per task) equals separate
    launches of the same chunk length, bit for bit."""
    import torch
    from dis_project_b200 import ops
    monkeypatch.setenv("LFM_BATCHED_TEAM", str(team))
    G, T, R = 5, 7, 3
    x, y, var = het_problem(G, T, R, 131)
    rng = np.random.default_rng(132)
    TH = start_points(G, B, 133)
    Y = y[None, :] + 0.05 * rng.standard_normal((B, y.shape[0]))
    V = var[None, :] * rng.uniform(0.5, 2.0, (B, y.shape[0]))
    steps, chunk = 23, 5
    for yy, vv in ((y, var), (Y, V)):
        ref = ops.BatchedFitState(TH, G, steps)
        kref = torch.full((steps,), torch.iinfo(torch.int64).max, dtype=torch.int64, device="cuda")
        for c0 in range(0, steps, chunk):
            ops.batched_fit_steps(ref, x, yy, 1e-4, min(chunk, steps - c0), step_keys=kref, variances=vv)
        monkeypatch.setenv("LFM_BATCHED_QUEUE", "1")
        st = ops.BatchedFitState(TH, G, steps)
        keys = torch.full((steps,), torch.iinfo(torch.int64).max, dtype=torch.int64, device="cuda")
        ops.batched_fit_steps(st, x, yy, 1e-4, steps, step_keys=keys, queue_chunk=chunk, variances=vv)
        monkeypatch.delenv("LFM_BATCHED_QUEUE")
        assert st.queue_ws is not None and st.step == steps
        assert torch.equal(st.hist, ref.hist) and torch.equal(st.theta, ref.theta) and torch.equal(st.u, ref.u)
        assert torch.equal(st.adam, ref.adam) and torch.equal(st.info, ref.info) and torch.equal(keys, kref)
    th_ref, h_ref = o.fit(TH[1], x, Y[1], 1e-4, num_iters=steps, variances=V[1])
    assert relerr(st.hist[1].cpu().numpy(), h_ref) < 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("team", TEAMS)
def test_batched_het_none_and_zero_variances(cuda, team, monkeypatch):
    """variances=None is the existing entry point (identical results); zero variances agree with it to 1e-12."""
    import torch
    from dis_project_b200 import ops
    tg = _use(monkeypatch, team)
    G, T, R = 5, 7, 3
    x, y, var = het_problem(G, T, R, 141)
    TH = start_points(G, 4, 142)
    U = o.unconstrain(TH)
    a = ops.batched_nlml_grad_unc(x, y, U, 1e-4, G, time_grid=tg)
    b = ops.batched_nlml_grad_unc(x, y, U, 1e-4, G, time_grid=tg, variances=None)
    z = ops.batched_nlml_grad_unc(x, y, U, 1e-4, G, time_grid=tg, variances=np.zeros_like(var))
    assert all(torch.equal(p, q) for p, q in zip(a, b))
    assert relerr(z[0].cpu().numpy(), a[0].cpu().numpy()) < 1e-12 and relerr(z[1].cpu().numpy(), a[1].cpu().numpy()) < 1e-12
    fits = []
    for v in (None, np.zeros_like(var)):
        st = ops.BatchedFitState(TH, G, 40)
        if tg is not None:
            st.time_grid = tg
        for chunk in (15, 25):
            ops.batched_fit_steps(st, x, y, 1e-4, chunk, variances=v)
        fits.append(st)
    plain = ops.BatchedFitState(TH, G, 40)
    if tg is not None:
        plain.time_grid = tg
    for chunk in (15, 25):
        ops.batched_fit_steps(plain, x, y, 1e-4, chunk)
    assert torch.equal(fits[0].hist, plain.hist) and torch.equal(fits[0].theta, plain.theta)
    assert relerr(fits[1].hist.cpu().numpy(), plain.hist.cpu().numpy()) < 1e-12
    assert relerr(fits[1].theta.cpu().numpy(), plain.theta.cpu().numpy()) < 1e-11


@pytest.mark.gpu
@pytest.mark.parametrize("team", TEAMS)
def test_batched_het_negative_variances_are_reported(cuda, team, monkeypatch):
    """Variances negative enough to make Sigma indefinite: info > 0 and NaN objective and gradient from every kernel."""
    from dis_project_b200 import ops
    tg = _use(monkeypatch, team)
    G, T, R = 5, 7, 3
    x, y, var = het_problem(G, T, R, 151)
    U = o.unconstrain(start_points(G, 3, 152))
    bad = var.copy()
    bad[::4] = -50.0
    with pytest.raises(np.linalg.LinAlgError):
        o.nlml_and_grad_unc(U[0], x, y, 1e-4, variances=bad)
    val, grad, info = ops.batched_nlml_grad_unc(x, y, U, 1e-4, G, time_grid=tg, variances=bad)
    assert np.all(info.cpu().numpy() > 0)
    assert np.all(np.isnan(val.cpu().numpy())) and np.all(np.isnan(grad.cpu().numpy()))


@pytest.mark.gpu
@pytest.mark.parametrize("team", [1, 4, 0])
def test_batched_het_non_uniform_design(cuda, team, monkeypatch):
    """Non-uniformly duplicated rows are fitted at full size (U = N) with the variances."""
    from dis_project_b200 import ops
    tg = _use(monkeypatch, team)
    x, y, var = non_uniform_design(161)
    G = 4
    assert ops.unique_rows(x) == x.shape[0]
    TH = start_points(G, 2, 162)
    val, grad, info = ops.batched_nlml_grad_unc(x, y, o.unconstrain(TH), 1e-4, G, time_grid=tg, variances=var)
    assert np.all(info.cpu().numpy() == 0)
    for b in range(2):
        v_ref, g_ref = o.nlml_and_grad_unc(o.unconstrain(TH[b]), x, y, 1e-4, variances=var)
        assert abs(val[b].item() - v_ref) <= RTOL * abs(v_ref) and relerr(grad[b].cpu().numpy(), g_ref) < RTOL
    st = ops.BatchedFitState(TH, G, 20)
    if tg is not None:
        st.time_grid = tg
    ops.batched_fit_steps(st, x, y, 1e-4, 20, fix_params=False, variances=var)
    theta, hist, info, _ = ops.batched_to_host(st)
    assert np.all(info == 0)
    for b in range(2):
        th_ref, h_ref = o.fit(TH[b], x, y, 1e-4, num_iters=20, fix_params=False, variances=var)
        assert relerr(hist[b], h_ref) < 1e-9 and relerr(theta[b], th_ref) < 1e-8


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["rep0", "rep2"])
def test_batched_het_matches_the_gpytorch_twin(cuda, name):
    """The executed GPyTorch twin's loss (NLML / N) and gradient, reproduced by the batched evaluation (unconstrained
    leaves; the twin's parameters are float32, hence 1e-5 / 1e-4)."""
    from dis_project_b200 import ops
    with open(os.path.join(GOLD, f"ref_twin_{name}.json")) as fh:
        c = json.load(fh)
    G = c["G"]
    t, y, var = np.array(c["train_t"]), np.array(c["train_y"]), np.array(c["variances"])
    N = t.size
    X = np.stack((t, np.repeat(np.arange(G), N // G).astype(np.float64), np.ones(N)), axis=1)
    sig = lambda r: 1.0 / (1.0 + np.exp(-np.asarray(r, dtype=np.float64)))
    thetas, grads = [], []
    for pt in c["points"]:   # d(NLML)/d(theta) from the twin's d(loss)/d(raw): see tests/test_ref_parity.py
        sigma = float(np.sqrt(pt["noise"]))
        thetas.append(np.concatenate([pt["decay"], pt["sensitivity"], pt["basal"], [pt["lengthscale"], sigma]]))
        sl = sig(pt["raw"]["lengthscale"])
        grads.append(np.concatenate([np.array(pt["grad_raw"]["decay"]) / sig(pt["raw"]["decay"]),
                                     np.array(pt["grad_raw"]["sensitivity"]) / sig(pt["raw"]["sensitivity"]),
                                     np.array(pt["grad_raw"]["basal"]) / sig(pt["raw"]["basal"]),
                                     np.array(pt["grad_raw"]["lengthscale"]) / (3.0 * sl * (1.0 - sl)),
                                     np.array(pt["grad_raw"]["noise"]) / sig(pt["raw"]["noise"]) * 2.0 * sigma]) * N)
    U = np.stack([o.unconstrain(th) for th in thetas])
    val, grad, info = ops.batched_nlml_grad_unc(X, y, U, c["kernel_jitter"], G, variances=var)
    assert not info.cpu().numpy().any()
    val, grad = val.cpu().numpy(), grad.cpu().numpy()
    for b, pt in enumerate(c["points"]):
        assert abs(val[b] / N - pt["loss"]) <= 1e-5 * abs(pt["loss"])
        g_unc = grads[b] * o.constrain_jac(U[b])
        assert np.max(np.abs(grad[b] - g_unc)) <= 1e-4 * np.max(np.abs(g_unc))


@pytest.mark.gpu
def test_batched_fit_het_host_equals_device_path(cuda):
    """lfm_batched_fit_het_host (host buffers, one H2D copy) equals the device entry point, with variances and with NULL
    variances (the homoscedastic fit); a second NULL-variance call on the same handle repeats the fit bit for bit."""
    from dis_project_b200 import _lib, ops
    G, T, R, B, steps = 5, 7, 3, 4, 25
    x, y, var = het_problem(G, T, R, 171)
    TH = start_points(G, B, 172)
    st = ops.BatchedFitState(TH, G, steps)
    ops.batched_fit_steps(st, x, y, 1e-4, steps, variances=var)
    st0 = ops.BatchedFitState(TH, G, steps)
    ops.batched_fit_steps(st0, x, y, 1e-4, steps)
    lib = _lib.lib()
    h = C.c_void_p()
    assert lib.lfm_handle_create(C.byref(h)) == 0
    P = 3 * G + 2
    for v in (var, None):
        th, hist, info = np.empty((B, P)), np.empty((B, steps)), np.empty(B, dtype=np.int32)
        TH_c = np.ascontiguousarray(TH)
        assert lib.lfm_batched_fit_het_host(h, B, x.shape[0], G, x.ctypes.data, y.ctypes.data,
                                            v.ctypes.data if v is not None else None, TH_c.ctypes.data, 1e-4, 0.01, 0.9,
                                            0.999, 1e-8, steps, 1, 1000, th.ctypes.data, hist.ctypes.data,
                                            info.ctypes.data) == 0
        assert not info.any()
        if v is not None:
            assert relerr(hist, st.hist.cpu().numpy()) < 1e-12 and relerr(th, st.theta.cpu().numpy()) < 1e-12
        else:
            assert relerr(hist, st0.hist.cpu().numpy()) < 1e-12 and relerr(th, st0.theta.cpu().numpy()) < 1e-12
            th2, hist2 = np.empty((B, P)), np.empty((B, steps))
            assert lib.lfm_batched_fit_het_host(h, B, x.shape[0], G, x.ctypes.data, y.ctypes.data, None,
                                                TH_c.ctypes.data, 1e-4, 0.01, 0.9, 0.999, 1e-8, steps, 1, 1000,
                                                th2.ctypes.data, hist2.ctypes.data, info.ctypes.data) == 0
            assert np.array_equal(hist, hist2) and np.array_equal(th, th2)
    assert lib.lfm_handle_destroy(h) == 0
