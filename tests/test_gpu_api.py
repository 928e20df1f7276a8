"""Golden vectors, the reference-facing Python surface, the host-buffer C-ABI and full-size
property checks, all on the GPU through liblfm_b200.so."""
import ctypes as C
import glob
import json
import os

import numpy as np
import pytest
import torch

from oracle import lfm_oracle as o

pytestmark = pytest.mark.gpu
RTOL = 1e-9
# oracle-generated vectors (make_golden.py); the reference-executed ref_*.json are consumed by test_ref_parity.py
GOLDEN = sorted(g for g in glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.json"))
                if not os.path.basename(g).startswith("ref_"))


def relerr(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(g) for g in GOLDEN])
def test_golden_vectors(cuda, path):
    from dis_project_b200 import ops
    g = json.load(open(path))
    G, jit = g["G"], g["jitter"]
    th = np.array(g["theta"]); x = np.array(g["X"]); y = np.array(g["y"]); var = np.array(g["variances"])
    rows = np.array(g["K_rows"])
    assert relerr(ops.cross_covariance(rows, rows, th, G).cpu().numpy(), g["K_block"]) < 1e-12
    assert relerr(ops.mean_function(x, th, G).cpu().numpy().reshape(-1), g["mean_function"]) < 1e-15
    out, info = ops.nlml_grad(x, y, th, jit, G)
    out = out.cpu().numpy()
    assert int(info.item()) == 0
    assert abs(out[0] - g["nlml"]) <= RTOL * abs(g["nlml"])
    assert relerr(out[1:], g["grad_constrained"]) < RTOL
    out, _ = ops.nlml_grad_unc(x, y, np.array(g["theta_unc"]), jit, G)
    assert relerr(out.cpu().numpy()[1:], g["grad_unconstrained"]) < RTOL
    m, v, info = ops.latent_posterior(x, y, var, th, jit, np.array(g["Xstar"]), G)
    assert relerr(m.cpu().numpy(), g["posterior_mean"]) < RTOL
    assert relerr(v.cpu().numpy(), g["posterior_var"]) < RTOL
    if "fit_theta" in g:
        st = ops.BatchedFitState(th[None, :], G, 150)
        ops.batched_fit_steps(st, x, y, jit, 150)
        assert relerr(st.hist[0].cpu().numpy(), g["fit_history"]) < 1e-8
        assert relerr(st.theta[0].cpu().numpy(), g["fit_theta"]) < 1e-7


def test_reference_call_sequence_main_py(cuda):
    """The call sequence of the reference's src/main.py:30-66 against the same steps on the oracle."""
    from dis_project_b200.dataset import JaxP53Data, dataset_3d
    from dis_project_b200.gpx_compat import Dataset, adam
    from dis_project_b200.model import ExactLFM
    from dis_project_b200.objectives import CustomConjMLL
    from dis_project_b200.trainer import JaxTrainer
    from dis_project_b200.utils import generate_test_times

    p53_data = JaxP53Data.synthetic(replicate=0)
    training_times, gene_expressions, variances = dataset_3d(p53_data)
    dataset_train = Dataset(training_times, gene_expressions)
    custom_posterior = ExactLFM(jitter=np.array(1e-4), data=p53_data)
    loss = CustomConjMLL(negative=True)
    p0 = o.Params.reference_init(5)
    assert loss(custom_posterior, dataset_train) == pytest.approx(o.nlml(p0, training_times, gene_expressions), rel=RTOL)
    trainer = JaxTrainer(model=custom_posterior, objective=loss, training_data=dataset_train, optim=adam(0.01),
                         key=None, num_iters=150)
    trained_model, history = trainer.fit(num_steps_per_epoch=1000)
    th_ref, h_ref = o.fit(p0.pack(), training_times, gene_expressions, 1e-4, num_iters=150)
    assert relerr(history, h_ref) < 1e-8
    assert relerr(trained_model.pack(), th_ref) < 1e-7
    assert trained_model.true_s[3] == 1.0 and trained_model.true_d[3] == 0.8  # p21 pinned (trainer.py:218-220)
    # generic (per-step) loop gives the same trajectory as the persistent kernel
    tr2 = JaxTrainer(ExactLFM(jitter=1e-4, data=p53_data), loss, dataset_train, adam(0.01), None, 20)
    tr2._device_scan_ok = lambda: False
    m2, h2 = tr2.fit()
    _, h_ref20 = o.fit(p0.pack(), training_times, gene_expressions, 1e-4, num_iters=20)
    assert relerr(h2, h_ref20) < 1e-9
    # latent posterior of the trained model (main.py:66-67)
    testing_times = generate_test_times()
    dist = trained_model.latent_predict(testing_times, p53_data)
    m_ref, v_ref = o.latent_predict(o.Params.unpack(trained_model.pack(), 1e-4), testing_times, training_times,
                                    gene_expressions, variances)
    assert relerr(dist.mean(), m_ref) < RTOL and relerr(dist.stddev(), np.sqrt(v_ref)) < RTOL
    assert dist.mean().shape == (100,)


def test_model_kernel_methods(cuda):
    from dis_project_b200.model import ExactLFM
    rng = np.random.default_rng(0)
    m = ExactLFM(jitter=1e-4, data=False)
    m = m.replace(true_d=rng.uniform(0.2, 1, 5), true_s=rng.uniform(0.5, 1.5, 5), l=np.asarray(1.7))
    p = o.Params.unpack(m.pack(), 1e-4)
    a = np.array([3.0, 2.0, 1.0]); b = np.array([7.5, 4.0, 1.0]); f = np.array([5.0, -1.0, 0.0])
    assert m.kernel(a, b) == pytest.approx(float(o.kernel_xx(p, 3.0, 2, 7.5, 4)), rel=1e-12)
    assert m.kernel_xx(a, b) == pytest.approx(float(o.kernel_xx(p, 3.0, 2, 7.5, 4)), rel=1e-12)
    assert m.kernel(a, f) == pytest.approx(float(o.kernel_xf(p, 3.0, 2, 5.0)), rel=1e-12)
    assert m.kernel_xf(f, a) == pytest.approx(float(o.kernel_xf(p, 3.0, 2, 5.0)), rel=1e-12)
    assert m.kernel_ff(f, np.array([6.0, -1, 0])) == pytest.approx(float(o.kernel_ff(p, 5.0, 6.0)), rel=1e-14)
    assert m.h(1, 3, 2.0, 9.0) == pytest.approx(float(o.h(p, 1, 3, 2.0, 9.0)), rel=1e-12)
    x = o.make_inputs(5, 7)
    K = m.gram(m.kernel, x).to_dense().cpu().numpy()
    assert relerr(K, o.gram(p, x)) < 1e-12
    assert relerr(m.cross_covariance(m.kernel, x, x[:9]).cpu().numpy(), o.cross_covariance(p, x, x[:9])) < 1e-12
    assert relerr(m.mean_function(x).cpu().numpy().reshape(-1), o.mean_function(p, x)) < 1e-15


def test_host_buffer_capi(cuda):
    """lfm_*_host: numpy pointers in, numpy out (what a cgo/ctypes caller binds)."""
    from dis_project_b200 import _lib
    lib = _lib.lib()
    h = C.c_void_p()
    assert lib.lfm_handle_create(C.byref(h)) == 0
    x, y, var, _ = o.synthetic_problem(5, 7, 3, seed=5)
    p = o.Params.reference_init(5)
    th = p.pack()
    out = np.empty(18); info = C.c_int(-1)
    assert lib.lfm_nlml_grad_host(h, 105, 5, x.ctypes.data, y.ctypes.data, th.ctypes.data, 1e-4, 0, out.ctypes.data,
                                  C.byref(info)) == 0
    v, g = o.nlml_and_grad(p, x, y)
    assert info.value == 0 and abs(out[0] - v) <= RTOL * abs(v) and relerr(out[1:], g) < RTOL
    xs = o.generate_test_times(100)
    mean = np.empty(100); pv = np.empty(100)
    assert lib.lfm_latent_posterior_host(h, 105, 5, x.ctypes.data, y.ctypes.data, var.ctypes.data, th.ctypes.data, 1e-4,
                                         100, xs.ctypes.data, mean.ctypes.data, pv.ctypes.data, C.byref(info)) == 0
    m_ref, v_ref = o.latent_predict(p, xs, x, y, var)
    assert relerr(mean, m_ref) < RTOL and relerr(pv, v_ref) < RTOL
    B = 4
    TH = np.ascontiguousarray(np.tile(th, (B, 1))); TH[1:, :5] *= np.array([[1.1], [0.9], [1.3]])
    oth = np.empty((B, 17)); hist = np.empty((B, 30)); infos = (C.c_int * B)()
    assert lib.lfm_batched_fit_het_host(h, B, 105, 5, x.ctypes.data, y.ctypes.data, None, TH.ctypes.data, 1e-4, 0.01,
                                        0.9, 0.999, 1e-8, 30, 1, 1000, oth.ctypes.data, hist.ctypes.data, infos) == 0
    for b in range(B):
        t_ref, h_ref = o.fit(TH[b], x, y, 1e-4, num_iters=30)
        assert relerr(hist[b], h_ref) < 1e-9 and relerr(oth[b], t_ref) < 1e-8
    # error behaviour: invalid arguments are rejected with a status, not a crash
    assert lib.lfm_nlml_grad_host(h, 104, 5, x.ctypes.data, y.ctypes.data, th.ctypes.data, 1e-4, 0, out.ctypes.data,
                                  C.byref(info)) == -1
    assert lib.lfm_batched_fit_het_host(h, 1, 640, 5, x.ctypes.data, y.ctypes.data, None, TH.ctypes.data, 1e-4, 0.01,
                                        0.9, 0.999, 1e-8, 1, 1, 1000, oth.ctypes.data, hist.ctypes.data, infos) == -3
    assert lib.lfm_handle_destroy(h) == 0


def test_multi_start_single_rank(cuda):
    from dis_project_b200.batched import make_restarts, multi_start_fit
    x, y, _, _ = o.synthetic_problem(5, 7, 3, seed=6)
    TH = make_restarts(o.Params.reference_init(5).pack(), 12)
    res = multi_start_fit(x, y, TH, 1e-4, num_iters=40, chunk=7)
    assert res.theta.shape == (12, 17) and res.history.shape == (12, 40) and (res.lo, res.hi) == (0, 12)
    final = np.where(np.isfinite(res.history[:, -1]), res.history[:, -1], np.inf)
    assert res.best_id == int(np.argmin(final)) and res.best_loss == final.min()
    assert np.array_equal(res.best_theta, res.theta[res.best_id])
    t_ref, h_ref = o.fit(TH[5], x, y, 1e-4, num_iters=40)
    assert relerr(res.history[5], h_ref) < 1e-9
    assert np.all(np.diff(res.best_trace) <= 1e-9)  # best objective after each chunk never increases much
    assert res.best_trace[-1] == res.best_loss      # the atomicMin key of the last chunk IS the winner's loss, bit for bit


def test_multi_start_per_step_trace(cuda):
    """trace=True: the kernels record the best objective of EVERY optimiser step (step_keys, include/lfm_b200.h) whatever
    the launch boundaries; it equals the column-wise minimum of the loss history bit for bit, and the fit itself is the
    same as with per-chunk keys."""
    from dis_project_b200.batched import make_restarts, multi_start_fit
    x, y, _, _ = o.synthetic_problem(5, 7, 3, seed=6)
    TH = make_restarts(o.Params.reference_init(5).pack(), 12)
    ref = multi_start_fit(x, y, TH, 1e-4, num_iters=40, chunk=7)
    for chunk in (None, 7, 1):
        res = multi_start_fit(x, y, TH, 1e-4, num_iters=40, chunk=chunk, trace=True)
        # (launch boundaries change the rounding of Adam's running bias products: same fit to 1e-11, not bit for bit)
        assert relerr(res.history, ref.history) < 1e-11 and relerr(res.theta, ref.theta) < 1e-10
        assert res.best_trace.shape == (40,)
        colmin = np.where(np.isfinite(res.history), res.history, np.inf).min(axis=0)
        assert np.array_equal(res.best_trace, colmin)
        assert res.best_id == ref.best_id and res.best_loss == colmin[-1]
        assert np.array_equal(res.best_theta, res.theta[res.best_id])
    # device-resident inputs are copied into the same plan's device buffer: the same fit
    res2 = multi_start_fit(torch.as_tensor(x).cuda(), torch.as_tensor(y).cuda(), TH, 1e-4, num_iters=40, chunk=1, trace=True)
    assert np.array_equal(res2.history, res.history) and np.array_equal(res2.best_trace, res.best_trace)


def test_multi_start_cached_plan_matches_a_fresh_plan(cuda):
    """Every fit runs over a per-shape plan (staging buffers, state, pointers built once) that later fits of the same shape
    reuse; the results on a reused plan are those on a freshly built one bit for bit, a second fit on the same plan with
    another X / y / start points is not polluted by the first, and the arrays handed back stay valid after later fits
    (they are not views of a reused buffer)."""
    from dis_project_b200 import batched
    from dis_project_b200.batched import make_restarts, multi_start_fit
    TH = make_restarts(o.Params.reference_init(5).pack(), 12)
    sets = [o.synthetic_problem(5, 7, 3, seed=s)[:2] for s in (6, 9)]

    def fresh(*args, **kw):
        batched._PLANS.clear()
        return multi_start_fit(*args, **kw)

    for kw in ({"chunk": 7}, {"chunk": None, "trace": True}, {"chunk": 10, "trace": True}):
        refs = [fresh(x, y, TH, 1e-4, num_iters=30, **kw) for x, y in sets]
        batched._PLANS.clear()
        got = [multi_start_fit(x, y, TH, 1e-4, num_iters=30, **kw) for x, y in sets]
        got.append(multi_start_fit(sets[0][0], sets[0][1], TH[::-1].copy(), 1e-4, num_iters=30, **kw))
        assert len(batched._PLANS) == 1
        for r, g in zip(refs, got):
            assert np.array_equal(r.theta, g.theta) and np.array_equal(r.history, g.history) and np.array_equal(r.info, g.info)
            assert np.array_equal(r.best_trace, g.best_trace) and r.best_id == g.best_id and r.best_loss == g.best_loss
            assert np.array_equal(r.best_theta, g.best_theta)
        assert np.array_equal(got[2].history[::-1], got[0].history)   # same data set, start points reversed
    # per-LFM observations through the plan
    Y = np.stack([sets[0][1] + 0.01 * b for b in range(12)])
    r = fresh(sets[0][0], Y, TH, 1e-4, num_iters=20, chunk=None, trace=True)
    multi_start_fit(sets[1][0], Y[::-1].copy(), TH, 1e-4, num_iters=20, chunk=None, trace=True)
    g = multi_start_fit(sets[0][0], Y, TH, 1e-4, num_iters=20, chunk=None, trace=True)
    assert np.array_equal(r.history, g.history) and np.array_equal(r.theta, g.theta)


_TWO_RANK_RUNS = [(B, name, kw) for B in (12, 1) for name, kw in (("chunk7", {"chunk": 7}),
                                                                   ("trace", {"chunk": None, "trace": True}))]


def _two_rank_inputs():
    from dis_project_b200.batched import make_restarts
    x, y, _, _ = o.synthetic_problem(5, 7, 3, seed=6)
    return x, y, make_restarts(o.Params.reference_init(5).pack(), 12)


def _two_rank_worker(rank, port, q):
    """One rank of test_multi_start_two_ranks_on_one_device: every run of _TWO_RANK_RUNS in a gloo world of two."""
    import traceback
    import torch.distributed as dist
    try:
        from dis_project_b200.batched import multi_start_fit
        torch.cuda.set_device(0)
        dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=2)
        try:
            x, y, TH = _two_rank_inputs()
            out = {}
            for B, name, kw in _TWO_RANK_RUNS:
                r = multi_start_fit(x, y, TH[:B], 1e-4, num_iters=40, **kw)
                out[(B, name)] = (r.lo, r.hi, r.history, r.theta, r.best_id, r.best_loss, r.best_theta, r.best_trace)
        finally:
            dist.destroy_process_group()
        q.put((rank, out))
    except Exception:
        q.put((rank, traceback.format_exc()))


def test_multi_start_two_ranks_on_one_device(cuda):
    """The multi-rank logic of multi_start_fit -- shards, the side-stream MIN all-reduce of the per-chunk keys, the gather
    of every rank's winner with the per-step trace, and an empty shard (B = 1 over two ranks) -- in a gloo world of two
    processes that share cuda:0.  Each rank's shard is the matching rows of a one-process fit (the team size may differ
    with the shard size, hence a tolerance), and both ranks report that fit's winner and best-objective trace exactly."""
    import socket
    import torch.multiprocessing as tmp
    from dis_project_b200.batched import multi_start_fit, shard_bounds
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    ctx = tmp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_two_rank_worker, args=(r, port, q)) for r in range(2)]
    try:
        for p in procs:
            p.start()
        got = dict(q.get(timeout=600) for _ in procs)
        for p in procs:
            p.join(timeout=120)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join()
    for rank in (0, 1):
        assert isinstance(got[rank], dict), got[rank]
    x, y, TH = _two_rank_inputs()
    for B, name, kw in _TWO_RANK_RUNS:
        ref = multi_start_fit(x, y, TH[:B], 1e-4, num_iters=40, **kw)
        for rank in (0, 1):
            lo, hi, hist, theta, best_id, best_loss, best_theta, best_trace = got[rank][(B, name)]
            assert (lo, hi) == shard_bounds(B, rank, 2), (B, name, rank)
            assert hist.shape == (hi - lo, 40) and theta.shape == (hi - lo, 17)
            if hi > lo:
                assert relerr(hist, ref.history[lo:hi]) < 1e-11 and relerr(theta, ref.theta[lo:hi]) < 1e-10, (B, name, rank)
            assert best_id == ref.best_id and best_loss == ref.best_loss, (B, name, rank)
            assert np.array_equal(best_theta, ref.best_theta) and np.array_equal(best_trace, ref.best_trace), (B, name, rank)


def test_examples_main_runs_the_reference_script(cuda, tmp_path):
    """examples/main.py = the reference's src/main.py call sequence: runs end to end on the synthetic p53 set and
    writes the tables behind the reference's three figures; p21 stays pinned (trainer.py:218-220)."""
    import csv
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "examples", "main.py"), "--out-dir", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert sorted(os.listdir(tmp_path)) == ["comparison.csv", "gene_expression.csv", "hyperparams.csv", "latent_force.csv", "plots"]
    assert sorted(os.listdir(tmp_path / "plots")) == ["gpjax_comparison.svg", "gpjax_gxpr.svg", "gpjax_lf.svg"]   # main.py:67-76
    lf = list(csv.DictReader(open(tmp_path / "latent_force.csv")))
    assert len(lf) == 100 and all(np.isfinite(float(x["mean"])) and float(x["stddev"]) > 0 for x in lf)
    # Figure-level check (the closest thing to the reference's visual validation that is possible without the Barenco
    # CSVs): the synthetic set is the SIM ODE driven by Barenco's measured profile (dataset.py:111-113), so the fitted
    # latent mean must follow that profile up to the scale / offset the model cannot identify (f enters through S_j f + B_j):
    # correlation with the profile at the seven measurement times, and the profile inside the 2-sigma band after the
    # best affine map.
    from dis_project_b200.dataset import F_BARENCO
    t = np.array([float(x["t"]) for x in lf]); m = np.array([float(x["mean"]) for x in lf]); sd = np.array([float(x["stddev"]) for x in lf])
    at = np.array([np.interp(tt, t, m) for tt in np.linspace(0, 12, 7)])
    sd_at = np.array([np.interp(tt, t, sd) for tt in np.linspace(0, 12, 7)])
    corr = np.corrcoef(at[1:], F_BARENCO[1:])[0, 1]      # (t = 0 is pinned to f(0) = 0 by the SIM kernel)
    A = np.stack([F_BARENCO[1:], np.ones(6)], axis=1)
    coef, *_ = np.linalg.lstsq(A, at[1:], rcond=None)
    resid = A @ coef - at[1:]
    # measured on a B200 in round 2: fitted mean [0.38 1.43 1.85 1.50 0.65 0.18 0.43] at t = 0, 2, ..., 12 against Barenco's
    # [0.18 1.18 1.62 0.82 0.69 -0.18 0.51]: correlation 0.91, slope 1.006, offset 0.23, largest residual 0.45 at t = 6
    # (the RBF prior rounds the corner of the piecewise-linear drive).  Band: correlation > 0.85, slope within 30 % of
    # one, residuals below 0.6.
    assert sd_at.min() > 0 and corr > 0.85, corr
    assert 0.7 < coef[0] < 1.3 and np.max(np.abs(resid)) < 0.6, (coef, resid)
    # learned sensitivities land where the reference's own figures put them (src/gpytorch_alfi/plots/gpytorch_comparison.png:
    # S ~ 0.71-0.77 for the non-p21 genes, p21 pinned to S = 1, D = 0.8; SURVEY.md 8c)
    S_learned = np.array([float(r["S_learned"]) for r in csv.DictReader(open(tmp_path / "comparison.csv"))])
    assert np.all((S_learned[[0, 1, 2, 4]] > 0.55) & (S_learned[[0, 1, 2, 4]] < 0.95))
    cmp_rows = list(csv.DictReader(open(tmp_path / "comparison.csv")))
    assert len(cmp_rows) == 5 and float(cmp_rows[3]["S_learned"]) == 1.0 and float(cmp_rows[3]["D_learned"]) == 0.8


def test_bench_dump_outputs_are_the_last_timed_step(cuda, tmp_path):
    """bench.py --dump-outputs: after the timed steps, the NLML+gradient and status the evaluation plan returned in the
    last one are written as float64 .npy files; two runs with the same arguments write the same bits (seeded inputs), and
    --impl reference writes the oracle's numbers for the same inputs, which they match to 1e-9.  Both arms run exactly
    --steps timed steps: the device arm's launch count is that many replays of the N = 4000 evaluation plan."""
    import subprocess
    import sys
    from dis_project_b200 import _lib, ops
    lib = _lib.lib()
    plan = ops.NlmlGradPlan(o.make_inputs(50, 80), np.zeros(4000), 50, 1e-4)   # bench.py's config-2 shape
    th = o.Params.reference_init(50).pack()
    plan(th)
    l0 = lib.lfm_debug_launch_count()
    plan(th)
    launches_per_step = lib.lfm_debug_launch_count() - l0
    plan.close()
    assert launches_per_step > 0
    bench = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py")
    dumps = []
    for run, extra in (("a", []), ("b", []), ("ref", ["--impl", "reference"])):
        d = tmp_path / run
        r = subprocess.run([sys.executable, bench, "--steps", "2", "--warmup", "1", "--no-secondary", "--no-cpu",
                            "--dump-outputs", str(d)] + extra, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        if extra:
            assert line["steps_executed"] == 2
        else:
            assert line["gpu_launches"] == 2 * launches_per_step, (line["gpu_launches"], launches_per_step)
        assert sorted(os.listdir(d)) == ["info.npy", "nlml_grad.npy"]
        dumps.append((np.load(d / "nlml_grad.npy"), np.load(d / "info.npy")))
    (out, info), (out2, info2), (ref, _) = dumps
    assert out.dtype == np.float64 and out.shape == (3 * 50 + 3,) and info.tolist() == [0.0]
    assert np.array_equal(out, out2) and np.array_equal(info, info2)
    assert abs(out[0] - ref[0]) <= RTOL * abs(ref[0]) and relerr(out[1:], ref[1:]) < RTOL


def test_batched_team_size_follows_the_batch(cuda):
    """lfm_batched_team_size: a shard that leaves SMs idle gets four warps per LFM, a full GPU one warp per LFM,
    shapes outside the warp / team kernels report 0 (CTA-per-LFM kernel)."""
    from dis_project_b200 import _lib
    lib = _lib.lib()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert lib.lfm_batched_team_size(sms, 105, 5, 35, 7) == 4
    assert lib.lfm_batched_team_size(64 * sms, 105, 5, 35, 7) == 1
    assert lib.lfm_batched_team_size(512, 105, 5, 105, 7) == 0      # 105 unique rows: beyond the register / tile kernels
    assert lib.lfm_batched_team_size(512, 105, 5, 35, 0) == 0       # no time grid


def test_batched_best_packs_the_winner(cuda):
    """lfm_batched_best: arg-min over the FINITE entries of one history column (ties -> smallest index), packed with
    the winner's theta; empty shards and all-NaN columns give [inf, -1]."""
    from dis_project_b200 import ops
    rng = np.random.default_rng(3)
    B, P, S = 1000, 17, 5
    hist = rng.standard_normal((B, S))
    hist[rng.integers(0, B, 50), 3] = np.nan
    hist[[700, 123], 3] = hist[:, 3][np.isfinite(hist[:, 3])].min() - 1.0   # a tie: index 123 wins
    hist[5, 3] = -np.inf                                                     # not finite: never wins
    theta = rng.standard_normal((B, P))
    out = torch.empty(P + 2, dtype=torch.float64, device="cuda")
    ops.batched_best(torch.as_tensor(hist).cuda(), 3, torch.as_tensor(theta).cuda(), 4000.0, out)
    got = out.cpu().numpy()
    assert got[0] == hist[123, 3] and got[1] == 4123.0 and np.array_equal(got[2:], theta[123])
    ops.batched_best(torch.full((7, S), float("nan"), dtype=torch.float64, device="cuda"), 0,
                     torch.zeros((7, P), dtype=torch.float64, device="cuda"), 0.0, out)
    assert out[0].item() == np.inf and out[1].item() == -1.0
    ops.batched_best(None, 0, None, 0.0, out)
    assert out[0].item() == np.inf and out[1].item() == -1.0


def test_config2_full_size_parity(cuda):
    """BASELINE config 2 (N=4000) against the oracle on the host cores."""
    from dis_project_b200 import ops
    x = o.make_inputs(50, 80)
    rng = np.random.default_rng(42)
    y = rng.standard_normal(4000)
    p = o.Params.reference_init(50)
    v_ref, g_ref = o.nlml_and_grad(p, x, y)
    out, info = ops.nlml_grad(x, y, p.pack(), 1e-4, 50)
    out = out.cpu().numpy()
    assert int(info.item()) == 0 and abs(out[0] - v_ref) <= RTOL * abs(v_ref) and relerr(out[1:], g_ref) < RTOL
    v1, _ = ops.nlml(x, y, p.pack(), 1e-4, 50)  # value-only path: recursive TRSV instead of the explicit inverse
    assert abs(v1.item() - v_ref) <= RTOL * abs(v_ref)


def test_config3_full_size_properties(cuda):
    """BASELINE config 3 (N=32768): size-independent properties -- determinism, agreement of the two
    NLML code paths (TRSV vs explicit inverse), directional finite difference of the gradient, and
    L L^T = Sigma, Sigma^-1 Sigma = I on probe vectors through the debug entry points."""
    from dis_project_b200 import ops
    free, _ = torch.cuda.mem_get_info()
    if free < 40 << 30:
        pytest.skip("needs ~40 GB of HBM")
    G, T = 256, 128
    x = o.make_inputs(G, T)
    rng = np.random.default_rng(1)
    y = rng.standard_normal(G * T)
    th = o.Params.reference_init(G).pack()
    th[:G] = rng.uniform(0.3, 0.9, G)
    out, info = ops.nlml_grad(x, y, th, 1e-4, G)
    out = out.cpu().numpy()
    out2, _ = ops.nlml_grad(x, y, th, 1e-4, G)
    assert int(info.item()) == 0 and np.all(np.isfinite(out))
    assert np.array_equal(out, out2.cpu().numpy())  # fixed reduction orders: bit-reproducible
    v, _ = ops.nlml(x, y, th, 1e-4, G)
    assert abs(v.item() - out[0]) <= 1e-10 * abs(out[0])
    dvec = rng.standard_normal(th.shape[0]) * th * 1e-2
    h = 1e-4
    vp, _ = ops.nlml(x, y, th + h * dvec, 1e-4, G)
    vm, _ = ops.nlml(x, y, th - h * dvec, 1e-4, G)
    fd = (vp.item() - vm.item()) / (2 * h)
    assert fd == pytest.approx(float(out[1:] @ dvec), rel=1e-5)
    ops.release_workspaces()
    torch.cuda.empty_cache()
    # dense factorisation properties at full size
    n = 32768
    K = ops.gram(x, th, G)
    K.diagonal().add_(1.0 + 1e-4)
    probe = torch.randn(n, 4, dtype=torch.float64, device=K.device)
    Kp = K @ probe
    L, Sinv, info = ops.debug_potrf_potri(K)  # in place: K now holds L
    assert int(info.item()) == 0
    Lt = torch.tril(L)
    assert relerr((Lt @ (Lt.T @ probe)).cpu().numpy(), Kp.cpu().numpy()) < 1e-11
    Si = torch.tril(Sinv) + torch.tril(Sinv, -1).T
    assert relerr((Si @ Kp).cpu().numpy(), probe.cpu().numpy()) < 1e-9


def test_config5_full_size_posterior_properties(cuda):
    """BASELINE config 5 (latent posterior at 102 400 test times from the N=32768 LFM): size-independent
    properties -- the streamed chunks are independent of each other (a random subset evaluated in its own
    call reproduces the same numbers), 0 < var <= prior variance 1 + 2 jitter, and at test times far
    outside the data the posterior returns to the prior."""
    from dis_project_b200 import ops
    free, _ = torch.cuda.mem_get_info()
    if free < 40 << 30:
        pytest.skip("needs ~40 GB of HBM")
    G, T, TS = 256, 128, 102400
    x = o.make_inputs(G, T)
    rng = np.random.default_rng(5)
    y = rng.standard_normal(G * T)
    var = rng.uniform(0.01, 0.1, G * T)
    th = o.Params.reference_init(G).pack()
    th[:G] = rng.uniform(0.3, 0.9, G)
    ts = np.stack((np.linspace(0, 13, TS), -np.ones(TS), np.zeros(TS)), axis=1)
    ts[-1, 0] = 60.0                                     # far from every observation
    m, v, info = ops.latent_posterior(x, y, var, th, 1e-4, ts, G)
    m, v = m.cpu().numpy(), v.cpu().numpy()
    assert int(info.item()) == 0 and np.all(np.isfinite(m)) and np.all(np.isfinite(v))
    assert np.all(v > 0) and np.all(v <= 1.0 + 2e-4 + 1e-12)
    assert abs(m[-1]) < 1e-12 and abs(v[-1] - (1.0 + 2e-4)) < 1e-12
    sub = np.sort(rng.choice(TS, 300, replace=False))
    m2, v2, _ = ops.latent_posterior(x, y, var, th, 1e-4, ts[sub], G)
    assert relerr(m2.cpu().numpy(), m[sub]) < 1e-12
    assert relerr(v2.cpu().numpy(), v[sub]) < 1e-12
    ops.release_workspaces()
    torch.cuda.empty_cache()


@pytest.mark.parametrize("G,T,R,Ts", [(5, 7, 1, 100), (5, 7, 3, 100), (6, 50, 1, 30)])
def test_multi_gene_predict(cuda, G, T, R, Ts):
    """SURVEY 8(f) row 1: ExactLFM.multi_gene_predict (model.py:465-514) incl. the off-by-one gene
    indices of generate_test_times_pred (clamped like jnp, Q6) and the third noise model (Q2)."""
    from dis_project_b200 import ops
    x, y, var, _ = o.synthetic_problem(G, T, R, seed=21)
    rng = np.random.default_rng(22)
    p = o.Params(d=rng.uniform(0.2, 1.0, G), s=rng.uniform(0.5, 1.5, G), b=rng.uniform(0.01, 0.1, G),
                 l=float(rng.uniform(0.8, 3.2)), sigma=float(rng.uniform(0.6, 1.4)), jitter=1e-4)
    t = o.generate_test_times_pred(Ts, G)
    m_ref, c_ref = o.multi_gene_predict(p, t, x, y, var)
    m, c, v, info = ops.gene_posterior(x, y, var, p.pack(), p.jitter, t, G)
    assert int(info.item()) == 0
    assert relerr(m.cpu().numpy(), m_ref) < RTOL
    assert relerr(c.cpu().numpy(), c_ref) < RTOL
    assert relerr(v.cpu().numpy(), np.diag(c_ref)) < RTOL
    m2, c2, v2, _ = ops.gene_posterior(x, y, var, p.pack(), p.jitter, t, G, full_cov=False)
    assert c2 is None and np.array_equal(v2.cpu().numpy(), v.cpu().numpy())


def test_gene_expression_predictor(cuda):
    from dis_project_b200.dataset import JaxP53Data, dataset_3d
    from dis_project_b200.model import ExactLFM
    from dis_project_b200.utils import GeneExpressionPredictor
    data = JaxP53Data.synthetic(replicate=0)
    model = ExactLFM(jitter=1e-4, data=data)
    times, means, stds = GeneExpressionPredictor(model, data, t=40).predict()
    x, y, var = dataset_3d(data)
    m_ref, c_ref = o.multi_gene_predict(o.Params.reference_init(5), o.generate_test_times_pred(40, 5), x, y, var)
    assert times.shape == (200, 3) and len(means) == 5 and means[0].shape == (40,)
    assert relerr(means[0], m_ref[:40]) < RTOL
    assert relerr(means[2], m_ref[120:160]) < RTOL  # blocks 3 and 4 swapped, as the reference does (utils.py:135-140)
    assert relerr(stds[4], np.sqrt(np.diag(c_ref))[160:]) < RTOL


@pytest.mark.parametrize("G,T,R", [(5, 7, 1), (5, 7, 3), (6, 50, 1), (12, 40, 2)])
def test_time_grid_tables_match_direct_evaluation(cuda, G, T, R):
    """Time-grid tables (include/lfm_b200.h, *_tg): same NLML / gradient as evaluating every entry, against the
    oracle too; a too-small bound falls back on the device; time_grid=0 is the direct path."""
    from dis_project_b200 import ops
    x, y, var, _ = o.synthetic_problem(G, T, R, seed=31)
    rng = np.random.default_rng(32)
    p = o.Params(d=rng.uniform(0.2, 1.0, G), s=rng.uniform(0.5, 1.5, G), b=rng.uniform(0.01, 0.1, G),
                 l=float(rng.uniform(0.8, 3.2)), sigma=float(rng.uniform(0.6, 1.4)), jitter=1e-4)
    assert ops.distinct_times(x) == T
    v_ref, g_ref = o.nlml_and_grad(p, x, y)
    direct, info0 = ops.nlml_grad(x, y, p.pack(), p.jitter, G, time_grid=0)
    tab, info1 = ops.nlml_grad(x, y, p.pack(), p.jitter, G)                   # bound counted from X
    small, info2 = ops.nlml_grad(x, y, p.pack(), p.jitter, G, time_grid=max(T - 2, 1))  # bound too small
    loose, _ = ops.nlml_grad(x, y, p.pack(), p.jitter, G, time_grid=T + 5)
    direct, tab, small, loose = (t.cpu().numpy() for t in (direct, tab, small, loose))
    assert int(info0.item()) == 0 and int(info1.item()) == 0 and int(info2.item()) == 0
    for out in (direct, tab, small, loose):
        assert abs(out[0] - v_ref) <= RTOL * abs(v_ref)
        assert np.max(np.abs(out[1:] - g_ref)) <= RTOL * np.max(np.abs(g_ref))
    assert np.array_equal(small, direct)                    # the fallback IS the direct path
    assert abs(tab[0] - direct[0]) <= 1e-13 * abs(direct[0])
    assert np.max(np.abs(tab[1:] - direct[1:])) <= 1e-12 * np.max(np.abs(direct[1:]))
    assert np.max(np.abs(loose - tab)) <= 1e-12 * np.max(np.abs(tab))
    v, _ = ops.nlml(x, y, p.pack(), p.jitter, G)
    assert abs(v.item() - v_ref) <= RTOL * abs(v_ref)


def test_time_grid_irregular_times_use_direct_path(cuda):
    """Every row its own time: the tables would be larger than the matrix, the library evaluates directly."""
    from dis_project_b200 import ops
    G, T = 4, 30
    x, y, var, _ = o.synthetic_problem(G, T, 1, seed=33)
    x = x.copy()
    x[:, 0] += np.random.default_rng(34).uniform(0, 0.05, x.shape[0])
    p = o.Params.reference_init(G)
    assert ops.distinct_times(x) == G * T
    v_ref, g_ref = o.nlml_and_grad(p, x, y)
    out, info = ops.nlml_grad(x, y, p.pack(), p.jitter, G)
    out0, _ = ops.nlml_grad(x, y, p.pack(), p.jitter, G, time_grid=0)
    assert np.array_equal(out.cpu().numpy(), out0.cpu().numpy())
    out = out.cpu().numpy()
    assert abs(out[0] - v_ref) <= RTOL * abs(v_ref)
    assert np.max(np.abs(out[1:] - g_ref)) <= RTOL * np.max(np.abs(g_ref))


def test_evaluation_plan_replays_the_eager_path(cuda):
    """CUDA-graph evaluation plans (include/lfm_b200.h): bit-identical to the stream-launched evaluation, at several
    theta values written into the bound buffer, constrained and unconstrained; also through CustomConjMLL."""
    from dis_project_b200 import ops
    for (G, T, R) in ((5, 7, 3), (12, 50, 1)):
        x, y, var, _ = o.synthetic_problem(G, T, R, seed=51)
        rng = np.random.default_rng(52)
        plan = ops.NlmlGradPlan(x, y, G, 1e-4)
        plan_u = ops.NlmlGradPlan(x, y, G, 1e-4, unconstrained=True)
        for _ in range(3):
            p = o.Params(d=rng.uniform(0.2, 1.0, G), s=rng.uniform(0.5, 1.5, G), b=rng.uniform(0.01, 0.1, G),
                         l=float(rng.uniform(0.8, 3.2)), sigma=float(rng.uniform(0.6, 1.4)), jitter=1e-4)
            out, info = plan(p.pack())
            ref, _ = ops.nlml_grad(x, y, p.pack(), 1e-4, G)
            assert int(info.item()) == 0 and torch.equal(out, ref)
            v_ref, g_ref = o.nlml_and_grad(p, x, y)
            assert abs(out[0].item() - v_ref) <= RTOL * abs(v_ref)
            u = o.unconstrain(p.pack())
            out_u, _ = plan_u(u)
            ref_u, _ = ops.nlml_grad_unc(x, y, u, 1e-4, G)
            assert torch.equal(out_u, ref_u)
        plan.close(); plan_u.close()
    # the trainer's eager loop (N > 128) goes through the plan held by the objective
    from dis_project_b200 import gpx_compat as gpx
    from dis_project_b200.model import ExactLFM
    from dis_project_b200.objectives import CustomConjMLL
    from dis_project_b200.trainer import JaxTrainer
    from dis_project_b200.dataset import JaxP53Data
    G, T = 6, 30
    x, y, var, _ = o.synthetic_problem(G, T, 1, seed=53)
    data = gpx.Dataset(x, y.reshape(-1, 1))
    model = ExactLFM(jitter=1e-4, num_genes=G)
    tr = JaxTrainer(model, CustomConjMLL(negative=True), data, gpx.adam(0.01), None, 5)
    assert not tr._device_scan_ok()     # N = 180 > 128: the host loop with one plan replay per step
    m2, hist = tr.fit()
    _, h_ref = o.fit(model.pack(), x, y, 1e-4, num_iters=5)
    assert relerr(hist, h_ref) < 1e-9


def test_sm_partition_is_a_scheduling_choice_only(cuda, tmp_path):
    """The factorisation's streams live in green contexts (8-SM chain partition, 140-SM bulk partition, 72-SM
    sub-partition: csrc/chol.cu).  Which SMs a kernel runs on must not change a single bit of the result: the same
    N = 2048 evaluation (one right-looking sweep with the interleaved inverse, 16 blocks) in a child process with
    LFM_SM_PARTITION=0 (ordinary priority streams) equals this process's, eager and through a CUDA-graph plan."""
    import subprocess
    import sys
    from dis_project_b200 import ops
    G, T = 32, 64
    x, y, var, _ = o.synthetic_problem(G, T, 1, seed=61)
    th = o.Params.reference_init(G).pack()
    out, info = ops.nlml_grad(x, y, th, 1e-4, G)
    plan = ops.NlmlGradPlan(x, y, G, 1e-4)
    out_p, _ = plan(th)
    assert int(info.item()) == 0 and torch.equal(out, out_p)
    plan.close()
    v_ref, g_ref = o.nlml_and_grad(o.Params.reference_init(G), x, y)
    got = out.cpu().numpy()
    assert abs(got[0] - v_ref) <= RTOL * abs(v_ref) and relerr(got[1:], g_ref) < RTOL
    np.savez(tmp_path / "in.npz", x=x, y=y, th=th)
    code = ("import sys, numpy as np; sys.path.insert(0, %r); from dis_project_b200 import ops; "
            "d = np.load(%r); out, info = ops.nlml_grad(d['x'], d['y'], d['th'], 1e-4, %d); "
            "np.save(%r, out.cpu().numpy())"
            % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), str(tmp_path / "in.npz"), G,
               str(tmp_path / "out.npy")))
    env = dict(os.environ, LFM_SM_PARTITION="0")
    subprocess.run([sys.executable, "-c", code], check=True, env=env, timeout=300)
    other = np.load(tmp_path / "out.npy")
    assert np.array_equal(other, got)


def test_configs_3_and_5_full_size_oracle_parity(cuda, tmp_path):
    """BASELINE configs 3 and 5 against the oracle at FULL size (N = 32768; 102 400 test times, the oracle on a sample of
    256 of them): 1e-9 relative, north_star's tolerance.  The oracle takes minutes of host time (about 2.5 on 16 cores,
    profiles/fullsize_parity_r2.json, whose record tests/test_host.py checks)."""
    import subprocess
    import sys
    out = tmp_path / "fullsize.json"
    subprocess.run([sys.executable, os.path.join(os.path.dirname(os.path.dirname(__file__)), "tools", "fullsize_parity.py"),
                    "--out", str(out)], check=True)
    res = json.load(open(out))
    assert res["config3"]["pass"] and res["config5"]["pass"]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs in one process")
def test_two_devices_in_one_process(cuda):
    """ADVICE r1 / VERDICT r1 weak 9: kernel attributes (opt-in shared memory), the SM partition, the occupancy cache of
    the team-size choice and the side streams are per DEVICE; one process that drives two GPUs, from two host threads
    at once, gets the same results on both."""
    import threading
    from dis_project_b200 import ops
    x, y, var, _ = o.synthetic_problem(6, 50, 1, seed=71)       # N = 300: three 128-blocks through the DMMA Cholesky
    p = o.Params.reference_init(6)
    xb, yb, _, _ = o.synthetic_problem(5, 7, 3, seed=72)
    TH = np.stack([o.Params.reference_init(5).pack() * s for s in (1.0, 1.1, 0.9)])
    results = {}

    def work(dev):
        with torch.cuda.device(dev):
            out, info = ops.nlml_grad(torch.as_tensor(x).cuda(), torch.as_tensor(y).cuda(), p.pack(), p.jitter, 6)
            m, v, _ = ops.latent_posterior(x, y, var, p.pack(), p.jitter, o.generate_test_times(60), 6)
            st = ops.BatchedFitState(TH, 5, 12)
            ops.batched_fit_steps(st, xb, yb, 1e-4, 12)
            torch.cuda.synchronize()
            results[dev] = (out.cpu().numpy(), int(info.item()), m.cpu().numpy(), v.cpu().numpy(), st.hist.cpu().numpy(),
                            st.info.cpu().numpy())

    work(1)            # device 1 FIRST: a per-process "configured" flag set on device 0 would have hidden the bug
    work(0)
    first = dict(results)
    threads = [threading.Thread(target=work, args=(d,)) for d in (0, 1)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    v_ref, g_ref = o.nlml_and_grad(p, x, y)
    for d in (0, 1):
        out, info, m, v, hist, binfo = results[d]
        assert info == 0 and np.all(binfo == 0)
        assert abs(out[0] - v_ref) <= RTOL * abs(v_ref) and relerr(out[1:], g_ref) < RTOL
        for a, b in zip(results[d], first[d]):
            assert np.array_equal(a, b)                       # threads vs sequential: bit-identical
    for a, b in zip(results[0], results[1]):
        assert np.array_equal(a, b)                           # device 0 vs device 1: bit-identical
