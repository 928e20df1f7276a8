"""Host-side logic and the C-ABI surface (no GPU, no compute calls)."""
import ctypes
import os
import re

import numpy as np
import torch
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_capi_library_exports_every_declared_symbol():
    import __graft_entry__ as ge
    from dis_project_b200 import _lib

    if not os.path.exists(_lib.LIB_PATH):
        ge.build()
    header = open(os.path.join(ROOT, "include", "lfm_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(lfm_[a-z0-9_]+)\s*\(", header))
    declared -= {"lfm_status", "lfm_stream_t", "lfm_handle"}
    assert len(declared) >= 25
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/lfm_b200.h but not exported"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature in dis_project_b200/_lib.py"
    l = _lib.lib()
    assert l.lfm_abi_version() == 3
    assert l.lfm_status_string(-5).decode().startswith("no sm_100")
    assert l.lfm_nlml_workspace_bytes_tg(4000, 50, 0) >= 2 * 4096 * 4096 * 8
    assert l.lfm_nlml_workspace_bytes_tg(0, 5, 0) == 0


def test_product_path_has_no_cpu_fallback_and_never_imports_the_oracle():
    import torch
    from dis_project_b200 import _lib, ops

    for dirpath, _, files in os.walk(os.path.join(ROOT, "dis_project_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            ops.cross_covariance(np.zeros((2, 3)), np.zeros((2, 3)), np.ones(17), 5)
        with pytest.raises(RuntimeError):
            _lib.require_device()


def test_dataset_layout_and_errors():
    from dis_project_b200.dataset import JaxP53Data, dataset_3d, flatten_dataset_jax

    d0 = JaxP53Data.synthetic(replicate=0)
    X, y, v = dataset_3d(d0)
    assert X.shape == (35, 3) and y.shape == (35, 1) and v.shape == (35, 1)
    assert np.array_equal(X[:, 0], np.tile(np.linspace(0, 12, 7), 5))
    assert np.array_equal(X[:, 1], np.repeat(np.arange(5), 7)) and np.all(X[:, 2] == 1)
    da = JaxP53Data.synthetic()
    X, y, v = dataset_3d(da)
    assert X.shape == (105, 3) and len(da) == 15 and da.shape == (15, 2, 7)
    assert np.array_equal(X[:, 1], np.tile(np.repeat(np.arange(5), 7), 3))  # gene-major inside, replicate-major outside
    t, yy = flatten_dataset_jax(da)
    assert t.shape == (105,) and np.array_equal(yy, y.reshape(-1))
    with pytest.raises(AssertionError):
        JaxP53Data.synthetic(replicate=3)
    with pytest.raises(ValueError, match="Invalid gene names"):
        JaxP53Data.synthetic(selected_genes=["p21", "XYZ"])
    with pytest.raises(ValueError, match="Duplicate"):
        JaxP53Data.synthetic(selected_genes=["p21", "p21"])
    with pytest.raises(ValueError, match="Empty"):
        JaxP53Data.synthetic(selected_genes=[])
    with pytest.raises(IndexError):
        da[15]
    sub = JaxP53Data.synthetic(replicate=1, selected_genes=["p21", "DDB2"])
    assert sub.num_genes == 2 and sub.selected_indices == [3, 0]
    B, S, D = sub.params_ground_truth()
    assert D[0] == 0.8 and S[0] == 1.0
    with pytest.raises(FileNotFoundError):
        JaxP53Data(data_dir="/nonexistent")
    assert np.allclose(da.f_observed.reshape(-1), [0.1845, 1.1785, 1.6160, 0.8156, 0.6862, -0.1828, 0.5131])


def test_load_barenco_data_preprocessing(tmp_path):
    """CSV -> log-normal moments -> rescale by replicate-1 std (reference dataset.py:213-321)."""
    import pandas as pd
    from dis_project_b200.dataset import PROBE_TO_GENE, load_barenco_data

    rng = np.random.default_rng(0)
    cols = [f"cARP{r}-{t}hrs.CEL" for r in (1, 2, 3) for t in range(0, 14, 2)]
    probes = list(PROBE_TO_GENE) + ["1000_at", "1001_at"]
    ex = pd.DataFrame(rng.normal(2.0, 0.5, (len(probes), 21)), index=probes, columns=cols)
    se = pd.DataFrame(rng.uniform(0.05, 0.3, (len(probes), 21)), index=probes, columns=cols)
    ex.to_csv(tmp_path / "barencoPUMA_exprs.csv"); se.to_csv(tmp_path / "barencoPUMA_se.csv")
    out = load_barenco_data(str(tmp_path))
    assert out["gene_names"] == ["DDB2", "BIK", "DR5", "p21", "SESN1"]
    assert out["gene_expressions"].shape == (3, 5, 7) and out["p53_variances"].shape == (3, 1, 7)
    m = ex.loc["202284_s_at"].to_numpy(); v = se.loc["202284_s_at"].to_numpy() ** 2  # p21 -> index 3
    full = np.exp(m + v / 2)
    scale = np.std(full[:7], ddof=1)
    assert np.allclose(out["gene_expressions"][:, 3, :].reshape(-1), full / scale, rtol=1e-13)
    var_full = (np.exp(v) - 1) * np.exp(2 * m + v)
    assert np.allclose(out["gene_variances"][:, 3, :].reshape(-1), var_full / scale**2, rtol=1e-12)


def test_model_bijectors_and_module_surface():
    from dis_project_b200.model import ExactLFM
    from oracle import lfm_oracle as o

    m = ExactLFM(jitter=1e-4)
    assert m.num_genes == 5 and m.jitter == 1e-4 and float(m.l) == 2.5 and float(m.obs_stddev) == 1.0
    assert np.all(m.true_d == 0.4) and np.all(m.true_s == 1.0) and np.all(m.true_b == 0.05)
    u = m.unconstrain()
    assert np.allclose(u.pack(), o.unconstrain(m.pack()), rtol=1e-15)
    assert np.allclose(u.constrain().pack(), m.pack(), rtol=1e-15)
    assert m.stop_gradient() is m
    r = m.replace(true_s=np.arange(5.0))
    assert np.array_equal(r.true_s, np.arange(5.0)) and np.all(m.true_s == 1.0)
    with pytest.raises(ValueError):
        m.replace(nope=1)
    assert np.allclose(m.gamma(np.array([0, 1])), 0.4 * 2.5 / 2)
    with pytest.raises(NotImplementedError):
        m.gram(lambda a, b: 0.0, np.zeros((2, 3)))


def test_adam_and_gpx_compat():
    from dis_project_b200.gpx_compat import Dataset, GaussianDistribution, adam

    opt = adam(0.01)
    p = np.array([1.0, -2.0, 3.0])
    st = opt.init(p)
    m = np.zeros(3); v = np.zeros(3)
    for t in range(1, 4):
        g = np.array([0.5, -1.0, 2.0]) * t
        upd, st = opt.update(g, st, p)
        m = 0.9 * m + 0.1 * g; v = 0.999 * v + 0.001 * g * g
        ref = -0.01 * (m / (1 - 0.9**t)) / (np.sqrt(v / (1 - 0.999**t)) + 1e-8)
        assert np.allclose(upd, ref, rtol=1e-14)
        p = p + upd
    with pytest.raises(ValueError):
        Dataset(np.zeros((3, 3)), np.zeros((4, 1)))
    with pytest.raises(ValueError):
        Dataset(np.zeros((3, 3)), np.zeros(3))
    gd = GaussianDistribution(np.arange(3.0), np.array([1.0, 4.0, 9.0]))
    assert np.array_equal(gd.stddev(), [1, 2, 3]) and np.array_equal(gd.mean(), np.arange(3.0))


def test_restart_generation_sharding_and_winner_reduction():
    from dis_project_b200.batched import make_restarts, reduce_best_gathered, shard_bounds
    from oracle import lfm_oracle as o

    th0 = o.Params.reference_init(5).pack()
    TH = make_restarts(th0, 9)
    assert TH.shape == (9, 17) and np.allclose(TH[0], th0, rtol=1e-14)
    assert np.all(TH > 0) and np.all((TH[:, 15] > 0.5) & (TH[:, 15] < 3.5))
    u = o.unconstrain(TH[4])
    assert np.allclose(u, o.unconstrain(th0) + 0.5 * np.random.default_rng(46).standard_normal(17), rtol=1e-10)
    for B, w in ((4096, 8), (10, 4), (3, 8), (0, 2)):
        b = [shard_bounds(B, r, w) for r in range(w)]
        assert b[0][0] == 0 and b[-1][1] == B and all(b[i][1] == b[i + 1][0] for i in range(w - 1))
        assert max(h - l for l, h in b) - min(h - l for l, h in b) <= 1
    assert np.array_equal(reduce_best_gathered(np.array([[3.0, 7.0], [np.nan, 8.0], [1.5, 9.0]])), [1.5, 9.0])
    assert reduce_best_gathered(np.zeros((0, 2)))[1] == -1                 # an empty shard never wins
    rows = np.array([[2.0, 5.0, 0.0], [1.5, 9.0, 0.0], [np.nan, 1.0, 0.0], [1.5, 3.0, 0.0]])
    assert np.array_equal(reduce_best_gathered(rows), [1.5, 3.0])
    assert reduce_best_gathered(np.array([[np.inf, -1.0]]))[1] == -1


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    from dis_project_b200.batched import reduce_best_gathered, shard_bounds

    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    B = 11
    losses = np.array([5.0, 4.0, 9.0, 3.5, 8.0, 3.5, 7.0, 6.0, np.nan, 10.0, 12.0])
    lo, hi = shard_bounds(B, rank, world)
    # the shard's packed winner [loss, id, theta...] (lfm_batched_best on the device; theta stands in as 100 + id)
    ids = np.arange(lo, hi, dtype=np.float64)
    mine = reduce_best_gathered(np.stack([losses[lo:hi], ids], axis=1))
    row = torch.tensor([mine[0], mine[1], 100.0 + mine[1]], dtype=torch.float64)
    rows = [torch.empty(3, dtype=torch.float64) for _ in range(world)]
    dist.all_gather(rows, row)
    allp = torch.stack(rows).numpy()
    best = reduce_best_gathered(allp)
    owner = int(np.flatnonzero((allp[:, 0] == best[0]) & (allp[:, 1] == best[1]))[0])
    q.put((rank, lo, hi, float(best[0]), int(best[1]), float(allp[owner, 2])))
    dist.destroy_process_group()


def test_best_objective_gather_gloo_world2():
    """N > 1 host logic on CPU: contiguous shards, every rank's packed winner gathered through gloo and reduced as
    multi_start_fit does (MIN on the loss, ties -> lowest id, NaN never wins)."""
    import torch.multiprocessing as tmp

    ctx = tmp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert [(r[1], r[2]) for r in res] == [(0, 6), (6, 11)]
    assert all(r[3] == 3.5 and r[4] == 3 and r[5] == 103.0 for r in res)


def test_multi_start_fit_rejects_bad_shapes_before_any_device_work(monkeypatch):
    """multi_start_fit checks the shapes of X, y, the variances and the start points on the host and raises ValueError
    before it touches a device, for numpy arrays and torch tensors alike; a y of one value is not broadcast to every
    observation."""
    from dis_project_b200 import _lib, batched
    from dis_project_b200.batched import multi_start_fit
    from oracle import lfm_oracle as o

    def no_device():
        raise AssertionError("multi_start_fit reached the device with inputs it should have rejected")

    monkeypatch.setattr(_lib, "require_device", no_device)
    x, y, var, _ = o.synthetic_problem(5, 7, 3, seed=6)
    B, N = 4, x.shape[0]
    TH = np.tile(o.Params.reference_init(5).pack(), (B, 1))
    plans = dict(batched._PLANS)
    bad = [((x, np.array([2.5]), TH), {}),                        # one value for N = 105 observations
           ((x, y[:-1], TH), {}),                                  # wrong length
           ((x, np.tile(y, (B + 1, 1)), TH), {}),                  # (B + 1, N)
           ((x[:, :2], y, TH), {}),                                # X not (N, 3)
           ((x.reshape(-1), y, TH), {}),
           ((x, y, TH), {"variances": var[:-1]}),                  # variances neither (N,), (N, 1) nor (B, N)
           ((x, y, TH), {"variances": np.tile(var, (B + 1, 1))}),
           ((x, y, TH[:, :-1]), {})]                               # start points not (B, 3G+2)
    for args, kw in bad:
        with pytest.raises(ValueError):
            multi_start_fit(*args, 1e-4, num_iters=5, **kw)
        with pytest.raises(ValueError):   # the same shapes as CPU tensors
            multi_start_fit(*(torch.as_tensor(a) for a in args[:2]), args[2], 1e-4, num_iters=5,
                            **{k: torch.as_tensor(v) for k, v in kw.items()})
    assert batched._PLANS == plans


def test_count_distinct_times():
    import ctypes as C
    from dis_project_b200 import _lib
    lib = _lib.lib()
    x = np.stack((np.tile(np.linspace(0, 12, 7), 5), np.repeat(np.arange(5.0), 7), np.ones(35)), axis=1)
    assert lib.lfm_count_distinct_times(35, x.ctypes.data) == 7
    x2 = np.ascontiguousarray(np.concatenate([x, x + [[0.5, 0, 0]]]))
    assert lib.lfm_count_distinct_times(70, x2.ctypes.data) == 14
    assert lib.lfm_count_distinct_times(0, None) == 0
    assert lib.lfm_nlml_workspace_bytes_tg(4000, 50, 80) > lib.lfm_nlml_workspace_bytes_tg(4000, 50, 0)
    assert lib.lfm_nlml_workspace_bytes_tg(120, 4, 120) == lib.lfm_nlml_workspace_bytes_tg(120, 4, 0)  # tables not worthwhile


def test_count_distinct_times_many_values_and_unique_rows_rule():
    """Host helpers: the distinct-time count switches to a sort beyond 512 values (never O(N^2)); the unique-row
    hint mirrors the batched kernels' rule -- compress only when every distinct row occurs equally often."""
    from dis_project_b200 import _lib, ops
    lib = _lib.lib()
    rng = np.random.default_rng(0)
    t = rng.permutation(np.repeat(np.linspace(0, 50, 3000), 2))
    x = np.ascontiguousarray(np.stack((t, np.zeros_like(t), np.ones_like(t)), axis=1))
    assert lib.lfm_count_distinct_times(x.shape[0], x.ctypes.data) == 3000
    base = np.stack((np.tile(np.linspace(0, 12, 7), 5), np.repeat(np.arange(5.0), 7), np.ones(35)), axis=1)
    assert ops.unique_rows(base) == 35                                   # R = 1: no compression
    assert ops.unique_rows(np.tile(base, (3, 1))) == 35                   # three replicates: 105 rows -> 35
    ragged = np.ascontiguousarray(np.tile(base, (3, 1))[:-1])             # one replicate lost a measurement
    assert ops.unique_rows(ragged) == 104                                 # non-uniform multiplicity: sized for N
    assert lib.lfm_count_unique_rows(0, None) == 0


def test_training_rows_must_carry_flag_one():
    from dis_project_b200 import ops
    x = np.stack((np.tile(np.linspace(0, 12, 7), 5), np.repeat(np.arange(5.0), 7), np.ones(35)), axis=1)
    x[3, 2] = 0.0
    with pytest.raises(ValueError, match="flag 1"):
        ops._check_training_flags(x)
    ops._check_training_flags(np.where(np.arange(3) == 2, 1.0, x))     # all flags 1: fine


def test_objective_plan_key_follows_contents_not_object_ids():
    """ADVICE r1: the CUDA-graph plan of CustomConjMLL must not be replayed for a different data set that happens to
    live at the same address, nor after an in-place edit."""
    from dis_project_b200.objectives import _content_token
    a = np.arange(12.0).reshape(4, 3)
    b = a.copy()
    assert _content_token(a) == _content_token(b)
    b[2, 1] = np.nextafter(b[2, 1], 100.0)
    assert _content_token(a) != _content_token(b)
    c = a.copy(); c[[0, 1]] = c[[1, 0]]                                  # same multiset of values, different order
    assert _content_token(a) != _content_token(c)
    assert _content_token(a.reshape(2, 6)) != _content_token(a)
    t = torch.zeros(5, dtype=torch.float64)
    k0 = _content_token(t)
    t[1] = 3.0
    assert _content_token(t) != k0                                        # torch version counter


def test_loss_key_is_order_preserving():
    """include/lfm_b200.h best_key: double -> int64 map used for the atomicMin / MIN all-reduce of the best objective."""
    from dis_project_b200.ops import loss_key_to_float
    v = np.array([-np.inf, -1e300, -104.74, -1.0, -1e-300, -0.0, 0.0, 1e-300, 3.5, 1e300, np.inf])
    bits = v.view(np.int64)
    keys = np.where(bits >= 0, bits, bits ^ np.int64(0x7FFFFFFFFFFFFFFF))
    assert np.all(np.diff(keys) >= 0) and np.all(np.diff(keys)[[0, 1, 2, 3, 6, 7, 8, 9]] > 0)
    back = loss_key_to_float(keys)
    assert np.array_equal(back, v)
    assert loss_key_to_float(np.array([np.iinfo(np.int64).max]))[0] == np.inf


def test_library_links_against_the_runtime_only():
    """The SM partition of the factorisation uses driver-API entry points (green contexts) obtained through
    cudaGetDriverEntryPoint at run time: the shared library must not gain a link-time dependency on libcuda, or it
    would stop loading on a host without a driver (this container, a reference maintainer's build box)."""
    import re
    import subprocess
    from dis_project_b200 import _lib
    out = subprocess.run(["readelf", "-d", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    needed = re.findall(r"\(NEEDED\)\s+Shared library: \[([^\]]+)\]", out)
    assert any(n.startswith("libcudart") for n in needed), needed
    assert not any(n.startswith("libcuda.so") for n in needed), needed


def test_full_size_parity_record():
    """The committed record of tools/fullsize_parity.py (run on a B200 box in round 2): configs 3 and 5 against the
    oracle at full size, inside north_star's 1e-9."""
    import json
    rec = json.load(open(os.path.join(os.path.dirname(os.path.dirname(__file__)), "profiles", "fullsize_parity_r2.json")))
    assert rec["N"] == 32768 and rec["Tstar"] == 102400 and rec["config5"]["sampled_test_points"] >= 256
    assert rec["config3"]["rel_err_nlml"] < 1e-9 and rec["config3"]["rel_err_grad_vs_max_component"] < 1e-9
    assert rec["config5"]["rel_err_mean"] < 1e-9 and rec["config5"]["rel_err_var"] < 1e-9
    assert rec["config3"]["info"] == 0 and rec["config5"]["info"] == 0


def test_xla_ffi_translation_unit_matches_its_bindings():
    """csrc/lfm_xla_ffi.cc (the JAX leg, SURVEY 8b; serves src/trainer.py:126) compiles against a structural mock of
    xla/ffi/api/ffi.h: every handler is invocable with exactly the stream / argument / attribute / result types its
    Ffi::Bind() chain declares, and it only calls entry points that include/lfm_b200.h declares.  The real header is absent
    from this image, so the shared object itself is built by `make xla_ffi` where jaxlib is installed."""
    import shutil
    import subprocess
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    src = os.path.join(ROOT, "dis_project_b200", "csrc", "lfm_xla_ffi.cc")
    cmd = ["g++", "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "tests", "xla_ffi_mock"), "-I",
           "/usr/local/cuda/include", src]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    text = open(src).read()
    handlers = re.findall(r"XLA_FFI_DEFINE_HANDLER_SYMBOL\((\w+),", text)
    assert set(handlers) == {"LfmNlml", "LfmNlmlGrad", "LfmNlmlGradUnc", "LfmCrossCovariance", "LfmMeanFunction",
                             "LfmLatentPosterior", "LfmGenePosterior", "LfmBatchedFit"}
    shim = open(os.path.join(ROOT, "dis_project_b200", "jax_ffi.py")).read()
    for h in handlers:
        assert f'"{h}"' in shim, f"{h} is not registered by dis_project_b200/jax_ffi.py"
    # negative control: swapping two parameters of a handler must trip the static_assert of the mock
    bad = text.replace("ffi::Error MeanFunction(cudaStream_t stream, F64 X, F64 theta, int64_t G, RF64 out)",
                       "ffi::Error MeanFunction(cudaStream_t stream, F64 X, int64_t G, F64 theta, RF64 out)")
    assert bad != text
    res = subprocess.run(cmd[:-1] + ["-x", "c++", "-I", os.path.dirname(src), "-"], input=bad.replace(
        '#include "../../include/lfm_b200.h"', f'#include "{os.path.join(ROOT, "include", "lfm_b200.h")}"'),
        capture_output=True, text=True)
    assert res.returncode != 0 and "static assertion failed" in res.stderr


def test_jax_ffi_shim_refuses_cleanly_without_jax():
    try:
        import jax  # noqa: F401
        pytest.skip("jax is importable here")
    except ImportError:
        pass
    with pytest.raises(ImportError, match="jax"):
        import dis_project_b200.jax_ffi  # noqa: F401


def test_plotter_writes_the_reference_figures(tmp_path):
    """plotter.py: the three figures of src/main.py:67-76 (plot_lf, plot_predictions, plot_comparison_gpjax) with the
    reference's signatures and file names, drawn by the dependency-free SVG writer (host-side; fake predictive
    distributions stand in for the CUDA results here)."""
    from dis_project_b200 import plotter
    from dis_project_b200.dataset import JaxP53Data
    from dis_project_b200.gpx_compat import GaussianDistribution
    from dis_project_b200.utils import GeneExpressionPredictor, generate_test_times

    plotter.PLOTS_DIR = str(tmp_path)
    data = JaxP53Data.synthetic(replicate=0)
    tt = generate_test_times(50)
    dist = GaussianDistribution(np.sin(tt[:, 0] / 2.0), 0.01 + 0.05 * np.cos(tt[:, 0] / 5.0) ** 2)
    plotter.plot_lf(tt, dist, y_scatter=data.f_observed.squeeze(), stddev=2)
    plotter.plot_lf(tt, dist, stddev=1, title="Replicate 3", save_name="replicate3")

    class FakeModel:
        true_b, true_s, true_d = np.full(5, 0.05), np.ones(5), np.full(5, 0.4)

        def multi_gene_predict(self, x, d):
            n = x.shape[0]
            return GaussianDistribution(np.linspace(0, 1, n), np.full(n, 0.04))

    plotter.plot_comparison_gpjax(FakeModel(), data)
    gp = GeneExpressionPredictor(FakeModel(), data, t=20)
    gp.plot_predictions(data)
    files = sorted(os.listdir(tmp_path))
    assert files == ["gpjax_comparison.svg", "gpjax_gxpr.svg", "gpjax_lf.svg", "gpjax_lf_replicate3.svg"]
    lf = open(tmp_path / "gpjax_lf.svg").read()
    assert lf.startswith("<svg") and "Latent Force Model (GPJax)" in lf and "Predictive mean" in lf and "True values" in lf
    assert lf.count("<path") == 7            # Barenco's seven measured points as crosses
    assert "Replicate 3" in open(tmp_path / "gpjax_lf_replicate3.svg").read()
    cmp_svg = open(tmp_path / "gpjax_comparison.svg").read()
    assert all(g in cmp_svg for g in data.gene_names) and cmp_svg.count("<rect") >= 30
    assert open(tmp_path / "gpjax_gxpr.svg").read().count("Expression Over Time") == 5
