"""Parity against REFERENCE SOURCE EXECUTED HERE.

``tests/golden/ref_*.json`` were produced by importing the reference's own, unmodified
``src/{dataset,model,objectives,trainer,utils}.py`` under ``tests/refshim`` (torch-fp64 stand-ins
for jax / gpjax / cola / optax / tfp) and calling its functions on the CSVs of
``tests/golden/ref_csv`` (``tests/golden/make_ref_golden.py``).  Three layers are checked against them:

* CPU: the oracle (``oracle/lfm_oracle.py``) -- this is what pins the oracle to the reference;
* CPU: the host layer (``dis_project_b200/dataset.py``, ``utils.py``) -- loader, layout, selectors;
* GPU: the CUDA path through the C-ABI and the reference-shaped Python classes.

Tolerances (stated per assertion): 1e-9 relative on NLML / gradient / posterior moments
(north_star), 1e-11 of the matrix scale on covariance entries, 1e-8 / 1e-7 on 150-step optimiser
trajectories.  One documented exception: the reference writes ``erf(a) + erf(b)`` literally
(model.py:276-278, 349-351); where that sum cancels (SURVEY.md Q7) its own rounding noise reaches
2.4e-9 of the latent posterior mean at the 'random' point of the 3-gene case.  The oracle reproduces
that noise to 1e-12 when ``LITERAL_ERF_SUMS`` is set (asserted below); the product evaluates the
same quantity as erfc differences, which is the more accurate of the two.
"""
import json
import os

import numpy as np
import pytest

from oracle import lfm_oracle as o

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
CASES = ("p53_rep0", "p53_all", "p53_sub3")
RTOL = 1e-9
LITERAL_NOISE_TOL = 1e-8   # latent mean at a 'random' point: bounded by the reference's own erf-sum noise


def load(name):
    with open(os.path.join(GOLD, f"ref_{name}.json")) as fh:
        return json.load(fh)


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def arrays(c):
    return (np.array(c["X"]), np.array(c["y"]), np.array(c["variances"]), np.array(c["Xstar"]), np.array(c["Xgene"]),
            np.array(c["K_rows"]))


# ------------------------------------------------------------------------------------------------
# provenance
# ------------------------------------------------------------------------------------------------
def test_fixtures_carry_reference_provenance():
    for name in CASES + ("dataset",):
        c = load(name)
        assert c["provenance"].startswith("reference source executed")
        assert "src/model.py" in c["reference_files"] and c["generator"] == "tests/golden/make_ref_golden.py"
    c = load("p53_rep0")
    assert c["N"] == 35 and c["G"] == 5 and c["fix_params"] is True            # main.py:32,59
    assert load("p53_all")["N"] == 105 and load("p53_all")["fix_params"] is False   # notebook.py:36,73-75
    # the reference's own initial state (model.py:65,100-104,114)
    assert c["points"][0]["theta"] == [0.4] * 5 + [1.0] * 5 + [0.05] * 5 + [2.5, 1.0]


# ------------------------------------------------------------------------------------------------
# CPU: the oracle against the reference
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_execution(name):
    c = load(name)
    X, y, var, xs, xg, rows = arrays(c)
    G = c["G"]
    for pt in c["points"]:
        p = o.Params.unpack(np.array(pt["theta"]), c["jitter"])
        assert rel(o.unconstrain(p.pack()), pt["theta_unc"]) < 1e-13             # tfp bijector inverses
        assert rel(o.constrain(np.array(pt["theta_unc"])), pt["theta"]) < 1e-13
        val, g = o.nlml_and_grad(p, X, y)
        assert abs(val - pt["nlml"]) <= 1e-12 * abs(pt["nlml"])
        assert abs(pt["nlml_via_trainer_loss"] - pt["nlml"]) <= 1e-12 * abs(pt["nlml"])
        assert rel(g, pt["grad_constrained"]) < 1e-10
        vu, gu = o.nlml_and_grad_unc(np.array(pt["theta_unc"]), X, y, c["jitter"])
        assert abs(vu - pt["nlml"]) <= 1e-12 * abs(pt["nlml"]) and rel(gu, pt["grad_unconstrained"]) < 1e-10
        assert rel(o.mean_function(p, X), pt["mean_function"]) < 1e-15
        assert rel(o.cross_covariance(p, rows, rows), pt["K_block"]) < 1e-11      # mixed flags, gene index G clamps
        assert rel(np.diag(o.gram(p, X)), pt["gram_diag"]) < 1e-12
        m, v = o.latent_predict(p, xs, X, y, var)
        assert rel(m, pt["latent_mean"]) < (RTOL if pt["label"] == "init" else LITERAL_NOISE_TOL)
        assert rel(np.sqrt(v), pt["latent_std"]) < RTOL
        gm, gc = o.multi_gene_predict(p, xg, X, y, var)
        assert rel(gm, pt["gene_mean"]) < RTOL and rel(np.sqrt(np.diag(gc)), pt["gene_std"]) < RTOL
        assert rel(gc[0], pt["gene_cov_row0"]) < RTOL
        e = pt["entries"]
        for j, k, t1, t2, ref in e["h"]:
            assert abs(o.h(p, j, k, t1, t2) - ref) <= 1e-12 * max(abs(ref), 1.0)
        assert rel([o.gamma(p, i) for i in range(G)], e["gamma"]) < 1e-15
        assert abs(o.kernel_xx(p, 2.0, 1, 7.5, G - 1) - e["kernel_xx"]) <= 1e-12 * abs(e["kernel_xx"])
        assert abs(o.kernel_xf(p, 6.0, 1, 2.5) - e["kernel_xf"]) <= 1e-12 * abs(e["kernel_xf"])
        assert e["kernel_xf_swapped"] == e["kernel_xf"]                           # model.py:262-263
        assert abs(o.kernel_ff(p, 6.0, 2.5) - e["kernel_ff"]) <= 1e-14
    theta_fit, hist = o.fit(np.array(c["points"][0]["theta"]), X, y, c["jitter"], num_iters=150,
                            fix_params=c["fix_params"])
    assert rel(hist, c["fit"]["history"]) < 1e-9 and rel(theta_fit, c["fit"]["theta"]) < 1e-9
    if c["fix_params"] and G > 3:
        assert c["fit"]["theta"][3] == 0.8 and c["fit"]["theta"][G + 3] == 1.0    # Q5: pinned in constrained space


def test_oracle_literal_erf_form_reproduces_the_reference_noise():
    """With the literal erf(a)+erf(b) arithmetic of the reference the oracle agrees to 1e-12 even at the
    point where the default (erfc) form differs by 2.4e-9: the difference is the reference's rounding noise."""
    c = load("p53_sub3")
    X, y, var, xs, xg, rows = arrays(c)
    pt = c["points"][1]
    p = o.Params.unpack(np.array(pt["theta"]), c["jitter"])
    default = rel(o.latent_predict(p, xs, X, y, var)[0], pt["latent_mean"])
    o.LITERAL_ERF_SUMS = True
    try:
        literal = rel(o.latent_predict(p, xs, X, y, var)[0], pt["latent_mean"])
        assert rel(o.cross_covariance(p, rows, rows), pt["K_block"]) < 1e-14
    finally:
        o.LITERAL_ERF_SUMS = False
    assert literal < 1e-11 and default < LITERAL_NOISE_TOL


# ------------------------------------------------------------------------------------------------
# CPU: host layer (loader, selectors, layout, test-time generators) against the reference
# ------------------------------------------------------------------------------------------------
def test_host_dataset_layer_matches_reference_loader():
    from dis_project_b200.dataset import JaxP53Data, dataset_3d, flatten_dataset_jax, load_barenco_data
    from dis_project_b200 import utils

    ref = load("dataset")
    csv = os.path.join(GOLD, "ref_csv")
    raw = load_barenco_data(csv)
    assert raw["gene_names"] == ref["load_barenco_data"]["gene_names"]
    for k in ("gene_expressions", "gene_variances", "p53_expressions", "p53_variances"):
        assert rel(raw[k], ref["load_barenco_data"][k]) < 1e-13, k
    for v in ref["variants"]:
        d = JaxP53Data(data_dir=csv, **v["kwargs"])
        assert list(d.gene_names) == v["gene_names"] and list(d.selected_indices) == v["selected_indices"]
        assert d.num_genes == v["num_genes"] and len(d) == v["len"] and list(d.shape) == v["shape"]
        assert rel(d.timepoints, v["timepoints"]) == 0 and rel(d.f_observed, v["f_observed"]) == 0
        assert rel(d.gene_expressions, v["gene_expressions"]) < 1e-13
        assert rel(d.gene_variances, v["gene_variances"]) < 1e-13
        X, y, var = dataset_3d(d)
        assert np.array_equal(X, np.array(v["X"])) and rel(y, v["y"]) < 1e-13 and rel(var, v["variances"]) < 1e-13
        ft, fy = flatten_dataset_jax(d)
        assert np.array_equal(ft, np.array(v["flatten_t"])) and rel(fy, v["flatten_y"]) < 1e-13
        B, S, D = d.params_ground_truth()
        assert np.array_equal(B, v["B_exact"]) and np.array_equal(S, v["S_exact"]) and np.array_equal(D, v["D_exact"])
        assert rel(d[0][0], v["item0"][0]) == 0 and rel(d[0][1], v["item0"][1]) < 1e-13
    for kind, kw in (("invalid", {"selected_genes": ["p21", "nope"]}), ("duplicate", {"selected_genes": ["p21", "p21"]}),
                     ("empty", {"selected_genes": []})):
        with pytest.raises(ValueError) as ei:
            JaxP53Data(data_dir=csv, **kw)
        assert str(ei.value) == ref["errors"][kind]
    assert np.array_equal(utils.generate_test_times(5), np.array(ref["generate_test_times_5"]))
    assert np.array_equal(utils.generate_test_times_pred(2), np.array(ref["generate_test_times_pred_2"]))


# ------------------------------------------------------------------------------------------------
# GPU: the CUDA path against the reference
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_cuda_ops_match_reference_execution(cuda, name):
    from dis_project_b200 import ops

    c = load(name)
    X, y, var, xs, xg, rows = arrays(c)
    G, jit = c["G"], c["jitter"]
    for pt in c["points"]:
        th, thu = np.array(pt["theta"]), np.array(pt["theta_unc"])
        assert rel(ops.unconstrain(th, G).cpu().numpy(), thu) < 1e-12
        assert rel(ops.constrain(thu, G).cpu().numpy(), th) < 1e-12
        v, info = ops.nlml(X, y, th, jit, G)
        assert int(info.item()) == 0 and abs(v.item() - pt["nlml"]) <= RTOL * abs(pt["nlml"])
        out, info = ops.nlml_grad(X, y, th, jit, G)
        out = out.cpu().numpy()
        assert abs(out[0] - pt["nlml"]) <= RTOL * abs(pt["nlml"]) and rel(out[1:], pt["grad_constrained"]) < RTOL
        out, info = ops.nlml_grad_unc(X, y, thu, jit, G)
        out = out.cpu().numpy()
        assert abs(out[0] - pt["nlml"]) <= RTOL * abs(pt["nlml"]) and rel(out[1:], pt["grad_unconstrained"]) < RTOL
        bv, bg, binfo = ops.batched_nlml_grad_unc(X, y, thu[None, :], jit, G)      # the batched small-N kernels
        assert int(binfo.item()) == 0 and abs(bv.item() - pt["nlml"]) <= RTOL * abs(pt["nlml"])
        assert rel(bg.cpu().numpy()[0], pt["grad_unconstrained"]) < RTOL
        assert rel(ops.mean_function(X, th, G).cpu().numpy().reshape(-1), pt["mean_function"]) < 1e-15
        assert rel(ops.cross_covariance(rows, rows, th, G).cpu().numpy(), pt["K_block"]) < 1e-11
        assert rel(np.diag(ops.gram(X, th, G).cpu().numpy()), pt["gram_diag"]) < 1e-11
        m, pv, info = ops.latent_posterior(X, y, var, th, jit, xs, G)
        assert rel(m.cpu().numpy(), pt["latent_mean"]) < (RTOL if pt["label"] == "init" else LITERAL_NOISE_TOL)
        assert rel(np.sqrt(pv.cpu().numpy()), pt["latent_std"]) < RTOL
        gm, gc, gv, info = ops.gene_posterior(X, y, var, th, jit, xg, G)
        assert rel(gm.cpu().numpy(), pt["gene_mean"]) < RTOL
        assert rel(np.sqrt(gv.cpu().numpy()), pt["gene_std"]) < RTOL
        assert rel(gc.cpu().numpy()[0], pt["gene_cov_row0"]) < RTOL
        e = pt["entries"]
        hh = ops.h_terms(np.array([r[0] for r in e["h"]], dtype=np.float64), np.array([r[1] for r in e["h"]], dtype=np.float64),
                         np.array([r[2] for r in e["h"]]), np.array([r[3] for r in e["h"]]), th, G).cpu().numpy()
        assert rel(hh, [r[4] for r in e["h"]]) < 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_reference_call_sequence_on_cuda_matches_reference_execution(cuda, name):
    """main.py:30-78 / notebook.py:33-116 with this package's classes, on the reference's CSV format, against
    what the reference's own classes produced: entries, objective, 150-step fit, both posteriors."""
    from dis_project_b200.dataset import JaxP53Data, dataset_3d
    from dis_project_b200.gpx_compat import Dataset, adam
    from dis_project_b200.model import ExactLFM
    from dis_project_b200.objectives import CustomConjMLL
    from dis_project_b200.trainer import JaxTrainer
    from dis_project_b200.utils import GeneExpressionPredictor, generate_test_times

    c = load(name)
    G = c["G"]
    p53 = JaxP53Data(data_dir=os.path.join(GOLD, "ref_csv"), **c["data_kwargs"])
    X, y, var = dataset_3d(p53)
    assert np.array_equal(X, np.array(c["X"])) and rel(y.reshape(-1), c["y"]) < 1e-13
    train = Dataset(X, y)
    model = ExactLFM(jitter=1e-4, num_genes=G, data=p53)
    loss = CustomConjMLL(negative=True)
    pt = c["points"][0]
    assert abs(loss(model, train) - pt["nlml"]) <= RTOL * abs(pt["nlml"])
    e = pt["entries"]
    assert abs(model.kernel_xx([2.0, 1.0, 1.0], [7.5, G - 1.0, 1.0]) - e["kernel_xx"]) <= 1e-11 * abs(e["kernel_xx"])
    assert abs(model.kernel_xf([6.0, 1.0, 1.0], [2.5, -1.0, 0.0]) - e["kernel_xf"]) <= 1e-11 * abs(e["kernel_xf"])
    assert abs(model.kernel_xf([2.5, -1.0, 0.0], [6.0, 1.0, 1.0]) - e["kernel_xf"]) <= 1e-11 * abs(e["kernel_xf"])
    assert abs(model.kernel_ff([6.0, -1.0, 0.0], [2.5, -1.0, 0.0]) - e["kernel_ff"]) <= 1e-13
    assert abs(model.h(1, G - 1, 2.0, 7.5) - e["h"][0][4]) <= 1e-12 * abs(e["h"][0][4])
    trainer = JaxTrainer(model=model, objective=loss, training_data=train, optim=adam(0.01), key=None, num_iters=150)
    val, grad = loss.value_and_grad(trainer.model, train)
    assert abs(val - pt["nlml"]) <= RTOL * abs(pt["nlml"]) and rel(grad, pt["grad_unconstrained"]) < RTOL
    trained, history = trainer.fit(fix_params=c["fix_params"], num_steps_per_epoch=1000)
    assert rel(history, c["fit"]["history"]) < 1e-8
    assert rel(trained.pack(), c["fit"]["theta"]) < 1e-7
    xs = generate_test_times(100 - 100 % G)
    assert np.array_equal(xs, np.array(c["Xstar"]))
    lat = trained.latent_predict(xs, p53)
    assert rel(lat.mean(), c["fit"]["latent_mean"]) < 1e-6      # 150 chained Adam steps, then a posterior
    assert rel(lat.stddev(), c["fit"]["latent_std"]) < 1e-6
    # the posterior at the reference's OWN fitted parameters isolates the posterior kernels from the trajectory
    at_ref = model.with_leaves(np.array(c["fit"]["theta"]))
    lat = at_ref.latent_predict(xs, p53)
    assert rel(lat.mean(), c["fit"]["latent_mean"]) < LITERAL_NOISE_TOL and rel(lat.stddev(), c["fit"]["latent_std"]) < RTOL
    gp = GeneExpressionPredictor(at_ref, p53, t=12)
    assert np.array_equal(gp.generate_test_times_pred(), np.array(c["Xgene"]))
    gene = at_ref.multi_gene_predict(gp.generate_test_times_pred(), p53)
    assert rel(gene.mean(), c["fit"]["gene_mean"]) < RTOL and rel(gene.stddev(), c["fit"]["gene_std"]) < RTOL
    dec = gp.decompose_predictions2(gene.mean()) if G == 5 else gp.decompose_predictions(gene.mean())
    for a, b in zip(dec, c["fit"]["gene_mean_decomposed"]):
        assert rel(a, b) < RTOL


# ------------------------------------------------------------------------------------------------
# The reference's GPyTorch twin (src/gpytorch_alfi), executed under tests/refshim/shim_gpytorch.py: the heteroscedastic
# training objective K_xx + 1e-4 I + diag(variances) + noise I (model_alfi.py:294-299) and its block-structured Gram.
# The twin keeps its kernel parameters in float32 (model_alfi.py:191), so its numbers carry ~1e-7 relative rounding:
# tolerances here are 1e-5 (value, entries) and 1e-4 of the largest gradient component.
# ------------------------------------------------------------------------------------------------
TWIN_CASES = ("rep0", "rep2")


def _twin(name):
    with open(os.path.join(GOLD, f"ref_twin_{name}.json")) as fh:
        c = json.load(fh)
    G = c["G"]
    t, y, var = np.array(c["train_t"]), np.array(c["train_y"]), np.array(c["variances"])
    N = t.size
    X = np.stack((t, np.repeat(np.arange(G), N // G).astype(np.float64), np.ones(N)), axis=1)   # the twin's block layout
    return c, G, N, X, y, var


def _twin_theta_and_grad(pt, G, N):
    """theta = [d, s, b, l, sigma] of include/lfm_b200.h and d(NLML)/d(theta) from the twin's d(loss)/d(raw): loss =
    NLML / N; Positive = softplus (derivative sigmoid), Interval(0.5, 3.5) = 0.5 + 3 sigmoid, noise = softplus(raw) + 1e-4
    = sigma^2."""
    sig = lambda r: 1.0 / (1.0 + np.exp(-np.asarray(r, dtype=np.float64)))
    sigma = float(np.sqrt(pt["noise"]))
    theta = np.concatenate([pt["decay"], pt["sensitivity"], pt["basal"], [pt["lengthscale"], sigma]])
    sl = sig(pt["raw"]["lengthscale"])
    g = np.concatenate([np.array(pt["grad_raw"]["decay"]) / sig(pt["raw"]["decay"]),
                        np.array(pt["grad_raw"]["sensitivity"]) / sig(pt["raw"]["sensitivity"]),
                        np.array(pt["grad_raw"]["basal"]) / sig(pt["raw"]["basal"]),
                        np.array(pt["grad_raw"]["lengthscale"]) / (3.0 * sl * (1.0 - sl)),
                        np.array(pt["grad_raw"]["noise"]) / sig(pt["raw"]["noise"]) * 2.0 * sigma]) * N
    return theta, g


@pytest.mark.parametrize("name", TWIN_CASES)
def test_oracle_heteroscedastic_objective_matches_the_gpytorch_twin(name):
    c, G, N, X, y, var = _twin(name)
    assert c["provenance"].startswith("reference GPyTorch twin executed")
    for pt in c["points"]:
        theta, g_twin = _twin_theta_and_grad(pt, G, N)
        p = o.Params.unpack(theta, c["kernel_jitter"])
        val, g = o.nlml_and_grad(p, X, y, variances=var)
        assert abs(val / N - pt["loss"]) <= 1e-5 * abs(pt["loss"])                       # trainer_alfi.py:173
        K = o.gram(p, X) + np.diag(var) + c["kernel_jitter"] * np.eye(N)                # model_alfi.py:282-299
        assert rel(K, pt["K_xx"]) < 1e-6
        assert rel(o.mean_function(p, X), pt["mean"]) < 1e-7                             # model_alfi.py:540-546
        assert np.max(np.abs(g - g_twin)) <= 1e-4 * np.max(np.abs(g_twin))


@pytest.mark.gpu
@pytest.mark.parametrize("name", TWIN_CASES)
def test_cuda_heteroscedastic_objective_matches_the_gpytorch_twin(cuda, name):
    from dis_project_b200 import ops
    c, G, N, X, y, var = _twin(name)
    for pt in c["points"]:
        theta, g_twin = _twin_theta_and_grad(pt, G, N)
        out, info = ops.nlml_grad(X, y, theta, c["kernel_jitter"], G, variances=var)
        out = out.cpu().numpy()
        assert int(info.item()) == 0 and abs(out[0] / N - pt["loss"]) <= 1e-5 * abs(pt["loss"])
        assert np.max(np.abs(out[1:] - g_twin)) <= 1e-4 * np.max(np.abs(g_twin))
        K = ops.gram(X, theta, G).cpu().numpy() + np.diag(var) + c["kernel_jitter"] * np.eye(N)
        assert rel(K, pt["K_xx"]) < 1e-6

# ---- the twin's posteriors (model_alfi.py:68-150: predict_f / predict_m as main_alfi.py:55-57 calls them) ---------------
# Conventions the twin has and latent_predict / multi_gene_predict of src/model.py do not, expressed through the SAME entry
# points: no mean function (basal = 0), Sigma = K_xx + 1e-4 I + diag(variances) WITHOUT the likelihood noise (latent: sigma
# = 0 with jitter 1e-4; genes: sigma^2 = 1e-4), K_ff + 1e-3 I before and `jitter` after the Schur complement.  The fixture
# holds the run with the twin's float32 parameters (float32 rounding, amplified by torch.inverse) and the same unmodified
# methods after model.double(), where only K_xf's float32 buffer is left: predict_m then pins the conventions to 1e-9.
def _twin_posterior_problem(c, pt, which):
    G = c["G"]
    po = pt["posterior"]
    src = po["f64"] if which == "f64" else pt
    ts = np.array(po["t_predict"])
    T = ts.size
    d, s_, l = np.array(src["decay"]), np.array(src["sensitivity"]), float(src["lengthscale"])
    Xs = np.stack((ts, -np.ones(T), np.zeros(T)), axis=-1)                                         # utils.py:268-287 layout
    Xg = np.stack((np.tile(ts, G), np.repeat(np.arange(G), T).astype(np.float64), np.ones(G * T)), axis=-1)
    want = po["f64"] if which == "f64" else po
    f_mean, f_var = np.array(want["f_mean"]), np.array(want["f_var"])
    m_mean, m_var = np.array(want["m_mean"]).T.reshape(-1), np.array(want["m_var"]).T.reshape(-1)   # (80, G) -> gene-major
    return d, s_, l, Xs, Xg, f_mean, f_var, m_mean, m_var, po["jitter"]


TWIN_POST_TOL = {"f32": (5e-4, 2e-5, 5e-4, 2e-5), "f64": (5e-5, 5e-6, 1e-8, 1e-9)}   # f mean, f var, m mean, m var


@pytest.mark.parametrize("which", ["f32", "f64"])
@pytest.mark.parametrize("name", TWIN_CASES)
def test_oracle_posteriors_match_the_gpytorch_twin(name, which):
    c, G, N, X, y, var = _twin(name)
    tol = TWIN_POST_TOL[which]
    for pt in c["points"]:
        d, s_, l, Xs, Xg, f_mean, f_var, m_mean, m_var, jit = _twin_posterior_problem(c, pt, which)
        p = o.Params(d=d, s=s_, b=np.zeros(G), l=l, sigma=0.0, jitter=c["kernel_jitter"])
        m, v = o.latent_predict(p, Xs, X, y, var)                    # var = 1 + 2 * 1e-4 - k^T Sigma^-1 k
        v = v - 2 * c["kernel_jitter"] + 1e-3 + jit                  # twin: K_ff + 1e-3 I (model_alfi.py K_ff), + jitter (:143)
        assert rel(m, f_mean) < tol[0] and rel(v, f_var) < tol[1]
        p2 = o.Params(d=d, s=s_, b=np.zeros(G), l=l, sigma=np.sqrt(c["kernel_jitter"]), jitter=c["kernel_jitter"])
        mm, cov = o.multi_gene_predict(p2, Xg, X, y, var)            # cov = K_tt - ... + 1e-4 I  (K_tt + 1e-4 I: model_alfi.py:294-296)
        assert rel(mm, m_mean) < tol[2] and rel(np.diag(cov) + jit, m_var) < tol[3]                 # + jitter (:107)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["f32", "f64"])
@pytest.mark.parametrize("name", TWIN_CASES)
def test_cuda_posteriors_match_the_gpytorch_twin(cuda, name, which):
    from dis_project_b200 import ops
    c, G, N, X, y, var = _twin(name)
    tol = TWIN_POST_TOL[which]
    kj = c["kernel_jitter"]
    for pt in c["points"]:
        d, s_, l, Xs, Xg, f_mean, f_var, m_mean, m_var, jit = _twin_posterior_problem(c, pt, which)
        theta = np.concatenate([d, s_, np.zeros(G), [l, 0.0]])
        m, v, info = ops.latent_posterior(X, y, var, theta, kj, Xs, G)
        assert int(info.item()) == 0
        assert rel(m.cpu().numpy(), f_mean) < tol[0] and rel(v.cpu().numpy() - 2 * kj + 1e-3 + jit, f_var) < tol[1]
        theta2 = np.concatenate([d, s_, np.zeros(G), [l, np.sqrt(kj)]])
        mm, cov, vv, info2 = ops.gene_posterior(X, y, var, theta2, kj, Xg, G)
        assert int(info2.item()) == 0
        assert rel(mm.cpu().numpy(), m_mean) < tol[2] and rel(vv.cpu().numpy() + jit, m_var) < tol[3]
        # the same through the model class (dis_project_b200.ExactLFM.predict_f / predict_m mirror the twin's methods)
        from dis_project_b200.model import ExactLFM
        T7 = N // G

        class _Arrays:   # what dataset_3d reads of a JaxP53Data: one (times, expressions) entry per gene, the variances
            num_genes, gene_variances = G, var.reshape(G, T7)
            def __len__(self): return G
            def __getitem__(self, i): return np.stack((np.array(c["train_t"])[:T7], y.reshape(G, T7)[i]))

        data = _Arrays()
        mdl = ExactLFM(jitter=kj, data=data, num_genes=G).with_leaves(np.concatenate([d, s_, np.full(G, 0.05), [l, 1.0]]))
        fm, fv = mdl.predict_f(np.array(pt["posterior"]["t_predict"]), data, jitter=jit)
        pm, pv = mdl.predict_m(np.array(pt["posterior"]["t_predict"]), data, jitter=jit)
        assert rel(fm, f_mean) < tol[0] and rel(fv, f_var) < tol[1]
        assert rel(pm.T.reshape(-1), m_mean) < tol[2] and rel(pv.T.reshape(-1), m_var) < tol[3]
