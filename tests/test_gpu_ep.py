"""GPU parity for EP binary classification (BASELINE.json config 3) through the C ABI: tau, nu, logZ, class
probabilities at 1e-9 with identical sweep counts (SURVEY.md 8(d)).  The reference has NO test for this path
("parity unpinned"): the oracle is its line-by-line C restatement, cross-checked against a NumPy flavour in tests/."""
import os

import numpy as np
import pytest

import gp_algos_b200 as gp
from oracle import gp_oracle as orc

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RTOL = 1e-9


def close(a, b, rtol=RTOL):
    a, b = np.asarray(a), np.asarray(b)
    return np.all(np.abs(a - b) <= rtol * np.maximum(np.abs(b), np.abs(b).max() * 1e-6))


def test_golden_c3_small():
    g = np.load(os.path.join(G, "c3_small.npz"))
    kf = gp.GaussianRbfKernel(gp.GaussianRbfParams(g["theta"][0], g["theta"][1:-1], g["theta"][-1]))
    K = gp.MatrixUtils.buildKernelMatrix(kf, g["X"])
    site, L = gp.EpParameterEstimator(K, g["targets"], gp.FixedSweeps(5)).estimateSiteParams
    assert close(site.tauSiteParams, g["tau5"]) and close(site.niSiteParams, g["nu5"])
    assert abs(site.marginalLogLikelihood - float(g["logZ5"])) <= RTOL * abs(float(g["logZ5"]))
    assert close(np.diag(L), g["L5_diag"])
    est = gp.EpParameterEstimator(K, g["targets"], gp.AvgBasedStopCriterion(0.01))   # shipped criterion
    site, L = est.estimateSiteParams
    assert est.sweeps == int(g["sweeps"])
    assert close(site.tauSiteParams, g["tau"]) and close(site.niSiteParams, g["nu"])
    assert abs(site.marginalLogLikelihood - float(g["logZ"])) <= RTOL * abs(float(g["logZ"]))
    Ks = gp.MatrixUtils.buildKernelMatrix(kf, g["Xs"], g["X"]); Kss = gp.MatrixUtils.buildKernelMatrix(kf, g["Xs"])
    clf = gp.GpClassifier(gp.AvgBasedStopCriterion(0.01))
    p = clf.classify(gp.AfterEstimationClassifierInput(g["targets"], (site, L), None, K, Ks, Kss))
    assert close(p, g["prob"]) and close(clf.fMean, g["fmean"]) and close(clf.fVariance, g["fvar"])


@pytest.mark.parametrize("n,D,sweeps", [(50, 2, 2), (65, 2, 3), (130, 3, 3), (300, 4, 2)])   # 65, 130: a last block of 1 / 2 sites
def test_ep_vs_literal_oracle(n, D, sweeps):
    X, t, th = orc.make_c3(n=n, D=D, seed=n)
    K = orc.lit_build_kernel_matrix(X, th)
    site, L = gp.EpParameterEstimator(K, t, gp.FixedSweeps(sweeps)).estimateSiteParams
    o = orc.lit_ep_estimate(K, t, fixed_sweeps=sweeps)
    assert close(site.tauSiteParams, o["tau"]) and close(site.niSiteParams, o["nu"])
    assert abs(site.marginalLogLikelihood - o["logZ"]) <= RTOL * abs(o["logZ"])
    assert np.allclose(L, o["L"], rtol=1e-9, atol=1e-12)
    # without the line-break quirk the dropped term reappears (EpParameterEstimator.scala:91-92)
    site2, _ = gp.EpParameterEstimator(K, t, gp.FixedSweeps(sweeps), keep_linebreak_quirk=False).estimateSiteParams
    o2 = orc.lit_ep_estimate(K, t, fixed_sweeps=sweeps, keep_quirk=False)
    assert abs(site2.marginalLogLikelihood - o2["logZ"]) <= RTOL * abs(o2["logZ"])


@pytest.mark.parametrize("n,signal", [(300, 1.0), (1000, 1.0), (200, 40.0)])
def test_site_kernel_variants_agree(n, signal, monkeypatch):
    """The default site kernel (warp-specialised, branch-free scalar update with the erfcx table) against GPK_EP_SITES=4 (the
    reference kernel: libdevice erfc / exp chain, the formulas as written): same site parameters to rounding.  n = 300 ends in
    a ragged block (44 sites); signal = 40 drives |z| past 11.3, the table's libdevice fallback."""
    X, t, th = orc.make_c3(n=n, D=3, seed=n + 7)
    th = th.copy(); th[0] = signal
    K = orc.fast_build_kernel_matrix(X, th)
    res = {}
    for name, sites in (("w", "4"), ("p", None)):
        if sites is None:
            monkeypatch.delenv("GPK_EP_SITES", raising=False)
        else:
            monkeypatch.setenv("GPK_EP_SITES", sites)
        site, L = gp.EpParameterEstimator(K, t, gp.FixedSweeps(3)).estimateSiteParams
        res[name] = (site.tauSiteParams, site.niSiteParams, site.marginalLogLikelihood)
    o = orc.fast_ep_estimate(K, t, fixed_sweeps=3)
    assert np.all(np.isfinite(o["tau"])) and np.all(np.isfinite(res["p"][0]))
    assert close(res["p"][0], res["w"][0], 1e-11) and close(res["p"][1], res["w"][1], 1e-11)
    assert abs(res["p"][2] - res["w"][2]) <= 1e-11 * abs(res["w"][2])
    assert close(res["p"][0], o["tau"]) and close(res["p"][1], o["nu"])


def test_ep_classifier_end_to_end_vs_fast_oracle():
    X, t, th = orc.make_c3(n=700, D=4, seed=3)
    kf = gp.GaussianRbfKernel(gp.GaussianRbfParams(th[0], th[1:-1], th[-1]))
    Xs = np.random.default_rng(1).standard_normal((40, 4))
    K = gp.MatrixUtils.buildKernelMatrix(kf, X); Ks = gp.MatrixUtils.buildKernelMatrix(kf, Xs, X); Kss = gp.MatrixUtils.buildKernelMatrix(kf, Xs)
    clf = gp.GpClassifier(gp.AvgBasedStopCriterion(0.01))
    site, L = clf.trainClassifier(gp.ClassifierInput(K, t))
    o = orc.fast_ep_estimate(K, t, eps=0.01)
    assert close(site.tauSiteParams, o["tau"]) and close(site.niSiteParams, o["nu"])
    assert abs(site.marginalLogLikelihood - o["logZ"]) <= RTOL * abs(o["logZ"])
    p = clf.classify(gp.AfterEstimationClassifierInput(t, (site, L), None, K, Ks, Kss))
    po, fmo, fvo = orc.fast_ep_classify(K, Ks, Kss, o["tau"], o["nu"], o["L"])
    assert close(p, po)
    # MarginalLikelihoodEvaluator.logLikelihoodWithoutGrad (MarginalLikelihoodEvaluator.scala:24-31)
    ev = gp.MarginalLikelihoodEvaluator(gp.AvgBasedStopCriterion(0.01), kf)
    assert abs(ev.logLikelihoodWithoutGrad(X, t, th) - o["logZ"]) <= RTOL * abs(o["logZ"])
    # training accuracy sanity: probabilities on the training inputs side with the labels
    ptrain = clf.classify(gp.AfterEstimationClassifierInput(t, (site, L), None, K, K, K))
    assert np.mean((ptrain > 0.5) == (t > 0)) > 0.85


def test_golden_c3_grad_small():   # MarginalLikelihoodEvaluator.logLikelihood, MarginalLikelihoodEvaluator.scala:33-66
    g = np.load(os.path.join(G, "c3_grad_small.npz"))
    th = g["theta"]
    kf = gp.GaussianRbfKernel(gp.GaussianRbfParams(th[0], th[1:-1], th[-1]))
    ev = gp.MarginalLikelihoodEvaluator(gp.AvgBasedStopCriterion(0.01), kf)
    logz, grad = ev.logLikelihood(g["X"], g["targets"], th)
    assert ev.sweeps == int(g["sweeps"])
    assert abs(logz - float(g["logZ"])) <= RTOL * abs(float(g["logZ"]))
    assert close(grad, g["grad"])
    assert close(ev.siteParams.tauSiteParams, g["tau"]) and close(ev.siteParams.niSiteParams, g["nu"])


@pytest.mark.parametrize("n,D,sweeps,sn", [(60, 2, 2, 0.3), (200, 4, 3, 0.1), (333, 5, 2, 0.0)])
def test_ep_hyperparameter_gradient_vs_literal_oracle(n, D, sweeps, sn):
    X, t, th = orc.make_c3(n=n, D=D, seed=100 + n)
    th = th.copy(); th[-1] = sn
    kf = gp.GaussianRbfKernel(gp.GaussianRbfParams(th[0], th[1:-1], th[-1]))
    ev = gp.MarginalLikelihoodEvaluator(gp.FixedSweeps(sweeps), kf)
    logz, grad = ev.logLikelihood(X, t, th)
    lz_o, g_o, o = orc.lit_ep_loglik_with_derivs(X, t, th, fixed_sweeps=sweeps)
    assert abs(logz - lz_o) <= RTOL * abs(lz_o)
    assert close(grad, g_o)
    # the two-step route of the reference: estimateSiteParams, then logLikelihoodDerivativesAfterHyperParams
    K = gp.MatrixUtils.buildKernelMatrix(kf, X)
    site, L = gp.EpParameterEstimator(K, t, gp.FixedSweeps(sweeps)).estimateSiteParams
    g2 = ev.logLikelihoodDerivativesAfterHyperParams(gp.HyperParameterOptimInput(site, L, K, X), kf)
    assert close(g2, g_o)


def test_ep_gradient_medium_vs_fast_oracle():
    X, t, th = orc.make_c3(n=1100, D=4, seed=5)
    th = th.copy(); th[-1] = 0.1
    kf = gp.GaussianRbfKernel(gp.GaussianRbfParams(th[0], th[1:-1], th[-1]))
    ev = gp.MarginalLikelihoodEvaluator(gp.AvgBasedStopCriterion(0.01), kf)
    logz, grad = ev.logLikelihood(X, t, th)
    K = orc.fast_build_kernel_matrix(X, th)
    o = orc.fast_ep_estimate(K, t, eps=0.01)
    assert ev.sweeps == o["sweeps"]
    assert abs(logz - o["logZ"]) <= RTOL * abs(o["logZ"])
    assert close(grad, orc.fast_ep_loglik_derivs(X, th, K, o["tau"], o["nu"], o["L"]), rtol=1e-8)


def test_ep_requirements():
    with pytest.raises(ValueError):  # require(kernelMatrix.rows == targets.length)
        gp.EpParameterEstimator(np.eye(4), np.ones(3, dtype=np.int32), gp.FixedSweeps(1))
    with pytest.raises(TypeError):
        gp.EpParameterEstimator(np.eye(4), np.ones(4, dtype=np.int32), lambda ctx: True).estimateSiteParams


def test_c3_config_full_size_parity_and_properties():
    """BASELINE.json config 3 at full size (n = 4096, D = 4).  Parity: the committed golden tests/golden/c3_full.npz holds three
    fixed sweeps of the LAPACK-backed oracle on exactly this input (generated once in the build container by
    tests/golden/make_golden.py c3_full -- the CPU oracle needs minutes per sweep); tau, nu, mu, the cavity parameters, diag L and
    log Z must agree to 1e-9.  Then the size-independent properties of a finished EP run."""
    X, t, th = orc.make_c3()
    n = X.shape[0]
    kf = gp.GaussianRbfKernel(gp.GaussianRbfParams(th[0], th[1:-1], th[-1]))
    K = gp.MatrixUtils.buildKernelMatrix(kf, X)
    est = gp.EpParameterEstimator(K, t, gp.FixedSweeps(3))
    site, L = est.estimateSiteParams
    tau, nu = site.tauSiteParams, site.niSiteParams
    assert est.sweeps == 3 and np.all(np.isfinite(tau)) and np.all(tau > 0) and np.all(np.isfinite(nu))
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "c3_full.npz"))
    assert int(gold["n"]) == n and int(gold["sweeps"]) == 3
    assert float(gold["x_checksum"]) == float(X.sum()) and int(gold["t_checksum"]) == int(t.sum())   # same seeded input
    for name, got in (("tau", tau), ("nu", nu), ("mu", est.mu), ("diagL", np.diag(L))):
        want = gold[name]
        assert np.all(np.abs(got - want) <= 1e-9 * np.maximum(np.abs(want), 1e-3 * np.abs(want).max())), name
    assert abs(site.marginalLogLikelihood - float(gold["logZ"])) <= 1e-9 * abs(float(gold["logZ"]))
    st = np.sqrt(tau)
    Bm = np.eye(n) + (st[:, None] * st[None, :]) * K                          # EpParameterEstimator.scala:58
    assert np.linalg.norm(L @ L.T - Bm) <= 8 * n * np.finfo(float).eps * np.linalg.norm(Bm)
    assert np.all(np.triu(L, 1) == 0.0)
    # mu = Sigma nu with Sigma = (K^-1 + S)^-1 = K - K S^1/2 B^-1 S^1/2 K  (:60-61): check (K^-1 + S) mu = nu  <=>  mu + K S mu = K nu
    mu = est.mu
    assert np.linalg.norm(mu + K @ (tau * mu) - K @ nu) <= 1e-8 * np.linalg.norm(K @ nu)
    # a second, identical run is bit-identical (deterministic reductions, fixed stream order)
    site2, _ = gp.EpParameterEstimator(K, t, gp.FixedSweeps(3)).estimateSiteParams
    assert np.array_equal(site2.tauSiteParams, tau) and site2.marginalLogLikelihood == site.marginalLogLikelihood
    p = gp.GpClassifier(gp.FixedSweeps(3)).classify(gp.AfterEstimationClassifierInput(t, (site, L), None, K, K[:64], K[:64, :64]))
    assert np.all((p > 0) & (p < 1)) and np.mean((p > 0.5) == (t[:64] > 0)) > 0.85


# ---- callers of MarginalLikelihoodEvaluator (HyperParamsOptimization.scala, MeshHyperParamsLogLikelihoodEvaluator.scala) ----
def test_classification_hyperparameter_optimisers():
    X, t, th = orc.make_c3(n=180, D=2, seed=31)
    th = np.array([0.8, 2.0, 2.0, 0.2])
    kf = gp.GaussianRbfKernel(gp.GaussianRbfParams(th[0], th[1:-1], th[-1]))
    ev = gp.MarginalLikelihoodEvaluator(gp.FixedSweeps(3), kf)
    ll0, g0 = ev.logLikelihood(X, t, th)
    ctx = gp.ClassifierInput(None, t, kf.hyperParams, X)
    opt = gp.GradientHyperParamsOptimizer(ev, gp.BreezeLbfgsOptimizer(maxIter=6))
    hp = opt.optimizeHyperParams(ctx)
    assert isinstance(hp, gp.GaussianRbfParams) and opt.evaluations >= 2
    # every evaluation the optimiser saw is the oracle's objective: check the returned point
    ll1, g1 = ev.logLikelihood(X, t, hp.toDenseVector)
    lz_o, g_o, _ = orc.lit_ep_loglik_with_derivs(X, t, hp.toDenseVector, fixed_sweeps=3)
    assert abs(ll1 - lz_o) <= RTOL * abs(lz_o) and close(g1, g_o)
    assert ll1 >= ll0                                      # best-seen logic of Optimization.scala:44-55
    cg = gp.ApacheCommonsOptimizer(ev)
    hp2 = cg.optimizeHyperParams(ctx)
    assert cg.evaluations <= 20                            # MaxEval(20), HyperParamsOptimization.scala:121
    assert ev.logLikelihood(X, t, hp2.toDenseVector)[0] >= ll0
    with pytest.raises(LookupError):                       # trainData.get on None (:40)
        opt.optimizeHyperParams(gp.ClassifierInput(None, t, kf.hyperParams, None))


def test_mesh_evaluator_reproduces_the_reference_loop():
    X, t, th = orc.make_c3(n=90, D=1, seed=32)
    kf = gp.GaussianRbfKernel(gp.GaussianRbfParams(1.0, [1.0], 0.1))
    ev = gp.MarginalLikelihoodEvaluator(gp.FixedSweeps(2), kf)
    ranges = [[0.5, 1.0], [0.7, 1.4, 2.1], [0.1]]
    res = gp.MeshHyperParamsLogLikelihoodEvaluator(ev).evaluate(ranges, gp.ClassifierInput(None, t, kf.hyperParams, X))
    # one entry per loop iteration at every level: 2 * (1 + 3 * (1 + 1))
    assert len(res.paramsLikelihood) == 14
    K = orc.lit_build_kernel_matrix
    def lz(p):
        site = orc.lit_ep_estimate(K(X, np.asarray(p)), t, fixed_sweeps=2)
        return site["logZ"]
    # innermost level: stored under (a, b, 0.1), evaluated at the point before its own entry was replaced = (a, b, start) = same
    # middle level: stored under (a, b, start2), evaluated at (a, start1, start2) -- the quirk of :32-38
    p_last, v_last = res.paramsLikelihood[-1]
    assert np.array_equal(p_last, [1.0, 0.7, 0.1])          # outer level, second value
    assert abs(v_last - lz([0.5, 0.7, 0.1])) <= RTOL * abs(v_last)     # ... evaluated at the start point
    p_mid, v_mid = res.paramsLikelihood[3]                   # order: (0.5,0.7,[0.1]) inner, (0.5,0.7) mid, (0.5,1.4,[0.1]) inner, mid...
    assert np.array_equal(res.paramsLikelihood[0][0], [0.5, 0.7, 0.1])
    assert np.array_equal(res.paramsLikelihood[1][0], [0.5, 0.7, 0.1])
    assert np.array_equal(p_mid, [0.5, 1.4, 0.1]) and abs(v_mid - lz([0.5, 0.7, 0.1])) <= RTOL * abs(v_mid)
    assert abs(res.paramsLikelihood[2][1] - lz([0.5, 1.4, 0.1])) <= RTOL * abs(res.paramsLikelihood[2][1])
