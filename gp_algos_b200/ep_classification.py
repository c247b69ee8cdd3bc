"""Host mirror of gp/classification/{EpParameterEstimator, GpClassifier, MarginalLikelihoodEvaluator}.scala over
libgpk's EP entry points (gpk_ep_fit, gpk_ep_classify, gpk_ep_nll_grad[_batched])."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional

import numpy as np

from . import _lib
from . import batched as _batched
from . import matrix_utils as MU


@dataclass
class SiteParams:
    """EpParameterEstimator.scala:181-182."""
    tauSiteParams: np.ndarray
    niSiteParams: np.ndarray
    marginalLogLikelihood: Optional[float] = None


@dataclass
class AvgBasedStopCriterion:
    """EpParameterEstimator.scala:187-193: stop when abs(avgBetweenSiteParams(old, current)) < eps (spring-context.xml: 0.01)."""
    eps: float = 0.01
    max_sweeps: int = 100


@dataclass
class FixedSweeps:
    """Run exactly `sweeps` EP sweeps (the R prototype's `for (j in 1:5)`, EpParameterEstimator.scala:147)."""
    sweeps: int = 5


def _stop_args(stop):
    if isinstance(stop, FixedSweeps):
        return 0.0, int(stop.sweeps), int(stop.sweeps)
    if isinstance(stop, AvgBasedStopCriterion):
        return float(stop.eps), 0, int(stop.max_sweeps)
    raise TypeError("only AvgBasedStopCriterion / FixedSweeps can be lowered to the GPU path (arbitrary Scala closures cannot)")


class EpParameterEstimator:
    """EpParameterEstimator.scala:11-12: (kernelMatrix, targets, stopCriterion)."""

    def __init__(self, kernelMatrix, targets, stopCriterion, handle=None, keep_linebreak_quirk: bool = True):
        self.K = _lib.fmat(kernelMatrix)
        self.targets = np.ascontiguousarray(targets, dtype=np.int32)
        if self.K.shape[0] != len(self.targets):  # require(...) EpParameterEstimator.scala:20
            raise _lib.IllegalArgumentError(_lib.GPK_EINVAL, "requirement failed")
        self.stop = stopCriterion
        self._handle = handle
        self.keep_quirk = keep_linebreak_quirk
        self.sweeps = None
        self.mu = None
        self.cavity = None

    @property
    def estimateSiteParams(self):
        """-> (SiteParams(tau, nu, Some(logZ)), L)   (EpParameterEstimator.scala:29-69)."""
        h = self._handle or _lib.default_handle()
        n = self.K.shape[0]
        eps, fixed, mx = _stop_args(self.stop)
        tau = np.empty(n); nu = np.empty(n); mu = np.empty(n); ct = np.empty(n); cn = np.empty(n)
        L = np.empty((n, n), order="F")
        logz = C.c_double(); sw = C.c_int()
        h.check(h.lib.gpk_ep_fit(h.h, _lib.ptr(self.K), n, n, self.targets.ctypes.data_as(C.c_void_p), eps, fixed, mx,
                                 int(self.keep_quirk), _lib.ptr(tau), _lib.ptr(nu), _lib.ptr(mu), _lib.ptr(L), n, _lib.ptr(ct),
                                 _lib.ptr(cn), C.addressof(logz), C.addressof(sw)))
        self.sweeps, self.mu, self.cavity = sw.value, mu, (ct, cn)
        return SiteParams(tau, nu, logz.value), L


@dataclass
class ClassifierInput:
    """GpClassifier.scala:63-65."""
    trainKernelMatrix: np.ndarray
    targets: np.ndarray
    initHyperParams: object = None
    trainData: Optional[np.ndarray] = None


@dataclass
class AfterEstimationClassifierInput:
    """GpClassifier.scala:58-61."""
    targets: np.ndarray
    learnParams: Optional[tuple]
    hyperParams: object
    trainKernelMatrix: np.ndarray
    testTrainKernelMatrix: np.ndarray
    testKernelMatrix: np.ndarray


class GpClassifier:
    """GpClassifier.scala:11."""

    def __init__(self, stopCriterion, handle=None):
        self.stopCriterion = stopCriterion
        self._handle = handle

    def trainClassifier(self, classInput: ClassifierInput):
        return EpParameterEstimator(classInput.trainKernelMatrix, classInput.targets, self.stopCriterion, self._handle).estimateSiteParams

    def classify(self, input: AfterEstimationClassifierInput) -> np.ndarray:
        """Class-1 probabilities (GpClassifier.scala:24-47)."""
        h = self._handle or _lib.default_handle()
        site, L = input.learnParams if input.learnParams is not None else self.trainClassifier(
            ClassifierInput(input.trainKernelMatrix, input.targets, input.hyperParams, None))
        K = _lib.fmat(input.trainKernelMatrix); Ks = _lib.fmat(input.testTrainKernelMatrix); L = _lib.fmat(L)
        kss = np.ascontiguousarray(np.diag(np.asarray(input.testKernelMatrix, dtype=np.float64)))
        n, m = K.shape[0], Ks.shape[0]
        tau = np.ascontiguousarray(site.tauSiteParams, dtype=np.float64); nu = np.ascontiguousarray(site.niSiteParams, dtype=np.float64)
        prob = np.empty(m); self.fMean = np.empty(m); self.fVariance = np.empty(m)
        h.check(h.lib.gpk_ep_classify(h.h, _lib.ptr(K), n, n, _lib.ptr(Ks), m, m, _lib.ptr(kss), _lib.ptr(tau), _lib.ptr(nu),
                                      _lib.ptr(L), n, _lib.ptr(prob), _lib.ptr(self.fMean), _lib.ptr(self.fVariance)))
        return prob


@dataclass
class HyperParameterOptimInput:
    """MarginalLikelihoodEvaluator.scala:88-89."""
    siteParams: SiteParams
    lowerTriangular: np.ndarray
    kernelMatrix: np.ndarray
    trainInput: np.ndarray


class MarginalLikelihoodEvaluator:
    """MarginalLikelihoodEvaluator.scala:13 -- K build + EP + logZ (:18-31) and the hyper-parameter gradient (:33-66,
    reproduced as compiled: rMatrix = b b^t, see include/gpk.h gpk_ep_nll_grad)."""

    def __init__(self, stopCriterion, kernelFunc, handle=None, keep_linebreak_quirk: bool = True):
        self.stopCriterion, self.kernelFunc, self._handle = stopCriterion, kernelFunc, handle
        self.keep_quirk = keep_linebreak_quirk
        self.sweeps = None
        self.siteParams = None

    def logLikelihood(self, trainInput, targets, hyperParams):
        """-> (logZ, gradient[hyperParametersNum])   (MarginalLikelihoodEvaluator.scala:33-45), one fused device call."""
        h = self._handle or _lib.default_handle()
        kf = self.kernelFunc.changeHyperParams(hyperParams)
        X = _lib.fmat(trainInput)
        t = np.ascontiguousarray(targets, dtype=np.int32)
        theta = np.ascontiguousarray(kf.theta, dtype=np.float64)
        n, D = X.shape
        if t.shape[0] != n:
            raise _lib.IllegalArgumentError(_lib.GPK_EINVAL, "requirement failed")
        eps, fixed, mx = _stop_args(self.stopCriterion)
        P = kf.hyperParametersNum
        grad = np.empty(P); tau = np.empty(n); nu = np.empty(n)
        logz = C.c_double(); sw = C.c_int()
        h.check(h.lib.gpk_ep_nll_grad(h.h, _lib.ptr(X), n, D, n, _lib.ptr(theta), t.ctypes.data_as(C.c_void_p), eps, fixed, mx,
                                      int(self.keep_quirk), P, C.addressof(logz), _lib.ptr(grad), _lib.ptr(tau), _lib.ptr(nu),
                                      C.addressof(sw)))
        self.sweeps, self.siteParams = sw.value, SiteParams(tau, nu, logz.value)
        return logz.value, grad

    def logLikelihoodDerivativesAfterHyperParams(self, optimInput: "HyperParameterOptimInput", kernelFun) -> np.ndarray:
        """MarginalLikelihoodEvaluator.scala:47-66 from a finished EP run (siteParams, L, K, X)."""
        h = self._handle or _lib.default_handle()
        X = _lib.fmat(optimInput.trainInput); K = _lib.fmat(optimInput.kernelMatrix); L = _lib.fmat(optimInput.lowerTriangular)
        tau = np.ascontiguousarray(optimInput.siteParams.tauSiteParams, dtype=np.float64)
        nu = np.ascontiguousarray(optimInput.siteParams.niSiteParams, dtype=np.float64)
        theta = np.ascontiguousarray(kernelFun.theta, dtype=np.float64)
        n, D = X.shape
        P = kernelFun.hyperParametersNum
        grad = np.empty(P)
        h.check(h.lib.gpk_ep_grad_from_factor(h.h, _lib.ptr(X), n, D, n, _lib.ptr(theta), _lib.ptr(K), n, _lib.ptr(tau), _lib.ptr(nu),
                                              _lib.ptr(L), n, P, _lib.ptr(grad)))
        return grad

    def logLikelihoodWithKernelMatrixPassed(self, kernelMatrix, targets) -> float:
        site, _ = EpParameterEstimator(kernelMatrix, targets, self.stopCriterion, self._handle).estimateSiteParams
        return site.marginalLogLikelihood

    def logLikelihoodWithoutGrad(self, trainInput, targets, hyperParams) -> float:
        kf = self.kernelFunc.changeHyperParams(hyperParams)
        K = MU.buildKernelMatrix(kf, trainInput, handle=self._handle)
        return self.logLikelihoodWithKernelMatrixPassed(K, targets)


# ---- gp/classification/HyperParamsOptimization.scala: the callers of MarginalLikelihoodEvaluator.logLikelihood -----------
class GradientHyperParamsOptimizer:
    """HyperParamsOptimization.scala:31-55: maximise the EP log marginal likelihood with a GradientBasedOptimizer
    (optimization/Optimization.scala, `BreezeLbfgsOptimizer` in the shipped wiring).  Host control flow only: every
    objective/gradient evaluation is one fused gpk_ep_nll_grad call (K build + EP sweeps + gradient on the device)."""

    def __init__(self, marginalLikelihoodEvaluator: MarginalLikelihoodEvaluator, gradOptimizer):
        self.marginalLikelihoodEvaluator, self.gradOptimizer = marginalLikelihoodEvaluator, gradOptimizer
        self.evaluations = 0

    def optimizeHyperParams(self, optimizationInput: ClassifierInput):
        if optimizationInput.trainData is None:
            raise LookupError("None.get")                                   # optimizationInput.trainData.get (:40)
        targets = optimizationInput.targets
        init = optimizationInput.initHyperParams

        def funcWithGradient(hyperParams):
            ll, der = self.marginalLikelihoodEvaluator.logLikelihood(optimizationInput.trainData, targets, np.asarray(hyperParams))
            assert len(hyperParams) == len(der)                             # :43
            self.evaluations += 1
            return ll, der

        optimized = self.gradOptimizer.maximize(funcWithGradient, np.asarray(init.toDenseVector, dtype=np.float64))
        return init.fromDenseVector(np.asarray(optimized, dtype=np.float64))


class ApacheCommonsOptimizer:
    """HyperParamsOptimization.scala:57-136: commons-math3 NonLinearConjugateGradientOptimizer(POLAK_RIBIERE), stopped after 5
    iterations (IterationLimitConvergenceChecker), MaxIter(10), MaxEval(20), GoalType.MAXIMIZE, with the reference's
    value/gradient cache per point (:66-110).  commons-math 3.2 is un-vendored third-party code whose line search no reference
    test pins; SciPy's Polak-Ribiere CG with the same iteration cap stands in, the evaluation cap and the cache are reproduced."""

    def __init__(self, marginalLikelihoodEvaluator: MarginalLikelihoodEvaluator, iterationLimit: int = 5, maxEval: int = 20):
        self.marginalLikelihoodEvaluator = marginalLikelihoodEvaluator
        self.iterationLimit, self.maxEval = iterationLimit, maxEval
        self.evaluations = 0

    def optimizeHyperParams(self, optimizationInput: ClassifierInput):
        from scipy.optimize import minimize as sp_minimize
        if optimizationInput.trainData is None:
            raise LookupError("None.get")
        init = optimizationInput.initHyperParams
        cache = {}
        best = {"x": np.asarray(init.toDenseVector, dtype=np.float64), "v": -np.inf}

        class _TooManyEvaluations(Exception):                                # org.apache.commons.math3.exception.TooManyEvaluationsException
            pass

        def value_and_gradient(p):
            key = tuple(np.asarray(p, dtype=np.float64))
            if key not in cache:                                             # pointGradientMapping (:66-110)
                if self.evaluations >= self.maxEval:
                    raise _TooManyEvaluations()
                ll, g = self.marginalLikelihoodEvaluator.logLikelihood(optimizationInput.trainData, optimizationInput.targets,
                                                                       np.asarray(p, dtype=np.float64))
                self.evaluations += 1
                cache[key] = (ll, np.asarray(g, dtype=np.float64))
                if ll > best["v"]:
                    best["x"], best["v"] = np.asarray(p, dtype=np.float64).copy(), ll
            return cache[key]

        try:
            res = sp_minimize(lambda p: -value_and_gradient(p)[0], best["x"].copy(), jac=lambda p: -value_and_gradient(p)[1],
                              method="CG", options={"maxiter": self.iterationLimit})
            point = res.x if -res.fun >= best["v"] else best["x"]
        except _TooManyEvaluations:
            point = best["x"]
        return init.fromDenseVector(np.asarray(point, dtype=np.float64))


def log_likelihood_batched(X, targets, thetas, stopCriterion, nparams: Optional[int] = None, keep_linebreak_quirk: bool = True,
                           handle=None):
    """B evaluations of MarginalLikelihoodEvaluator.logLikelihood (MarginalLikelihoodEvaluator.scala:33-66) of one size n in one
    call (gpk_ep_nll_grad_batched): every problem runs EP to its own stop, all sweeps together on the device.
    X: (n, D) shared or (B, n, D); targets: (n,) shared or (B, n); thetas: (B, P) in the handle's kernel family.
    Returns (logZ[B], grad[B, nparams], sweeps[B], info[B]); a problem with info != 0 (not positive definite) has NaN logZ and
    gradient, the others are valid."""
    h = handle or _lib.default_handle()
    thetas = np.ascontiguousarray(np.atleast_2d(thetas), dtype=np.float64)
    B = thetas.shape[0]
    Xb, strideX, n, D = _batched._stack_problems(X, B)
    t = np.ascontiguousarray(targets, dtype=np.int32)
    if t.ndim == 1:
        strideT = 0
    elif t.ndim == 2 and t.shape[0] == B:
        strideT = n
    else:
        raise _lib.IllegalArgumentError(_lib.GPK_EINVAL, "targets must be (n,) or (B, n)")
    P = h.lib.gpk_theta_length(h.h, D)
    if t.shape[-1] != n or thetas.shape[1] != P:
        raise _lib.IllegalArgumentError(_lib.GPK_EINVAL, "requirement failed: shapes of X, targets and hyper-parameters disagree")
    nparams = P if nparams is None else int(nparams)
    eps, fixed, mx = _stop_args(stopCriterion)
    logz = np.empty(B); grad = np.zeros((B, max(nparams, 1))); sweeps = np.zeros(B, dtype=np.int32)
    info = np.zeros(B, dtype=np.int32)
    rc = h.lib.gpk_ep_nll_grad_batched(h.h, B, _lib.ptr(Xb), n, D, n, strideX, _lib.ptr(thetas), _lib.ptr(t), strideT, eps, fixed, mx,
                                       int(keep_linebreak_quirk), nparams, _lib.ptr(logz), _lib.ptr(grad), None, None,
                                       _lib.ptr(sweeps), _lib.ptr(info))
    if rc != _lib.GPK_ENOTPD:
        h.check(rc)
    return logz, grad[:, :nparams], sweeps, info


def obtain_optimal_ep_hyper_params_multistart(trainData, targets, initThetas, stopCriterion, maxIter: int = 20, handle=None):
    """GradientHyperParamsOptimizer (HyperParamsOptimization.scala:31-55) from R start points at once: the restarts share the
    training set and every lockstep round of batched.LockstepLbfgs is ONE gpk_ep_nll_grad_batched call.  The classification
    twin of batched.obtain_optimal_hyper_params_multistart.  Returns (thetas[R, P], logZ[R]) -- the best-seen point and value
    of every restart; a restart that never had a positive definite evaluation comes back as its start point with logZ = -inf."""
    X = np.asarray(trainData, dtype=np.float64)
    t = np.ascontiguousarray(targets, dtype=np.int32)
    init = np.atleast_2d(np.asarray(initThetas, dtype=np.float64))

    def objective(points, which):
        logz, grad, _, info = log_likelihood_batched(X, t, points, stopCriterion, handle=handle)
        return np.where(info == 0, logz, -np.inf), grad

    return _batched.LockstepLbfgs(maxIter=maxIter).maximize(objective, init)


class HyperParamsMeshValues:
    """MeshHyperParamsLogLikelihoodEvaluator.scala:51-90 (the Scala map is keyed by array identity; a list of pairs keeps
    every entry the same way)."""

    def __init__(self):
        self.paramsLikelihood = []

    def addResult(self, params, logLikelihood: float):
        self.paramsLikelihood.append((np.array(params, dtype=np.float64), float(logLikelihood)))

    def getLikelihood(self, params):
        for p, v in self.paramsLikelihood:
            if p is params:
                return v
        return None

    def writeToFile(self, fileName: str):
        with open(fileName, "w") as f:
            for p, v in self.paramsLikelihood:
                f.write("".join(f"{x}\t" for x in p) + f"{v}\n")


class MeshHyperParamsLogLikelihoodEvaluator:
    """MeshHyperParamsLogLikelihoodEvaluator.scala:12-45: EP log marginal likelihood on a mesh of hyper-parameter values.  As
    written (:32-38) the likelihood is evaluated at `currentHyperParams` -- the point BEFORE the entry of this recursion level
    is replaced -- and stored under the replaced copy; reproduced."""

    def __init__(self, likelihoodEvaluator: MarginalLikelihoodEvaluator):
        self.likelihoodEvaluator = likelihoodEvaluator

    def evaluate(self, hyperParamsRanges, classificationContext: ClassifierInput) -> HyperParamsMeshValues:
        init = np.array([r[0] for r in hyperParamsRanges], dtype=np.float64)     # hyperParamsRanges.map(_.start)
        result = HyperParamsMeshValues()
        self._rec(init, hyperParamsRanges, 0, classificationContext, result)
        return result

    def _rec(self, current, allRanges, rangeIndex, ctx, result):
        for hyperParam in allRanges[rangeIndex]:
            copied = current.copy()
            copied[rangeIndex] = hyperParam
            if rangeIndex + 1 < len(allRanges):
                self._rec(copied, allRanges, rangeIndex + 1, ctx, result)
            likelihood = self.likelihoodEvaluator.logLikelihoodWithoutGrad(ctx.trainData, ctx.targets, current)
            result.addResult(copied, likelihood)
