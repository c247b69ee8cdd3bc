"""gp_algos_b200 -- B200-native (sm_100a) drop-in for the dense-GP hot path of astroHaoPeng/gp_algos.

The numeric work lives in ``libgpk.so`` (hand-written CUDA, C ABI in include/gpk.h).  This package is
the host-side mirror of the reference's Scala interface for that path (same names, argument meaning
and error behaviour), used by the parity tests and the benchmark:

    utils.KernelRequisites  ->  gp_algos_b200.kernel_requisites  (GaussianRbfParams, GaussianRbfKernel)
    gp.regression.Co2Prediction -> gp_algos_b200.co2_prediction  (Co2HyperParams, Co2Kernel: the second closed-form kernel)
    utils.MatrixUtils       ->  gp_algos_b200.matrix_utils       (buildKernelMatrix, forwardSolve, ...)
    gp.regression.GpPredictor -> gp_algos_b200.gp_predictor      (GpPredictor, PredictionInput, ...)
    gp.classification.*      ->  gp_algos_b200.ep_classification (EpParameterEstimator, GpClassifier, ...)
    dynamicalsystems.filtering.GPUnscentedKalmanFilter -> gp_algos_b200.gp_ukf (the whole filter run is one device call)
    gp.optimization.GPOptimizer -> gp_algos_b200.gp_optimizer    (GP-UCB inner loop on a resident model)
    (batched independent GPs and their rank sharding: gp_algos_b200.batched;
     one large GP over a 2-D block-cyclic GPU grid: gp_algos_b200.distributed)

There is no CPU fallback: importing works anywhere, but every numeric call raises if libgpk.so or a
CUDA device is missing.
"""
import os as _os

# libgpk runs its look-ahead drivers and batch groups on up to ~20 CUDA streams per handle; with the default of 8 hardware work
# queues several streams share a queue and serialise falsely (measured: 3 / 4 batch groups 3.73 / 3.70 ms -> 3.38 ms for 64 problems
# of n = 1024, profiles/r02_c4_maxconn.log).  The variable is read when the CUDA context is created, so it is set at import time
# unless the host application already chose a value.
_os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

from .kernel_requisites import GaussianRbfKernel, GaussianRbfParams  # noqa: F401,E402
from .co2_prediction import Co2HyperParams, Co2Kernel, co2DataToYearWithValue  # noqa: F401
from .gp_predictor import GpPredictor, PredictionInput, PredictionTrainingInput, GaussianDistribution  # noqa: F401
from . import matrix_utils as MatrixUtils  # noqa: F401
from . import batched  # noqa: F401
from .ep_classification import (EpParameterEstimator, GpClassifier, MarginalLikelihoodEvaluator, SiteParams,  # noqa: F401
                                AvgBasedStopCriterion, FixedSweeps, ClassifierInput, AfterEstimationClassifierInput,
                                HyperParameterOptimInput, GradientHyperParamsOptimizer, ApacheCommonsOptimizer,
                                MeshHyperParamsLogLikelihoodEvaluator, HyperParamsMeshValues, log_likelihood_batched,
                                obtain_optimal_ep_hyper_params_multistart)
from .gp_optimizer import GPOptimizer, GPOInput, BreezeLbfgsOptimizer, ucb_with_gradient  # noqa: F401
from .gp_ukf import (GPUnscentedKalmanFilter, UnscentedTransformParams, UnscentedFilteringInput, SsmModel,  # noqa: F401
                     FilteringOutput)
from ._lib import GpkError, NotPositiveDefiniteError, MatrixNotSymmetricError, lib_path  # noqa: F401

__all__ = ["GaussianRbfKernel", "GaussianRbfParams", "Co2Kernel", "Co2HyperParams", "GpPredictor", "PredictionInput", "PredictionTrainingInput",
           "GaussianDistribution", "MatrixUtils", "GpkError", "NotPositiveDefiniteError", "MatrixNotSymmetricError"]
