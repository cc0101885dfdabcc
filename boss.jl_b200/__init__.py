"""boss_b200 -- B200-native (sm_100a) backend for the GP hot path of soldasim/BOSS.jl.

Layout:
  csrc/      hand-written CUDA kernels + the C ABI (include/boss_b200.h) -> lib/libboss_b200.so
  _lib.py    ctypes binding (no CPU fallback)
  the remaining modules mirror the reference's Julia interfaces for this path (same names, argument
  meaning and error behaviour) on top of the C ABI.
"""
from . import _lib  # noqa: F401  (raises loudly when the CUDA library has not been built)
from .types import (BIParams, BossOptions, BossProblem, Dirac, Domain, ExperimentData, ExprFitness, FixedParams, LinFitness,  # noqa: F401
                    LogNormal, MAPParams, NonlinFitness, Normal, Product, Uniform, generate_LHC, in_bounds, in_domain,
                    mvlognormal)
from .gaussian_process import (DiscreteKernel, ExponentialKernel, GaussianProcess, GaussianProcessParams,  # noqa: F401
                               GaussianProcessPosterior, Matern12Kernel, Matern32Kernel, Matern52Kernel, Parametric,
                               RationalQuadraticKernel, Semiparametric, SemiparametricParams, SqExponentialKernel,
                               data_loglike, data_loglike_and_grad, model_posterior_slice)
from .posterior import DefaultModelPosterior, average_mean, model_posterior  # noqa: F401
from .acquisition import (Acquisition, ExpectedImprovement, best_so_far, construct_acquisition,  # noqa: F401
                          construct_safe_acquisition)
from .acquisition_maximizers import (GridAM, OptimizationAM, SampleOptAM, SamplingAM, SequentialBatchAM,  # noqa: F401
                                     batched_lbfgs_maximize, maximize_acquisition)
from .model_fitters import OptimizationMAP, SampleOptMAP, SamplingMAP, estimate_parameters, model_loglike  # noqa: F401
from .bo import IterLimit, bo  # noqa: F401
from . import parallel  # noqa: F401

Nonparametric = GaussianProcess
