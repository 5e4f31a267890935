"""carma_pack_b200 -- B200-native (sm_100a) CARMA(p,q) Kalman log-likelihood + PT-MCMC hot path.

The GPU path is reached through the C ABI of include/carma_b200.h (libcarma_b200.so, ctypes in
`_lib`) and, for the reference's class surface, through the compiled `_carmcmc` module.  There is
no CPU fallback: importing this package fails when the CUDA library has not been built.
"""
from . import _lib
from ._lib import (CarmaError, Series, MultiSeries, Prior, PTOpts, KIND_CAR1, KIND_CARP, KIND_CARMA, KIND_ZCAR,
                   KIND_ZCARMA, IGNORE_BOUNDS, LOGLIK_ONLY, HESS_OK, HESS_REJECTED, HESS_NONFINITE, HESS_NOT_NEGDEF,
                   HESS_REL_STEP, LAPLACE_OK, LAPLACE_BAD_COV, LAPLACE_NO_WEIGHT, LAPLACE_MAX_DRAWS,
                   model_dim)
from .synth import get_ar_roots, carma_variance, carma_process, car1_process, power_spectrum
from .carma_pack import CarmaModel, CarmaSample, Car1Sample, MCMCSample, SurveySample, LaplaceSample, batched_lbfgs

__all__ = ["CarmaError", "Series", "MultiSeries", "Prior", "PTOpts", "KIND_CAR1", "KIND_CARP", "KIND_CARMA",
           "KIND_ZCAR", "KIND_ZCARMA", "IGNORE_BOUNDS", "LOGLIK_ONLY", "HESS_OK", "HESS_REJECTED", "HESS_NONFINITE",
           "HESS_NOT_NEGDEF", "HESS_REL_STEP", "LAPLACE_OK", "LAPLACE_BAD_COV", "LAPLACE_NO_WEIGHT",
           "LAPLACE_MAX_DRAWS", "model_dim", "get_ar_roots",
           "carma_variance", "carma_process", "car1_process", "power_spectrum", "CarmaModel", "CarmaSample",
           "Car1Sample", "MCMCSample", "SurveySample", "LaplaceSample", "batched_lbfgs"]
