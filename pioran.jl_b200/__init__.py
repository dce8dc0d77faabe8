"""pioran.jl_b200 — B200 (sm_100a) backend of Pioran.jl's celerite likelihood path.

The directory name carries a dot, so import it through the repo-root shim:  `import pioran_b200`.
Contents: csrc/ (CUDA kernels + C ABI, built into libpioran_b200.so), backend.py (ctypes handle),
api.py (mirror of the reference's Julia interface), build.py (nvcc recipe)."""
from . import _lib, api, backend, build, parallel, sampler  # noqa: F401
from .api import (QPO, SumOfPowerSpectralDensity, separate_psd, convert_feature, get_covariance_from_psd, BatchedCARMALikelihood, BatchedLikelihood, CARMA, Celerite, CustomMean, carma_celerite_coefs, celerite_repr, quad2roots, roots2coeffs, DoubleBendingPowerLaw, Exp, ScalableGP, SHO,  # noqa: F401
                  SingleBendingPowerLaw, SumOfCelerite, approx, celerite_coefs, log_likelihood,
                  log_likelihood_direct, logpdf, mean, mean_and_var, posterior, predict, predict_var, rand, simulate,
                  std, var, PosteriorGP)
from .backend import Context, get_context, make_spec  # noqa: F401
from ._lib import ApproxSpec, PioranError  # noqa: F401
