"""differentialevolutionmcmc.jl_b200 -- B200-native population step of DifferentialEvolutionMCMC.jl.

Holds only what the hot path needs: csrc/ (CUDA kernels + the C ABI, built into
libdemcmc_b200.so) and the host-side mirror of the reference's interface for that path
(DE, DEModel, GPULoglike, sample).  Import it as `demcmc_b200` through the loader at the repo
root (the directory name carries a dot, so it is not importable by its own name).
"""
from . import _ffi  # noqa: F401
from .handle import (Handle, comm_unique_id, copy_peak, fp64_peak, fp64_peaks, op_accept, op_de_proposal, op_project,  # noqa: F401
                     op_reset, op_select, op_snooker)
from .api import (DE, DEModel, GPUDEModel, Beta, Chains, Flat, GPULoglike, GPUPrior, HalfCauchy, MCMCThreads, Normal,  # noqa: F401
                  NormalRef, Particle, Uniform, compute_posterior, evaluate_fun, fixed_gamma, get_optimal, maximize,
                  mh_update, minimize, optimize, pointwise_loglikelihoods, loo, power_posterior, random_gamma, resample, sample, variable_gamma)
