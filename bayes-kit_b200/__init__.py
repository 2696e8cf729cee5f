"""bayes_kit_b200 -- B200-native (sm_100a) drop-in for bayes-kit's data-parallel
sampling hot path: many independent chains / particles advanced in lockstep by
hand-written CUDA kernels behind bayes-kit's own API surface.

Same names as ``bayes_kit/__init__.py:1-30``; models are device plugins
(``bayes_kit_b200.models``), chain state lives in torch CUDA tensors, and every
kernel is reached through the C ABI of ``include/bk.h`` (ctypes).  There is no
CPU fallback.
"""
from . import dist, models, peer
from .autocorr import autocorr
from .drghmc import DrGhmcDiag
from .ensemble import Stretcher
from .ess import ess, ess_imse, ess_ipse
from .hmc import HMCDiag
from .iat import iat, iat_imse, iat_ipse
from .mala import MALA
from .metropolis import (CudaProposal, GaussianRW, Metropolis, MetropolisHastings, metropolis_accept_test,
                         metropolis_hastings_accept_test)
from .models import Binomial, CudaModel, CudaPriorLikModel, DensePrecGauss, DiagGauss, GaussPriorLik, HierLogReg, IsoGauss, StdNormal
from .rhat import (chain_moments, rank_chains, rank_normalize_chains, rank_normalized_rhat, rhat,
                   split_chains, split_rhat)
from .smc import TemperedLikelihoodSMC, hmc_kernel, mala_kernel, metropolis_kernel, proposal_kernel

__all__ = [
    "DrGhmcDiag", "HMCDiag", "MALA", "Metropolis", "MetropolisHastings", "TemperedLikelihoodSMC",
    "Stretcher", "ess", "ess_imse", "ess_ipse", "iat", "iat_imse", "iat_ipse", "rhat", "autocorr",
    # device-side additions
    "GaussianRW", "metropolis_kernel", "mala_kernel", "hmc_kernel", "models", "dist", "peer", "Binomial", "IsoGauss", "StdNormal", "DiagGauss", "CudaModel", "CudaPriorLikModel",
    "CudaProposal", "proposal_kernel",
    "DensePrecGauss", "GaussPriorLik", "HierLogReg", "chain_moments",
    # rhat.py's split / rank-normalised family (not re-exported by the reference's __init__)
    "split_chains", "split_rhat", "rank_chains", "rank_normalize_chains", "rank_normalized_rhat",
]
