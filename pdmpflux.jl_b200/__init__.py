"""pdmpflux_b200 -- Python host mirror of the PDMPFlux.jl API over libpdmpflux_cuda.so (B200, sm_100a).

Only the grid-based Poisson-thinning hot path is here (SURVEY.md section 8): constructors, sample_skeleton,
sample_from_skeleton, sample, PDMPHistory.  Everything computes on the GPU through the C ABI; there is no CPU
fallback.  Import name: `pdmpflux_b200` (the directory name `pdmpflux.jl_b200` is not a Python identifier;
the shim `pdmpflux_b200.py` at the repository root maps it).
"""
from ._lib import (ArgumentError, CapacityError, ChainError, CompileError, CudaError, DimensionMismatch, UnsupportedError,
                   LIB_PATH, build, lib)
from .device import DeviceChains, device_history_view
from . import dist
from .history import PDMPHistory, PDMPHistoryBatch
from .potentials import (Banana, BananaReadmeScalar, CudaPotential, GaussDense, GaussDiag, GaussEquicorr, GaussStd, LogReg,
                         Potential)
from .sample import (RV_diagnostic, ess_from_chain_means, sample, sample_from_skeleton, sample_skeleton,
                     sample_skeleton_until, sample_skeleton_with_diagnostic, skeleton_moments)
from .samplers import (BPS, BPSAD, AbstractPDMP, Boomerang, BoomerangAD, ForwardECMC, ForwardECMCAD, SpeedUpZigZag,
                       SpeedUpZigZagAD, StickyZigZag, StickyZigZagAD, ZigZag, ZigZagAD)

__all__ = [
    "ZigZag", "ZigZagAD", "BPS", "BPSAD", "ForwardECMC", "ForwardECMCAD", "Boomerang", "BoomerangAD", "StickyZigZag",
    "StickyZigZagAD", "SpeedUpZigZag", "SpeedUpZigZagAD",
    "AbstractPDMP", "sample", "sample_skeleton", "RV_diagnostic", "sample_skeleton_with_diagnostic", "sample_skeleton_until", "CapacityError", "sample_from_skeleton", "skeleton_moments",
    "ess_from_chain_means", "PDMPHistory", "PDMPHistoryBatch", "Potential", "GaussStd", "GaussDiag",
    "GaussEquicorr", "GaussDense", "Banana", "BananaReadmeScalar", "LogReg", "CudaPotential", "ArgumentError", "DimensionMismatch",
    "UnsupportedError", "CudaError", "ChainError", "CompileError", "build", "lib", "LIB_PATH", "DeviceChains",
    "device_history_view", "dist",
]
