"""Device potential descriptors: the second positional argument of the sampler constructors.

The reference takes a Julia closure (`grad U`, or `U` for the *AD constructors, ADBackend.jl:30-142); an
arbitrary closure cannot run on the device, so a descriptor names one of the hand-written device plugins
(pdmpflux.jl_b200/csrc/potentials.cuh) and carries its parameters.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib

GAUSS_STD, GAUSS_DIAG, GAUSS_EQUICORR, BANANA, BANANA_README_SCALAR, LOGREG, SOURCE, GAUSS_DENSE = range(8)


class Potential:
    kind = None

    def params(self, dim):
        return np.zeros(0)

    def _create(self, dim):
        p = np.ascontiguousarray(self.params(dim), dtype=np.float64)
        h = C.c_void_p()
        _lib.check(_lib.lib().pdmpflux_potential_create(self.kind, int(dim), p.ctypes.data if p.size else None,
                                                        p.size, C.byref(h)))
        return h


class GaussStd(Potential):
    """U(x) = |x|^2 / 2 (README.md:36-38)."""
    kind = GAUSS_STD


class GaussDiag(Potential):
    """U(x) = sum_i p_i x_i^2 / 2."""
    kind = GAUSS_DIAG

    def __init__(self, precisions):
        self.p = np.asarray(precisions, dtype=np.float64)

    def params(self, dim):
        if self.p.shape != (dim,):
            raise _lib.DimensionMismatch(f"GaussDiag has {self.p.size} precisions but dim = {dim}")
        return self.p


class GaussEquicorr(Potential):
    """'Slanted' Gaussian: Sigma = (1 - rho) I + rho 1 1^T (SURVEY.md 8d, config C3)."""
    kind = GAUSS_EQUICORR

    def __init__(self, rho):
        self.rho = float(rho)

    def params(self, dim):
        return np.array([self.rho])


class GaussDense(Potential):
    """U(x) = (x - mean)' P (x - mean) / 2 with a dense symmetric positive-definite precision matrix P (d <= 2048):
    a Gaussian with covariance inv(P).  Runs on the fast-path kernels of ZigZag (grid_size=0, or a vectorised grid bound
    with an exact AD_backend) and BPS (every configuration); other samplers and options raise UnsupportedError when the
    sampler is built.  The library checks that P is finite, symmetric (to 1e-12 max|P|; it uses (P + P')/2) and positive
    definite.  RV_diagnostic does not run it."""
    kind = GAUSS_DENSE

    def __init__(self, precision, mean=None):
        self.P = np.asarray(precision, dtype=np.float64)
        if self.P.ndim != 2 or self.P.shape[0] != self.P.shape[1]:
            raise _lib.ArgumentError(f"GaussDense needs a square precision matrix, got shape {self.P.shape}")
        self.mean = np.zeros(self.P.shape[0]) if mean is None else np.asarray(mean, dtype=np.float64)

    def params(self, dim):
        if self.P.shape != (dim, dim) or self.mean.shape != (dim,):
            raise _lib.DimensionMismatch(f"GaussDense has a {self.P.shape} precision and a {self.mean.shape} mean but dim = {dim}")
        return np.concatenate([self.P.ravel(), self.mean])


class Banana(Potential):
    """U = (x1^2 + (x2 - x1^2 + 1)^2 + sum_{i>=3} x_i^2) / 2 (test/test_config.jl:33-36)."""
    kind = BANANA


class BananaReadmeScalar(Potential):
    """README.md:62-65 verbatim: the manual 'gradient' returns a scalar broadcast to every coordinate.
    Not a gradient field; chains can drift to a region with zero rate and never produce another event
    (the library then reports STEP_LIMIT instead of hanging like the reference would)."""
    kind = BANANA_README_SCALAR


class LogReg(Potential):
    """Bayesian logistic regression posterior, prior N(0, sigma0^2 I) (BASELINE.json config 4)."""
    kind = LOGREG

    def __init__(self, X, y, sigma0=10.0):
        self.X = np.ascontiguousarray(X, dtype=np.float64)
        self.y = np.ascontiguousarray(y, dtype=np.float64)
        self.sigma0 = float(sigma0)

    def params(self, dim):
        n, d = self.X.shape
        if d != dim or self.y.shape != (n,):
            raise _lib.DimensionMismatch("LogReg design matrix does not match dim")
        return np.concatenate([[float(n), self.sigma0], self.X.ravel(), self.y])


class CudaPotential(Potential):
    """A potential written in CUDA C++: `source` defines `struct UserPotential` with the members of the built-in
    plugins (K linear functionals, accum, grad, eval; see include/pdmpflux_cuda.h or INTEGRATION.md), and `params`
    becomes `pp.vec[0 .. pp.n - 1]` on the device.  The source is compiled at run time with NVRTC: a contract check
    when each sampler is built (CompileError carries the compiler log) and the sampler's kernels right after it.
    Compiled kernels are cached per process by source, so samplers that only change `params` do not compile again.

    Optional members declare the line model of the built-in plugins: `static constexpr bool affine` (constant Hessian
    beyond the first `special` coordinates), `static constexpr int special` (coordinates that are their own
    functionals) and the split line sums `eval_local` / `line_corr`.  A declared potential runs on the fast-path kernels
    of Zig-Zag, BPS and ForwardECMC (Boomerang keeps the generic kernel); without them every sampler runs the generic
    kernel.  RV_diagnostic does not run a CudaPotential (the contract has no U value).

    `accum` must be linear in x_i, and a declared line model must hold exactly; the library can check neither, and a
    wrong declaration samples the wrong target."""
    kind = SOURCE

    def __init__(self, source, params=()):
        if not isinstance(source, str):
            raise TypeError("CudaPotential source must be a str of CUDA C++")
        self.source = source
        self.p = np.ascontiguousarray(params, dtype=np.float64).ravel()

    def params(self, dim):
        return self.p

    def _create(self, dim):
        h = C.c_void_p()
        _lib.check(_lib.lib().pdmpflux_potential_create_source(int(dim), self.source.encode(),
                                                               self.p.ctypes.data if self.p.size else None,
                                                               self.p.size, C.byref(h)))
        return h
