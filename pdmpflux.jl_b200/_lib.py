"""ctypes binding of libpdmpflux_cuda.so (include/pdmpflux_cuda.h).

This is the Python stand-in for the Julia `ccall` glue (julia/PDMPFluxCUDA.jl): Julia is not installed in
this image, so the host side above the C ABI is written in Python.  There is NO CPU fallback: if the shared
library is missing or fails to load, importing the package's compute entry points raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
# PDMPFLUX_CUDA_LIB points at another build of the same library (A/B experiments); the default is the in-tree build
LIB_PATH = os.environ.get("PDMPFLUX_CUDA_LIB") or os.path.join(_HERE, "lib", "libpdmpflux_cuda.so")

OK, ERR_ARGUMENT, ERR_DIMENSION_MISMATCH, ERR_UNSUPPORTED, ERR_CUDA, ERR_CHAIN, ERR_CAPACITY, ERR_COMPILE = 0, -1, -2, -3, -4, -5, -6, -7


class ArgumentError(ValueError):
    """Julia `ArgumentError` (e.g. ZigZagSamplers.jl:62-68, sample.jl:262-264, :476-478)."""


class DimensionMismatch(ValueError):
    """Julia `DimensionMismatch` (AbstractPDMP.jl:96-98)."""


class UnsupportedError(NotImplementedError):
    """Requested sampler/potential/option is outside the device path; there is no CPU fallback."""


class CudaError(RuntimeError):
    pass


class CompileError(ValueError):
    """The CUDA source of a CudaPotential did not compile; the message is the NVRTC log (lines of the user's text
    appear as `user_potential(<line>)`)."""


class CapacityError(RuntimeError):
    """Time-horizon variant: a chain needs more history columns than the capacity it was given."""


class ChainError(RuntimeError):
    """At least one chain stopped (tape exhausted, Categorical would throw, step limit)."""

    def __init__(self, msg, status=None):
        super().__init__(msg)
        self.status = status


class Config(C.Structure):
    _fields_ = [
        ("grid_size", C.c_int32), ("vectorized_bound", C.c_int32), ("signed_bound", C.c_int32),
        ("adaptive", C.c_int32), ("deriv_mode", C.c_int32), ("gaussian_velocity", C.c_int32),
        ("ran_p", C.c_int32), ("switch_", C.c_int32), ("positive", C.c_int32), ("max_steps", C.c_int32),
        ("tmax", C.c_double), ("refresh_rate", C.c_double), ("mix_p", C.c_double), ("speed_factor", C.c_double),
    ]


class Tape(C.Structure):
    _fields_ = [("E", C.c_void_p), ("U", C.c_void_p), ("N", C.c_void_p),
                ("nE", C.c_int64), ("nU", C.c_int64), ("nN", C.c_int64), ("on_device", C.c_int32)]


class History(C.Structure):
    _fields_ = [("X", C.c_void_p), ("V", C.c_void_p), ("t", C.c_void_p), ("horizon", C.c_void_p),
                ("ar", C.c_void_p), ("error_value_ar", C.c_void_p), ("errored_bound", C.c_void_p),
                ("rejected", C.c_void_p), ("hitting_horizon", C.c_void_p), ("status", C.c_void_p),
                ("tape_pos", C.c_void_p), ("counters", C.c_void_p), ("n_cols", C.c_int64),
                ("on_device", C.c_int32), ("is_active", C.c_void_p)]


# every symbol include/pdmpflux_cuda.h declares: (restype, argtypes)
SIGNATURES = {
    "pdmpflux_version": (C.c_int, []),
    "pdmpflux_last_error": (C.c_char_p, []),
    "pdmpflux_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "pdmpflux_set_device": (C.c_int, [C.c_int]),
    "pdmpflux_potential_create": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_int64, C.POINTER(C.c_void_p)]),
    "pdmpflux_potential_create_source": (C.c_int, [C.c_int, C.c_char_p, C.c_void_p, C.c_int64, C.POINTER(C.c_void_p)]),
    "pdmpflux_potential_destroy": (C.c_int, [C.c_void_p]),
    "pdmpflux_sampler_create": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "pdmpflux_sampler_create_sticky": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(Config), C.c_void_p, C.POINTER(C.c_void_p)]),
    "pdmpflux_sampler_destroy": (C.c_int, [C.c_void_p]),
    "pdmpflux_sampler_release_workspace": (C.c_int, [C.c_void_p]),
    "pdmpflux_sampler_get_config": (C.c_int, [C.c_void_p, C.POINTER(Config)]),
    "pdmpflux_sample_skeleton": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_uint64,
                                           C.c_int64, C.POINTER(Tape), C.POINTER(History), C.c_void_p]),
    "pdmpflux_sample_skeleton_resume": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p,
                                                  C.c_void_p, C.c_void_p, C.c_int64, C.c_uint64, C.c_int64,
                                                  C.POINTER(Tape), C.POINTER(History), C.c_void_p]),
    "pdmpflux_sample_skeleton_until": (C.c_int, [C.c_void_p, C.c_int64, C.c_double, C.c_int64, C.c_void_p, C.c_void_p,
                                                 C.c_uint64, C.c_int64, C.POINTER(Tape), C.POINTER(History), C.c_void_p,
                                                 C.c_void_p]),
    "pdmpflux_chains_enable_moments": (C.c_int, [C.c_void_p]),
    "pdmpflux_chains_get_moments": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]),
    "pdmpflux_chains_set_stop_time": (C.c_int, [C.c_void_p, C.c_double]),
    "pdmpflux_chains_get_ncols": (C.c_int, [C.c_void_p, C.c_void_p]),
    "pdmpflux_chains_set_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32]),
    "pdmpflux_chains_get_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]),
    "pdmpflux_chains_create": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.c_uint64,
                                         C.c_int64, C.POINTER(Tape), C.POINTER(C.c_void_p)]),
    "pdmpflux_chains_advance": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(History), C.c_int64, C.c_void_p]),
    "pdmpflux_chains_record": (C.c_int, [C.c_void_p, C.POINTER(History), C.c_int64, C.c_void_p]),
    "pdmpflux_chains_status": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pdmpflux_chains_destroy": (C.c_int, [C.c_void_p]),
    "pdmpflux_sample_from_skeleton": (C.c_int, [C.c_int, C.c_int, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p,
                                                C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "pdmpflux_sample_from_skeleton_sticky": (C.c_int, [C.c_int, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                                       C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "pdmpflux_sample_from_skeleton_dt": (C.c_int, [C.c_int, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                                   C.c_void_p, C.c_void_p, C.c_double, C.c_int64, C.c_int32, C.c_void_p,
                                                   C.c_int32, C.c_void_p]),
    "pdmpflux_skeleton_moments": (C.c_int, [C.c_int, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                            C.c_void_p]),
    "pdmpflux_moments_reduce": (C.c_int, [C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                          C.c_void_p]),
    "pdmpflux_comm_unique_id": (C.c_int, [C.c_void_p, C.c_size_t]),
    "pdmpflux_comm_create": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "pdmpflux_comm_destroy": (C.c_int, [C.c_void_p]),
    "pdmpflux_moments_allreduce": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "pdmpflux_rv_diagnostic": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_int64,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "pdmpflux_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_size_t]),
    "pdmpflux_host_free": (C.c_int, [C.c_void_p]),
    "pdmpflux_launch_count": (C.c_int64, []),
    "pdmpflux_jit_compile_count": (C.c_int64, []),
    "pdmpflux_last_transfer_bytes": (C.c_int, [C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
}

_lib = None


def build(verbose=False):
    """Compile libpdmpflux_cuda.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", os.path.join(_HERE, "csrc"), "-j8"]
    subprocess.check_call(cmd, stdout=None if verbose else subprocess.DEVNULL)
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C pdmpflux.jl_b200/csrc`).  pdmpflux_b200 has no CPU fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(l, name)  # AttributeError if the library does not export a declared symbol
            f.restype, f.argtypes = res, args
        if l.pdmpflux_version() < 200:
            raise ImportError("libpdmpflux_cuda.so is older than this binding")
        _lib = l
    return _lib


def check(rc, status=None):
    if rc == OK:
        return
    msg = lib().pdmpflux_last_error().decode("utf-8", "replace")
    if rc == ERR_ARGUMENT:
        raise ArgumentError(msg)
    if rc == ERR_DIMENSION_MISMATCH:
        raise DimensionMismatch(msg)
    if rc == ERR_UNSUPPORTED:
        raise UnsupportedError(msg)
    if rc == ERR_CHAIN:
        raise ChainError(msg, status)
    if rc == ERR_CAPACITY:
        raise CapacityError(msg)
    if rc == ERR_COMPILE:
        raise CompileError(msg)
    raise CudaError(msg)
