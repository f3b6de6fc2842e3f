"""Source potentials (CudaPotential) without a GPU: the user source is compiled at construction, so contract errors,
the per-sampler kernel compiles and the compile cache are all observable on a machine with no device."""
import numpy as np
import pytest

import pdmpflux_b200 as p

# Pot<PDMPFLUX_BANANA> (csrc/potentials.cuh) restated as a user potential: no parameters
BANANA_SRC = r"""
struct UserPotential {
    static constexpr int K = 2;
    __device__ static void accum(const pdmpflux::PotParams&, int i, double xi, double* acc) {
        if (i == 0) acc[0] += xi;
        if (i == 1) acc[1] += xi;
    }
    __device__ static double grad(const pdmpflux::PotParams&, int i, double xi, const double* Lx) {
        if (i >= 2) return xi;
        const double x0 = Lx[0], r = Lx[1] - x0 * x0 + 1.0;
        return i == 0 ? x0 - 2.0 * x0 * r : r;
    }
    __device__ static void eval(const pdmpflux::PotParams&, int i, double xi, double di, const double* Lx,
                                const double* Ld, double& g, double& hd) {
        if (i >= 2) { g = xi; hd = di; return; }
        const double x0 = Lx[0], r = Lx[1] - x0 * x0 + 1.0;
        if (i == 0) {
            g = x0 - 2.0 * x0 * r;
            hd = (1.0 - 2.0 * r + 4.0 * x0 * x0) * Ld[0] - 2.0 * x0 * Ld[1];
        } else {
            g = r;
            hd = -2.0 * x0 * Ld[0] + Ld[1];
        }
    }
};
"""

GAUSS_SRC = r"""
struct UserPotential {
    static constexpr int K = 0;
    __device__ static void accum(const pdmpflux::PotParams&, int, double, double*) {}
    __device__ static double grad(const pdmpflux::PotParams& pp, int, double xi, const double*) { return %s * xi; }
    __device__ static void eval(const pdmpflux::PotParams& pp, int, double xi, double di, const double*, const double*,
                                double& g, double& hd) { g = %s * xi; hd = %s * di; }
};
"""


def _no_gpu():
    import ctypes as C
    n = C.c_int(0)
    return p.lib().pdmpflux_device_count(C.byref(n)) != 0 or n.value == 0


needs_no_gpu = pytest.mark.skipif(not _no_gpu(), reason="checks the behaviour of a machine without a CUDA device")


def test_syntax_error_points_at_user_line():
    src = BANANA_SRC.replace("return i == 0 ? x0 - 2.0 * x0 * r : r;", "return i == 0 ? x0 - 2.0 * x0 * r : r")
    line = src.splitlines().index("        return i == 0 ? x0 - 2.0 * x0 * r : r") + 1
    with pytest.raises(p.CompileError) as e:
        p.ZigZag(5, p.CudaPotential(src))
    msg = str(e.value)
    assert "user_potential(" in msg
    # the error is reported on the offending line or the one after it (where the missing ';' is noticed)
    assert f"user_potential({line})" in msg or f"user_potential({line + 1})" in msg, msg


def test_missing_member_is_named():
    start = BANANA_SRC.index("    __device__ static void eval(")
    end = BANANA_SRC.index("};", start)
    with pytest.raises(p.CompileError, match="UserPotential::eval"):
        p.ZigZag(5, p.CudaPotential(BANANA_SRC[:start] + BANANA_SRC[end:]))


def test_wrong_signature_is_named():
    with pytest.raises(p.CompileError, match="UserPotential::grad"):
        p.BPS(5, p.CudaPotential(BANANA_SRC.replace("double grad(const pdmpflux::PotParams&, int i, double xi,",
                                                    "double grad(const pdmpflux::PotParams&, int i, float xi,")))


def test_k_out_of_range():
    with pytest.raises(p.CompileError, match="K must be in 0 .. 8"):
        p.ZigZag(5, p.CudaPotential(BANANA_SRC.replace("K = 2;", "K = 9;")))


def test_create_with_builtin_entry_point_is_refused():
    import ctypes as C
    from pdmpflux_b200 import _lib
    h = C.c_void_p()
    assert _lib.lib().pdmpflux_potential_create(6, 3, None, 0, C.byref(h)) == _lib.ERR_ARGUMENT
    assert b"pdmpflux_potential_create_source" in _lib.lib().pdmpflux_last_error()


@needs_no_gpu
def test_samplers_compile_without_a_device():
    pot = p.CudaPotential(BANANA_SRC)
    count = p.lib().pdmpflux_jit_compile_count
    for make in (lambda: p.ZigZag(12, pot), lambda: p.ZigZag(12, pot, grid_size=0),
                 lambda: p.BPS(12, pot), lambda: p.ForwardECMC(12, pot), lambda: p.Boomerang(12, pot),
                 lambda: p.SpeedUpZigZag(12, pot)):
        s = make()
        assert s._handle
    n0 = count()
    # d = 12 <= 16: teams of 1 and 8 are both possible, and a fresh kind compiles both; d = 300 needs a warp per chain
    p.BPS(300, pot)
    assert count() == n0 + 1
    with pytest.raises(p.CudaError):
        p.StickyZigZag(12, pot, np.full(12, 0.5))   # the kernels compile; only the kappa upload needs the device
    assert count() == n0 + 3


@needs_no_gpu
def test_compile_cache_and_count():
    count = p.lib().pdmpflux_jit_compile_count
    src = GAUSS_SRC % ("1.25", "1.25", "1.25")
    n0 = count()
    p.ZigZag(7, p.CudaPotential(src))
    n1 = count()
    assert n1 == n0 + 3                      # contract check + teams 1 and 8
    p.ZigZag(7, p.CudaPotential(src))        # same source, same kind: all cached
    p.ZigZag(9, p.CudaPotential(src), grid_size=0)   # other config, same generic kernels
    assert count() == n1
    p.BPS(7, p.CudaPotential(src))           # a new kind: two new kernels
    assert count() == n1 + 2
    p.ZigZag(7, p.CudaPotential(src + "\n// another source\n"))
    assert count() == n1 + 5


@needs_no_gpu
def test_sampling_without_a_device_raises():
    s = p.ZigZag(4, p.CudaPotential(GAUSS_SRC % ("1.0", "1.0", "1.0")))
    with pytest.raises(p.CudaError):
        p.sample_skeleton(s, 10, np.zeros((2, 4)), np.ones((2, 4)), seed=1)
    with pytest.raises(p.CudaError):
        p.ZigZag(4, p.CudaPotential(GAUSS_SRC % ("pp.vec[0]", "pp.vec[0]", "pp.vec[0]"), params=[2.0]))
