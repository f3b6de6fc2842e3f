"""Source potentials that declare a line model (`affine`, `special`, `eval_local` / `line_corr`), without a GPU: the
declaration is checked by the contract check at construction, and the samplers compile the fast-path kernels the
default policy picks for them (Boomerang excepted) before any CUDA call.

The restated sources here are also used by tests/test_gpu_source_line_model.py."""
import numpy as np
import pytest

import pdmpflux_b200 as p
from test_source_potential_cpu import BANANA_SRC, needs_no_gpu

LINE_MODEL = """    static constexpr bool affine = true;
    static constexpr int special = 2;
"""
OPEN = "struct UserPotential {\n"

# Pot<PDMPFLUX_BANANA> (csrc/potentials.cuh) restated with its line model: coordinates >= 2 are standard Gaussian,
# coordinates 0 and 1 are the functionals L0, L1
BANANA_LM_SRC = BANANA_SRC.replace(OPEN, OPEN + LINE_MODEL)

# Pot<PDMPFLUX_GAUSS_DIAG> restated with the split line sums; params: the d precisions
GAUSS_DIAG_SPLIT_SRC = r"""
struct UserPotential {
    static constexpr int K = 0;
    static constexpr bool affine = true;
    __device__ static void accum(const pdmpflux::PotParams&, int, double, double*) {}
    __device__ static double grad(const pdmpflux::PotParams& pp, int i, double xi, const double*) {
        return __ldg(pp.vec + i) * xi;
    }
    __device__ static void eval(const pdmpflux::PotParams& pp, int i, double xi, double di, const double*, const double*,
                                double& g, double& hd) {
        const double p = __ldg(pp.vec + i);
        g = p * xi; hd = p * di;
    }
    __device__ static void eval_local(const pdmpflux::PotParams& pp, int i, double xi, double di, double& gl, double& hl) {
        const double p = __ldg(pp.vec + i);
        gl = p * xi; hl = p * di;
    }
    __device__ static void line_corr(const pdmpflux::PotParams&, const double*, const double*, double& ca, double& cb) {
        ca = 0.0; cb = 0.0;
    }
};
"""

# Pot<PDMPFLUX_GAUSS_EQUICORR> restated with the split line sums, P = alpha I - beta 1 1^T.  alpha and beta are
# compiled in (equicorr_split_src), as the built-in reads them from the kernel parameters: a value loaded through
# pp.vec cannot be hoisted across the stores of the fused BPS reflection pass, which changes where the compiler
# contracts multiply-adds, so such a restatement matches the built-in only to rounding.
GAUSS_EQUICORR_SPLIT_SRC = r"""
struct UserPotential {
    static constexpr int K = 1;
    static constexpr bool affine = true;
    static constexpr double alpha = ALPHA, beta = BETA;
    __device__ static void accum(const pdmpflux::PotParams&, int, double xi, double* acc) { acc[0] += xi; }
    __device__ static double grad(const pdmpflux::PotParams&, int, double xi, const double* Lx) {
        return alpha * xi - beta * Lx[0];
    }
    __device__ static void eval(const pdmpflux::PotParams&, int, double xi, double di, const double* Lx,
                                const double* Ld, double& g, double& hd) {
        g = alpha * xi - beta * Lx[0];
        hd = alpha * di - beta * Ld[0];
    }
    __device__ static void eval_local(const pdmpflux::PotParams&, int, double xi, double di, double& gl, double& hl) {
        gl = alpha * xi; hl = alpha * di;
    }
    __device__ static void line_corr(const pdmpflux::PotParams&, const double* Lx, const double* Ld, double& ca,
                                     double& cb) {
        ca = -beta * Lx[0] * Ld[0];
        cb = -beta * Ld[0] * Ld[0];
    }
};
"""


def equicorr_split_src(alpha, beta):
    return GAUSS_EQUICORR_SPLIT_SRC.replace("ALPHA", float(alpha).hex()).replace("BETA", float(beta).hex())


# U = x0^2 / 2 + (x1 - x0^2 + 1)^2 / 2 + sum_{i >= 2} p_i x_i^2 / 2; params: p[0 .. d-1] (p0, p1 unused)
BANANA_PREC_SRC = r"""
struct UserPotential {
    static constexpr int K = 2;
    static constexpr bool affine = true;
    static constexpr int special = 2;
    __device__ static void accum(const pdmpflux::PotParams&, int i, double xi, double* acc) {
        if (i == 0) acc[0] += xi;
        if (i == 1) acc[1] += xi;
    }
    __device__ static double grad(const pdmpflux::PotParams& pp, int i, double xi, const double* Lx) {
        if (i >= 2) return pp.vec[i] * xi;
        const double x0 = Lx[0], r = Lx[1] - x0 * x0 + 1.0;
        return i == 0 ? x0 - 2.0 * x0 * r : r;
    }
    __device__ static void eval(const pdmpflux::PotParams& pp, int i, double xi, double di, const double* Lx,
                                const double* Ld, double& g, double& hd) {
        if (i >= 2) { g = pp.vec[i] * xi; hd = pp.vec[i] * di; return; }
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

# U = sum_i p_i (x_i - mu_i)^2 / 2 + sum_k (u_k . x)^2 / 2 with K = 2, i.e. N(Q^-1 D mu, Q^-1) for Q = D + U U^T;
# params: p[d], mu[d], u0[d], u1[d]
LOWRANK_SRC = r"""
struct UserPotential {
    static constexpr int K = 2;
    static constexpr bool affine = true;
    __device__ static int dim(const pdmpflux::PotParams& pp) { return (int)(pp.n / 4); }
    __device__ static void accum(const pdmpflux::PotParams& pp, int i, double xi, double* acc) {
        const int d = dim(pp);
        acc[0] += pp.vec[2 * d + i] * xi;
        acc[1] += pp.vec[3 * d + i] * xi;
    }
    __device__ static double grad(const pdmpflux::PotParams& pp, int i, double xi, const double* Lx) {
        const int d = dim(pp);
        return pp.vec[i] * (xi - pp.vec[d + i]) + pp.vec[2 * d + i] * Lx[0] + pp.vec[3 * d + i] * Lx[1];
    }
    __device__ static void eval(const pdmpflux::PotParams& pp, int i, double xi, double di, const double* Lx,
                                const double* Ld, double& g, double& hd) {
        const int d = dim(pp);
        const double u0 = pp.vec[2 * d + i], u1 = pp.vec[3 * d + i];
        g = pp.vec[i] * (xi - pp.vec[d + i]) + u0 * Lx[0] + u1 * Lx[1];
        hd = pp.vec[i] * di + u0 * Ld[0] + u1 * Ld[1];
    }
    __device__ static void eval_local(const pdmpflux::PotParams& pp, int i, double xi, double di, double& gl, double& hl) {
        const int d = dim(pp);
        gl = pp.vec[i] * (xi - pp.vec[d + i]);
        hl = pp.vec[i] * di;
    }
    __device__ static void line_corr(const pdmpflux::PotParams&, const double* Lx, const double* Ld, double& ca,
                                     double& cb) {
        ca = Lx[0] * Ld[0] + Lx[1] * Ld[1];
        cb = Ld[0] * Ld[0] + Ld[1] * Ld[1];
    }
};
"""


def lowrank_params(d, seed=0):
    g = np.random.default_rng(seed)
    prec = np.linspace(0.5, 2.0, d)
    mu = g.uniform(-1.0, 1.0, d)
    u = 0.4 * g.standard_normal((2, d))
    return prec, mu, u, np.concatenate([prec, mu, u[0], u[1]])


def _member(src, name):
    """the text of `__device__ static void <name>(...) { ... }` in src"""
    start = src.index(f"    __device__ static void {name}(")
    end = src.index("\n    }\n", start) + len("\n    }\n")
    return src[start:end]


def _refused(src, match, d=5):
    with pytest.raises(p.CompileError, match=match):
        p.ZigZag(d, p.CudaPotential(src), grid_size=0)


@pytest.mark.parametrize("special", ["3", "-1"])
def test_special_out_of_range(special):
    _refused(BANANA_LM_SRC.replace("special = 2;", f"special = {special};"), r"UserPotential::special must be in 0 \.\. K")


def test_special_without_affine():
    _refused(BANANA_LM_SRC.replace("    static constexpr bool affine = true;\n", ""), r"UserPotential::special > 0 needs")


def test_eval_local_without_line_corr():
    _refused(LOWRANK_SRC.replace(_member(LOWRANK_SRC, "line_corr"), ""), r"UserPotential::line_corr is missing")


def test_line_corr_without_eval_local():
    _refused(LOWRANK_SRC.replace(_member(LOWRANK_SRC, "eval_local"), ""), r"UserPotential::eval_local is missing")


def test_eval_local_wrong_signature():
    src = LOWRANK_SRC.replace("double xi, double di, double& gl, double& hl)", "double xi, double di, double& gl, float& hl)")
    _refused(src.replace("hl = pp.vec[i] * di;", "hl = (float)(pp.vec[i] * di);"), r"UserPotential::eval_local has the wrong signature")


def test_line_corr_wrong_signature():
    _refused(LOWRANK_SRC.replace("const double* Lx, const double* Ld, double& ca,", "const double* Lx, double* Ld, double& ca,"),
             r"UserPotential::line_corr has the wrong signature")


def test_split_without_affine():
    _refused(LOWRANK_SRC.replace("    static constexpr bool affine = true;\n", ""),
             r"UserPotential::eval_local / line_corr \(split line sums\) need UserPotential::affine = true")


def test_split_with_special():
    src = LOWRANK_SRC.replace("    static constexpr bool affine = true;\n", LINE_MODEL.replace("special = 2", "special = 1"))
    _refused(src, r"UserPotential::eval_local / line_corr \(split line sums\) need UserPotential::special = 0")


def test_declared_sources_compile():
    """every restated or new declared source passes the contract check"""
    _, _, _, lr = lowrank_params(6)
    for src, params in ((BANANA_LM_SRC, ()), (GAUSS_DIAG_SPLIT_SRC, np.ones(6)), (equicorr_split_src(1.5, 0.1), ()),
                        (BANANA_PREC_SRC, np.ones(6)), (LOWRANK_SRC, lr)):
        try:
            assert p.ZigZag(6, p.CudaPotential(src, params), grid_size=0)._handle
        except p.CudaError:   # parameter upload on a machine without a device: the compiles have passed
            pass


@needs_no_gpu
def test_declared_samplers_build_without_a_device():
    pot = p.CudaPotential(BANANA_LM_SRC)
    for make in (lambda: p.ZigZag(12, pot, grid_size=0), lambda: p.ZigZag(12, pot, AD_backend="ForwardDiff"),
                 lambda: p.BPS(12, pot), lambda: p.BPS(12, pot, grid_size=0), lambda: p.ForwardECMC(12, pot),
                 lambda: p.Boomerang(12, pot)):
        assert make()._handle


@needs_no_gpu
def test_fast_path_compile_set():
    count = p.lib().pdmpflux_jit_compile_count
    src = BANANA_LM_SRC + "\n// compile-set test\n"
    n0 = count()
    p.ZigZag(12, p.CudaPotential(src), grid_size=0)
    # contract check + team 1 (thread-per-chain compressed line model) + team 8 (transposed search)
    assert count() == n0 + 3
    n1 = count()
    p.ZigZag(12, p.CudaPotential(src), grid_size=0, tmax=3.0)   # other config, same kernels
    assert count() == n1
    p.ZigZag(100, p.CudaPotential(src), grid_size=0)             # d > 64: team 8 at any chain count (register model)
    assert count() == n1 + 1
    p.ZigZag(136, p.CudaPotential(src), grid_size=0)             # 17 owned coordinates: team 8, shared line model
    assert count() == n1 + 2
    p.ZigZag(200, p.CudaPotential(src), grid_size=0)             # 25 owned coordinates: widened to a warp per chain
    assert count() == n1 + 3
    p.ZigZag(12, p.CudaPotential(src), AD_backend="ForwardDiff")   # affine-cell grid bound: teams 1 and 8
    assert count() == n1 + 5
    p.ZigZag(12, p.CudaPotential(src), AD_backend="FiniteDiff")    # finite differences: the generic kernels
    assert count() == n1 + 7


@needs_no_gpu
def test_boomerang_keeps_generic_kernels():
    """Boomerang's fast path assumes grad U(0) = 0, which an affine declaration does not promise: a declared source
    compiles the same generic kernels there as a copy without the declaration, and nothing else"""
    count = p.lib().pdmpflux_jit_compile_count
    src = BANANA_LM_SRC.replace("special = 2", "special = 0") + "\n// boomerang test\n"
    n0 = count()
    p.Boomerang(12, p.CudaPotential(src))
    assert count() == n0 + 3              # contract check + generic teams 1 and 8
    n1 = count()
    p.Boomerang(12, p.CudaPotential(src), grid_size=0)   # the fast path would be kPathFastBrent: still generic
    assert count() == n1
