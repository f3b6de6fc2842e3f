// Device potential plugins: fused gradient / Hessian-vector evaluation per coordinate.
//
// The reference takes an arbitrary Julia closure `grad U` (ZigZagSamplers.jl:58, ADBackend.jl:30-142); on the
// device a potential is a compile-time functor (SURVEY.md H6).  A potential exposes K *linear functionals*
// L_k(x) (coordinate picks or sums).  Because both flows act on every coordinate with the same 2x2 map
// (x_t = a x + b v, v_t = c x + d v), L_k(x_t) = a L_k(x) + b L_k(v): the functionals are reduced once per
// (x, v) and every later evaluation along the flow line is purely coordinate-local (no cross-lane traffic).
//
//   accum(pp, i, xi, acc)                 acc[k] += contribution of coordinate i to L_k
//   grad (pp, i, xi, Lx)                  -> (grad U(x))_i
//   eval (pp, i, xi, di, Lx, Ld, g, hd)   g = (grad U(x))_i, hd = (H(x) dir)_i with dir_i = di, L(dir) = Ld
//
// Line structure used by the fast paths (chain.cuh): for `kAffine` potentials the Hessian is constant and
// decoupled for every coordinate i >= kSpecial, so along x + t v the signed coordinate rate is exactly
// A_i + t B_i with A_i = g_i(x) v_i, B_i = (H v)_i v_i; the first kSpecial coordinates are functions of the
// functionals L_0..L_{kSpecial-1} (= those coordinates themselves) and are evaluated per time by every lane.
//
// `kSplit` potentials also expose the line sums in split form (BPS / ForwardECMC: <grad U(x), d> and <H d, d>):
//   eval_local(pp, i, xi, di, gl, hl)     the parts of g_i, (H d)_i that do not involve the functionals
//   line_corr (pp, Lx, Ld, ca, cb)        sum_i (g_i - gl_i) d_i and sum_i ((H d)_i - hl_i) d_i, from the functionals alone
// so that one pass can accumulate the functionals of a new direction AND its line model (chain.cuh: prepare_line,
// accept_bps_fused).
//
// Formulas: SURVEY.md Appendix A (GAUSS_STD README.md:36-38; BANANA test/test_config.jl:33-36;
// BANANA_README_SCALAR README.md:62-65; the others are not defined upstream).
#pragma once
#include "common.cuh"

namespace pdmpflux {

template <int POT>
struct Pot;

template <>
struct Pot<PDMPFLUX_GAUSS_STD> {
    static constexpr int K = 0;
    static constexpr bool kAffine = true;   // g_i(x + t v) v_i is affine in t for every i >= kSpecial
    static constexpr int kSpecial = 0;
    __device__ static void accum(const PotParams&, int, double, double*) {}
    __device__ static double grad(const PotParams&, int, double xi, const double*) { return xi; }
    __device__ static void eval(const PotParams&, int, double xi, double di, const double*, const double*,
                                double& g, double& hd) {
        g = xi; hd = di;
    }
    static constexpr bool kSplit = true;
    __device__ static void eval_local(const PotParams&, int, double xi, double di, double& gl, double& hl) { gl = xi; hl = di; }
    __device__ static void line_corr(const PotParams&, const double*, const double*, double& ca, double& cb) { ca = 0.0; cb = 0.0; }
};

template <>
struct Pot<PDMPFLUX_GAUSS_DIAG> {
    static constexpr int K = 0;
    static constexpr bool kAffine = true;
    static constexpr int kSpecial = 0;
    __device__ static void accum(const PotParams&, int, double, double*) {}
    __device__ static double grad(const PotParams& pp, int i, double xi, const double*) {
        return __ldg(pp.vec + i) * xi;
    }
    __device__ static void eval(const PotParams& pp, int i, double xi, double di, const double*, const double*,
                                double& g, double& hd) {
        const double p = __ldg(pp.vec + i);
        g = p * xi; hd = p * di;
    }
    static constexpr bool kSplit = true;
    __device__ static void eval_local(const PotParams& pp, int i, double xi, double di, double& gl, double& hl) {
        const double p = __ldg(pp.vec + i);
        gl = p * xi; hl = p * di;
    }
    __device__ static void line_corr(const PotParams&, const double*, const double*, double& ca, double& cb) { ca = 0.0; cb = 0.0; }
};

template <>
struct Pot<PDMPFLUX_GAUSS_EQUICORR> {  // P = alpha I - beta 1 1^T
    static constexpr int K = 1;
    static constexpr bool kAffine = true;
    static constexpr int kSpecial = 0;
    __device__ static void accum(const PotParams&, int, double xi, double* acc) { acc[0] += xi; }
    __device__ static double grad(const PotParams& pp, int, double xi, const double* Lx) {
        return pp.alpha * xi - pp.beta * Lx[0];
    }
    __device__ static void eval(const PotParams& pp, int, double xi, double di, const double* Lx,
                                const double* Ld, double& g, double& hd) {
        g = pp.alpha * xi - pp.beta * Lx[0];
        hd = pp.alpha * di - pp.beta * Ld[0];
    }
    static constexpr bool kSplit = true;   // sum_i g_i d_i = alpha <x, d> - beta L(x) L(d), sum_i (H d)_i d_i = alpha <d, d> - beta L(d)^2
    __device__ static void eval_local(const PotParams& pp, int, double xi, double di, double& gl, double& hl) {
        gl = pp.alpha * xi; hl = pp.alpha * di;
    }
    __device__ static void line_corr(const PotParams& pp, const double* Lx, const double* Ld, double& ca, double& cb) {
        ca = -pp.beta * Lx[0] * Ld[0];
        cb = -pp.beta * Ld[0] * Ld[0];
    }
};

template <>
struct Pot<PDMPFLUX_BANANA> {  // L0 = x_1, L1 = x_2 (1-based); r = x2 - x1^2 + 1
    static constexpr bool kSplit = false;
    static constexpr int K = 2;
    static constexpr bool kAffine = true;   // coordinates >= 2 are standard-Gaussian
    static constexpr int kSpecial = 2;      // coordinates 0, 1 are polynomial in t and functions of (L0, L1) only
    static constexpr bool kPickFunctionals = true;   // L_k = x_k for k < K: picks, not sums (chain.cuh: compute_functionals)
    __device__ static void accum(const PotParams&, int i, double xi, double* acc) {
        if (i == 0) acc[0] += xi;
        if (i == 1) acc[1] += xi;
    }
    __device__ static double grad(const PotParams&, int i, double xi, const double* Lx) {
        if (i >= 2) return xi;
        const double x0 = Lx[0], r = Lx[1] - x0 * x0 + 1.0;
        return i == 0 ? x0 - 2.0 * x0 * r : r;
    }
    __device__ static void eval(const PotParams&, int i, double xi, double di, const double* Lx,
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

template <>
struct Pot<PDMPFLUX_BANANA_README_SCALAR> {  // every coordinate = x1 + (x2 - (x1^2 - 1)) + sum_{i>=3} x_i
    static constexpr bool kSplit = false;
    static constexpr int K = 3;
    static constexpr bool kAffine = false;
    static constexpr int kSpecial = 0;
    __device__ static void accum(const PotParams&, int i, double xi, double* acc) {
        if (i == 0) acc[0] += xi;
        else if (i == 1) acc[1] += xi;
        else acc[2] += xi;
    }
    __device__ static double grad(const PotParams&, int, double, const double* Lx) {
        return Lx[0] + (Lx[1] - (Lx[0] * Lx[0] - 1.0)) + Lx[2];
    }
    __device__ static void eval(const PotParams&, int, double, double, const double* Lx, const double* Ld,
                                double& g, double& hd) {
        g = Lx[0] + (Lx[1] - (Lx[0] * Lx[0] - 1.0)) + Lx[2];
        hd = Ld[0] + (Ld[1] - 2.0 * Lx[0] * Ld[0]) + Ld[2];
    }
};

// U = (x - mu)' P (x - mu) / 2 with a dense symmetric positive-definite P (pp.vec = P row-major, pp.vec2 = mu).  The
// gradient needs all of x, not K <= 8 functionals, so the chain keeps g = P (x - mu) and h = P v itself (chain.cuh,
// kDense) and uses (g_i, h_i) wherever the fast paths take (grad U(x))_i and (H v)_i; the line model is exact.  The
// members below are never called: they let the generic code that the fast-path kernels compile (but never reach)
// type-check, and a NaN would show at once if a path did reach them.
template <>
struct Pot<PDMPFLUX_GAUSS_DENSE> {
    static constexpr int K = 0;
    static constexpr bool kAffine = true;
    static constexpr int kSpecial = 0;
    static constexpr bool kSplit = true;
    __device__ static void accum(const PotParams&, int, double, double*) {}
    __device__ static double grad(const PotParams&, int, double, const double*) { return CUDART_NAN; }
    __device__ static void eval(const PotParams&, int, double, double, const double*, const double*, double& g, double& hd) {
        g = CUDART_NAN; hd = CUDART_NAN;
    }
    __device__ static void eval_local(const PotParams&, int, double, double, double& gl, double& hl) { gl = CUDART_NAN; hl = CUDART_NAN; }
    __device__ static void line_corr(const PotParams&, const double*, const double*, double& ca, double& cb) { ca = 0.0; cb = 0.0; }
};

}  // namespace pdmpflux
