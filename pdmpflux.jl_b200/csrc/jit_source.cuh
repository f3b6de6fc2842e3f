// Wraps a user-written potential (struct UserPotential, compiled at run time by jit.cu) as Pot<PDMPFLUX_SOURCE>.
//
// The user text comes right before this header and must define, at global scope:
//
//   struct UserPotential {
//       static constexpr int K = ...;   // number of linear functionals, 0 <= K <= 8
//       __device__ static void accum(const pdmpflux::PotParams& pp, int i, double xi, double* acc);
//       __device__ static double grad(const pdmpflux::PotParams& pp, int i, double xi, const double* Lx);
//       __device__ static void eval(const pdmpflux::PotParams& pp, int i, double xi, double di, const double* Lx,
//                                   const double* Ld, double& g, double& hd);
//   };
//
// with the meaning of the built-in plugins (potentials.cuh): accum adds coordinate i's contribution to each functional
// L_k (it must be linear in xi: along the flow the kernels evaluate L(x_t) as a L(x) + b L(v)), grad returns
// (grad U(x))_i, eval returns g = (grad U(x))_i and hd = (H(x) dir)_i for dir_i = di with functionals Ld = L(dir).
// pp.vec[0 .. pp.n - 1] are the parameters given when the potential was created.  The library cannot check linearity.
//
// No line model is declared (kAffine = false), so every sampler runs the generic kernel with this potential.
#pragma once
#include "potentials.cuh"

namespace pdmpflux {
namespace user_contract {

template <class... T> struct voider { using type = void; };
template <class T, class = void> struct has_K { static constexpr bool value = false; };
template <class T> struct has_K<T, typename voider<decltype(T::K)>::type> { static constexpr bool value = true; };
template <class T, class = void> struct has_accum { static constexpr bool value = false; };
template <class T>
struct has_accum<T, typename voider<decltype(static_cast<void (*)(const PotParams&, int, double, double*)>(&T::accum))>::type> {
    static constexpr bool value = true;
};
template <class T, class = void> struct has_grad { static constexpr bool value = false; };
template <class T>
struct has_grad<T, typename voider<decltype(static_cast<double (*)(const PotParams&, int, double, const double*)>(&T::grad))>::type> {
    static constexpr bool value = true;
};
template <class T, class = void> struct has_eval { static constexpr bool value = false; };
template <class T>
struct has_eval<T, typename voider<decltype(static_cast<void (*)(const PotParams&, int, double, double, const double*, const double*,
                                                                 double&, double&)>(&T::eval))>::type> {
    static constexpr bool value = true;
};
template <class T, bool = has_K<T>::value> struct k_of { static constexpr int value = 0; };
template <class T> struct k_of<T, true> { static constexpr int value = T::K; };

static_assert(has_K<::UserPotential>::value, "UserPotential::K is missing: declare `static constexpr int K = <number of linear functionals>;`");
static_assert(k_of<::UserPotential>::value >= 0 && k_of<::UserPotential>::value <= 8, "UserPotential::K must be in 0 .. 8");
static_assert(has_accum<::UserPotential>::value,
              "UserPotential::accum is missing or has the wrong signature: declare "
              "`__device__ static void accum(const pdmpflux::PotParams&, int i, double xi, double* acc)`");
static_assert(has_grad<::UserPotential>::value,
              "UserPotential::grad is missing or has the wrong signature: declare "
              "`__device__ static double grad(const pdmpflux::PotParams&, int i, double xi, const double* Lx)`");
static_assert(has_eval<::UserPotential>::value,
              "UserPotential::eval is missing or has the wrong signature: declare `__device__ static void eval(const "
              "pdmpflux::PotParams&, int i, double xi, double di, const double* Lx, const double* Ld, double& g, double& hd)`");

}  // namespace user_contract

template <>
struct Pot<PDMPFLUX_SOURCE> {
    static constexpr int K = user_contract::k_of<::UserPotential>::value;
    static constexpr bool kAffine = false;
    static constexpr int kSpecial = 0;
    static constexpr bool kSplit = false;
    __device__ __forceinline__ static void accum(const PotParams& pp, int i, double xi, double* acc) {
        ::UserPotential::accum(pp, i, xi, acc);
    }
    __device__ __forceinline__ static double grad(const PotParams& pp, int i, double xi, const double* Lx) {
        return ::UserPotential::grad(pp, i, xi, Lx);
    }
    __device__ __forceinline__ static void eval(const PotParams& pp, int i, double xi, double di, const double* Lx,
                                                const double* Ld, double& g, double& hd) {
        ::UserPotential::eval(pp, i, xi, di, Lx, Ld, g, hd);
    }
};

// the host passes sizeof(KernelParams) as it was compiled into the library: both sides must agree on the layout
#ifdef PDMPFLUX_HOST_KERNEL_PARAMS_BYTES
static_assert(sizeof(KernelParams) == PDMPFLUX_HOST_KERNEL_PARAMS_BYTES, "KernelParams differs between the library and the run-time compiled kernel");
#endif

}  // namespace pdmpflux
