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
// Optional members declare a line model (potentials.cuh: kAffine, kSpecial, kSplit) and put the potential on the
// fast-path kernels:
//
//       static constexpr bool affine = true;   // g_i(x + t v) = g_i(x) + t (H v)_i exactly for every i >= special
//       static constexpr int special = 2;      // 0 <= special <= K, needs affine: L_k(x) = x_k for k < special (accum
//                                              // puts x_k, and nothing else, into acc[k]); the rates of these
//                                              // coordinates are evaluated per time from the functionals
//       __device__ static void eval_local(const pdmpflux::PotParams&, int i, double xi, double di, double& gl, double& hl);
//       __device__ static void line_corr(const pdmpflux::PotParams&, const double* Lx, const double* Ld, double& ca,
//                                        double& cb);
//                                              // both or neither; need affine and special = 0 (kSplit)
//
// Without them the potential has no line model (kAffine = false) and every sampler runs the generic kernel.  The
// library cannot check a declaration either: a wrong one samples the wrong target.
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

// optional line-model members: absent means no line model
template <class T, class = void> struct has_affine { static constexpr bool value = false; };
template <class T> struct has_affine<T, typename voider<decltype(T::affine)>::type> { static constexpr bool value = true; };
template <class T, bool = has_affine<T>::value> struct affine_of { static constexpr bool value = false; };
template <class T> struct affine_of<T, true> { static constexpr bool value = T::affine; };
template <class T, class = void> struct has_special { static constexpr bool value = false; };
template <class T> struct has_special<T, typename voider<decltype(T::special)>::type> { static constexpr bool value = true; };
template <class T, bool = has_special<T>::value> struct special_of { static constexpr int value = 0; };
template <class T> struct special_of<T, true> { static constexpr int value = T::special; };
// by name (any signature), then with the signature the kernels call
template <class T, class = void> struct names_eval_local { static constexpr bool value = false; };
template <class T> struct names_eval_local<T, typename voider<decltype(&T::eval_local)>::type> { static constexpr bool value = true; };
template <class T, class = void> struct names_line_corr { static constexpr bool value = false; };
template <class T> struct names_line_corr<T, typename voider<decltype(&T::line_corr)>::type> { static constexpr bool value = true; };
template <class T, class = void> struct has_eval_local { static constexpr bool value = false; };
template <class T>
struct has_eval_local<T, typename voider<decltype(static_cast<void (*)(const PotParams&, int, double, double, double&, double&)>(
                             &T::eval_local))>::type> {
    static constexpr bool value = true;
};
template <class T, class = void> struct has_line_corr { static constexpr bool value = false; };
template <class T>
struct has_line_corr<T, typename voider<decltype(static_cast<void (*)(const PotParams&, const double*, const double*, double&,
                                                                       double&)>(&T::line_corr))>::type> {
    static constexpr bool value = true;
};
template <class T> struct split_of { static constexpr bool value = has_eval_local<T>::value && has_line_corr<T>::value; };

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

using U = ::UserPotential;
static_assert(special_of<U>::value >= 0 && special_of<U>::value <= k_of<U>::value, "UserPotential::special must be in 0 .. K");
static_assert(special_of<U>::value == 0 || affine_of<U>::value,
              "UserPotential::special > 0 needs UserPotential::affine = true (the special coordinates are the "
              "exception to an affine gradient)");
static_assert(!names_eval_local<U>::value || has_eval_local<U>::value,
              "UserPotential::eval_local has the wrong signature: declare `__device__ static void eval_local(const "
              "pdmpflux::PotParams&, int i, double xi, double di, double& gl, double& hl)`");
static_assert(!names_line_corr<U>::value || has_line_corr<U>::value,
              "UserPotential::line_corr has the wrong signature: declare `__device__ static void line_corr(const "
              "pdmpflux::PotParams&, const double* Lx, const double* Ld, double& ca, double& cb)`");
static_assert(!names_eval_local<U>::value || names_line_corr<U>::value,
              "UserPotential::line_corr is missing: eval_local and line_corr declare the split line sums together");
static_assert(!names_line_corr<U>::value || names_eval_local<U>::value,
              "UserPotential::eval_local is missing: eval_local and line_corr declare the split line sums together");
static_assert(!split_of<U>::value || affine_of<U>::value,
              "UserPotential::eval_local / line_corr (split line sums) need UserPotential::affine = true");
static_assert(!split_of<U>::value || special_of<U>::value == 0,
              "UserPotential::eval_local / line_corr (split line sums) need UserPotential::special = 0");

// eval_local / line_corr exist exactly for split potentials (chain.cuh reaches them only under kSplit)
template <class T, bool = split_of<T>::value> struct split_members {};
template <class T>
struct split_members<T, true> {
    __device__ __forceinline__ static void eval_local(const PotParams& pp, int i, double xi, double di, double& gl, double& hl) {
        T::eval_local(pp, i, xi, di, gl, hl);
    }
    __device__ __forceinline__ static void line_corr(const PotParams& pp, const double* Lx, const double* Ld, double& ca,
                                                     double& cb) {
        T::line_corr(pp, Lx, Ld, ca, cb);
    }
};

}  // namespace user_contract

template <>
struct Pot<PDMPFLUX_SOURCE> : user_contract::split_members<::UserPotential> {
    static constexpr int K = user_contract::k_of<::UserPotential>::value;
    static constexpr bool kAffine = user_contract::affine_of<::UserPotential>::value;
    static constexpr int kSpecial = user_contract::special_of<::UserPotential>::value;
    static constexpr bool kSplit = user_contract::split_of<::UserPotential>::value;
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
