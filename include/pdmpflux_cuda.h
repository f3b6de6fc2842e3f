/*
 * libpdmpflux_cuda.so -- C ABI of the B200-native grid-based Poisson-thinning engine.
 *
 * Drop-in boundary for PDMPFlux.jl's hot path.  The reference has NO native/FFI layer (pure Julia,
 * SURVEY.md 8b): these entry points are what a Julia `ccall` binding (julia/PDMPFluxCUDA.jl) or a ctypes
 * binding (pdmpflux_b200/_lib.py) binds in place of the Julia functions cited on each declaration
 * (file:line relative to the reference root).
 *
 * Conventions
 *   - plain C, no exceptions cross the ABI: every call returns PDMPFLUX_OK (0) or a negative
 *     pdmpflux_error code; pdmpflux_last_error() returns a thread-local message.
 *   - all floating point is IEEE binary64; counters are int32 as in PDMPHistory (Composites.jl:138-149).
 *   - "chain-major" skeleton layout: chain c's slab of X is a column-major d x n_cols matrix starting at
 *     X + c*d*n_cols, i.e. exactly a Julia Matrix{Float64}(d, n_cols) (zero-copy unsafe_wrap).
 *   - caller owns every buffer; the library never retains caller pointers past return.
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with PDMPFLUX_ERR_CUDA.
 */
#ifndef PDMPFLUX_CUDA_H
#define PDMPFLUX_CUDA_H

#ifndef __CUDACC_RTC__ /* the run-time compiled kernels get the fixed-width types from common.cuh */
#include <stddef.h>
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define PDMPFLUX_VERSION 200 /* 0.2.1: potential kind PDMPFLUX_GAUSS_DENSE (appended; no layout change); 0.2.0:
                                 pdmpflux_history gained is_active (appended), Sticky Zig-Zag, reductions */

typedef enum pdmpflux_error {
    PDMPFLUX_OK = 0,
    PDMPFLUX_ERR_ARGUMENT = -1,           /* Julia ArgumentError (dim<=0, grid_size<0, n_sk<=0, N<=0 ...) */
    PDMPFLUX_ERR_DIMENSION_MISMATCH = -2, /* Julia DimensionMismatch (AbstractPDMP.jl:96-98) */
    PDMPFLUX_ERR_UNSUPPORTED = -3,        /* sampler/potential/option outside the device path (no fallback) */
    PDMPFLUX_ERR_CUDA = -4,               /* CUDA runtime error, or no device */
    PDMPFLUX_ERR_CHAIN = -5,              /* at least one chain stopped; see per-chain status */
    PDMPFLUX_ERR_CAPACITY = -6,           /* time-horizon variant: some chain needs more than `capacity` columns */
    PDMPFLUX_ERR_COMPILE = -7             /* a source potential did not compile; pdmpflux_last_error() holds the NVRTC log */
} pdmpflux_error;

/* src/Samplers/{ZigZagSamplers,BouncyParticleSamplers,ForwardEventChainMonteCarlo,BoomerangSamplers}.jl */
typedef enum pdmpflux_sampler_kind {
    PDMPFLUX_ZIGZAG = 0, PDMPFLUX_BPS = 1, PDMPFLUX_FECMC = 2, PDMPFLUX_BOOMERANG = 3,
    PDMPFLUX_STICKY_ZIGZAG = 4, /* src/Samplers/StickyZigZagSamplers.jl + src/StickySamplingLoop.jl; create it with
                                   pdmpflux_sampler_create_sticky (it needs the thawing rates kappa) */
    PDMPFLUX_SPEEDUP_ZIGZAG = 5 /* src/Samplers/SpeedUpZigZagSamplers.jl: Zig-Zag with speed sqrt(1 + |x|^2) (closed-form
                                   nonlinear flow :71-79, effective gradient :81-83); generic path, no fused moments */
} pdmpflux_sampler_kind;

/* Device potential plugins (replace the Julia closure `grad U`; SURVEY.md Appendix A).  params layout:
 *   GAUSS_STD            -                      U = |x|^2/2                      (README.md:36-38)
 *   GAUSS_DIAG           p[d]                   U = sum p_i x_i^2 / 2
 *   GAUSS_EQUICORR       rho                    Sigma = (1-rho) I + rho 11^T ("slanted Gaussian")
 *   BANANA               -                      test/test_config.jl:33-36
 *   BANANA_README_SCALAR -                      README.md:62-65 (scalar "gradient" broadcast to all coords)
 *   LOGREG               n, sigma0, X[n*d] row-major, y[n]
 *   SOURCE               p[n_params]            user-written CUDA source (pdmpflux_potential_create_source)
 *   GAUSS_DENSE          P[d*d] row-major, mu[d] U = (x - mu)' P (x - mu) / 2, P symmetric positive definite
 * GAUSS_DENSE: P must be finite, symmetric to 1e-12 max|P| (it is stored as (P + P')/2) and positive definite
 * (ERR_ARGUMENT otherwise); d <= 2048 (ERR_UNSUPPORTED above).  It runs on Zig-Zag and BPS only, on the configurations
 * with a fast-path kernel: Zig-Zag needs a Brent bound (grid_size = 0) or a vectorised grid bound with an exact
 * AD_backend; every BPS configuration qualifies.  Anything else is ERR_UNSUPPORTED at sampler creation.  The chains
 * keep g = P (x - mu) and h = P v next to x and v and update them per event (a Zig-Zag flip reads one row of P, a BPS
 * reflection or refresh all of it).  pdmpflux_rv_diagnostic does not run it (ERR_UNSUPPORTED).
 */
typedef enum pdmpflux_potential_kind {
    PDMPFLUX_GAUSS_STD = 0, PDMPFLUX_GAUSS_DIAG = 1, PDMPFLUX_GAUSS_EQUICORR = 2, PDMPFLUX_BANANA = 3,
    PDMPFLUX_BANANA_README_SCALAR = 4, PDMPFLUX_LOGREG = 5,
    PDMPFLUX_SOURCE = 6, /* created by pdmpflux_potential_create_source only */
    PDMPFLUX_GAUSS_DENSE = 7
} pdmpflux_potential_kind;

/* How d/dt of the rate is obtained on the time grid: JVP = analytic (what AD_backend="ForwardDiff" computes,
 * UpperBound.jl:102,210); FD = the reference's finite_difference_derivative (UpperBound.jl:50-76). */
typedef enum pdmpflux_deriv_mode { PDMPFLUX_DERIV_JVP = 0, PDMPFLUX_DERIV_FD = 1 } pdmpflux_deriv_mode;

/* per-chain status written to pdmpflux_history.status */
typedef enum pdmpflux_chain_status {
    PDMPFLUX_CHAIN_OK = 0,
    PDMPFLUX_CHAIN_TAPE_EXHAUSTED = 1, /* injected draw tape ran out */
    PDMPFLUX_CHAIN_NOT_PROBVEC = 2,    /* ZigZag jump with sum(lambda)==0/NaN: the reference's Categorical throws */
    PDMPFLUX_CHAIN_STEP_LIMIT = 3,     /* more than max_steps thinning steps inside one event */
    PDMPFLUX_CHAIN_DONE = 4            /* time-horizon variant: the chain reached t = T (not an error) */
} pdmpflux_chain_status;

/* Keyword arguments of the reference constructors (ZigZagSamplers.jl:58-60, BouncyParticleSamplers.jl:21-24,
 * ForwardEventChainMonteCarlo.jl:301-303, BoomerangSamplers.jl:21-23).  pdmpflux_sampler_create applies the
 * same rewrites the constructors do (tmax==0 -> 1 & adaptive; ZigZag signed&&!vectorized -> unsigned;
 * non-ZigZag -> vectorized_bound=0; FECMC -> refresh_rate=0, dim==2 -> mix_p=0). */
typedef struct pdmpflux_config {
    int32_t grid_size;        /* 0 = constant bound via Brent (UpperBound.jl:18-36); otherwise >= 2 */
    int32_t vectorized_bound; /* UpperBound.jl:203-247 vs :92-137 */
    int32_t signed_bound;     /* AbstractPDMP.jl:104-112 */
    int32_t adaptive;         /* horizon adaptation, SamplingLoopInplace.jl:98,140,194 */
    int32_t deriv_mode;       /* pdmpflux_deriv_mode */
    int32_t gaussian_velocity;/* BPS */
    int32_t ran_p;            /* FECMC */
    int32_t switch_;          /* FECMC `switch` */
    int32_t positive;         /* FECMC */
    int32_t max_steps;        /* 0 -> default 100000 thinning steps per event before STEP_LIMIT */
    double tmax;
    double refresh_rate;
    double mix_p;             /* FECMC */
    double speed_factor;      /* FECMC */
} pdmpflux_config;

/* Injected draws (parity mode): three typed streams per chain, consumed in the reference's order
 * (SURVEY.md 8a "RNG draw order").  Chain c reads E + c*nE, U + c*nU, N + c*nN.  NULL tape -> Philox4x32-10
 * keyed by (seed, global chain id, event index), see pdmpflux.jl_b200/csrc/philox.cuh. */
typedef struct pdmpflux_tape {
    const double* E; /* randexp  draws */
    const double* U; /* rand     draws */
    const double* N; /* randn    draws */
    int64_t nE, nU, nN;
    int32_t on_device; /* pointers are device pointers */
} pdmpflux_tape;

/* Output columns of PDMPHistory (Composites.jl:138-149), chain-major; any pointer may be NULL (not stored).
 * is_active (the BitMatrix of Composites.jl:143, written by record! :254-258) is stored as one byte per coordinate and
 * only by the Sticky Zig-Zag sampler; for the other samplers it is all-true and is left untouched (build trues(d, n)
 * host-side). */
typedef struct pdmpflux_history {
    double* X;               /* [C][n_cols][d] */
    double* V;               /* [C][n_cols][d] */
    double* t;               /* [C][n_cols]    */
    double* horizon;         /* [C][n_cols]    */
    double* ar;              /* [C][n_cols]    */
    double* error_value_ar;  /* [C][n_cols][5] */
    int32_t* errored_bound;  /* [C][n_cols]    */
    int32_t* rejected;       /* [C][n_cols]    */
    int32_t* hitting_horizon;/* [C][n_cols]    */
    int32_t* status;         /* [C] pdmpflux_chain_status */
    int64_t* tape_pos;       /* [C][3] draws consumed from (E,U,N) (tape mode) */
    int64_t* counters;       /* [C][2] (bound builds, rate evaluations) -- instrumentation */
    int64_t n_cols;          /* leading dimension (columns per chain slab) */
    int32_t on_device;       /* all pointers above and below are device pointers */
    uint8_t* is_active;      /* [C][n_cols][d] 0 / 1, Sticky Zig-Zag only (NULL: not stored) */
} pdmpflux_history;

typedef struct pdmpflux_potential_s* pdmpflux_potential_t;
typedef struct pdmpflux_sampler_s* pdmpflux_sampler_t;
typedef struct pdmpflux_chains_s* pdmpflux_chains_t;

#ifndef __CUDACC_RTC__ /* host entry points: not part of the run-time compiled kernels */
int pdmpflux_version(void);
const char* pdmpflux_last_error(void);
int pdmpflux_device_count(int* count);
int pdmpflux_set_device(int device);

/* replaces the `grad U` closure argument of the constructors; copies params to the device */
int pdmpflux_potential_create(int kind, int dim, const double* params, int64_t n_params,
                              pdmpflux_potential_t* out);
int pdmpflux_potential_destroy(pdmpflux_potential_t pot);

/* A potential written by the user in CUDA C++ (the closest thing to the reference's arbitrary `grad U` closure).
 * `source` defines one struct at global scope with the members of the built-in plugins (csrc/potentials.cuh):
 *
 *   struct UserPotential {   // U = sum_i log cosh(s_i x_i) + c/2 (sum_i x_i)^2 ; params = s[0..d-1], c
 *       static constexpr int K = 1;                                        // number of linear functionals, 0 <= K <= 8
 *       __device__ static void accum(const pdmpflux::PotParams&, int i, double xi, double* acc) { acc[0] += xi; }
 *       __device__ static double grad(const pdmpflux::PotParams& pp, int i, double xi, const double* Lx) {
 *           const double s = pp.vec[i];
 *           return s * tanh(s * xi) + pp.vec[pp.n - 1] * Lx[0];
 *       }
 *       __device__ static void eval(const pdmpflux::PotParams& pp, int i, double xi, double di, const double* Lx,
 *                                   const double* Ld, double& g, double& hd) {
 *           const double s = pp.vec[i], th = tanh(s * xi), c = pp.vec[pp.n - 1];
 *           g = s * th + c * Lx[0];
 *           hd = s * s * (1.0 - th * th) * di + c * Ld[0];
 *       }
 *   };
 *
 *   accum(pp, i, xi, acc)               acc[k] += contribution of coordinate i to the linear functional L_k(x).  It MUST
 *                                       be linear in xi: along the flow the kernels evaluate L(x_t) as a L(x) + b L(v).
 *   grad(pp, i, xi, Lx)                 (grad U(x))_i, given x_i and the functionals Lx = L(x)
 *   eval(pp, i, xi, di, Lx, Ld, g, hd)  g = (grad U(x))_i and hd = (H(x) dir)_i, where dir_i = di and Ld = L(dir)
 *
 * pp.vec is a device copy of params[0 .. n_params-1] and pp.n = n_params.  The gradient may depend on the whole vector
 * only through the K functionals.  The source is compiled with NVRTC (bound at run time; ERR_UNSUPPORTED without it):
 * a contract check here (ERR_COMPILE with the log, lines numbered as `user_potential(<line>)`), the kernels when a
 * sampler is created.  pdmpflux_rv_diagnostic does not run it (no U value).
 *
 * Optional members declare the line model of the built-in plugins and put the potential on the fast-path kernels
 * (Zig-Zag x Brent, the Zig-Zag affine-cell grid bound, the BPS / ForwardECMC line sums); without them every sampler
 * runs the generic kernel:
 *
 *   static constexpr bool affine = true;  for every i >= special the Hessian is constant along the flow line:
 *                                         g_i(x + t v) = g_i(x) + t (H v)_i exactly, (H v)_i being the hd of eval
 *   static constexpr int special = 2;     0 <= special <= K, needs affine: L_k(x) = x_k for k < special (accum puts
 *                                         x_k, and nothing else, into acc[k]); these coordinates' rates are evaluated
 *                                         per time from the functionals
 *   __device__ static void eval_local(const pdmpflux::PotParams&, int i, double xi, double di, double& gl, double& hl);
 *   __device__ static void line_corr(const pdmpflux::PotParams&, const double* Lx, const double* Ld, double& ca, double& cb);
 *                                         both or neither, need affine and special = 0: gl, hl are the parts of g_i and
 *                                         (H d)_i that do not involve the functionals; ca = sum_i (g_i - gl_i) d_i and
 *                                         cb = sum_i ((H d)_i - hl_i) d_i, from the functionals alone
 *
 * A declaration that breaks one of these rules is an ERR_COMPILE naming the member.  Whether the potential really has
 * the declared structure cannot be checked, just as the linearity of accum cannot: a wrong declaration samples the
 * wrong target.  Boomerang keeps the generic kernel for a source (its fast path needs grad U(0) = 0, which affine does
 * not promise). */
int pdmpflux_potential_create_source(int dim, const char* source, const double* params, int64_t n_params,
                                     pdmpflux_potential_t* out);

/* replaces ZigZag(dim, grad U; kw...) / BPS / ForwardECMC / Boomerang constructors */
int pdmpflux_sampler_create(int sampler_kind, int dim, pdmpflux_potential_t pot, const pdmpflux_config* cfg,
                            pdmpflux_sampler_t* out);
/* replaces StickyZigZag(dim, grad U, kappa; kw...) (StickyZigZagSamplers.jl:60-111): Zig-Zag closures plus the
 * thawing rates kappa[dim] (prior inclusion).  Runs on the generic (per-node) path; sample_skeleton* then produce the
 * sticky skeleton (flips, stickings and thawings are all skeleton points, with the is_active column).  The
 * time-horizon variant is not available for it (PDMPFLUX_ERR_UNSUPPORTED). */
int pdmpflux_sampler_create_sticky(int dim, pdmpflux_potential_t pot, const pdmpflux_config* cfg, const double* kappa,
                                   pdmpflux_sampler_t* out);
int pdmpflux_sampler_destroy(pdmpflux_sampler_t s);
/* Ownership / threading of a sampler handle: the host-buffer pipeline of pdmpflux_sample_skeleton* caches its device
 * slabs, pinned staging buffers and copy stream in the handle (they only grow; one large call keeps up to ~10 GiB of
 * device memory until the handle is destroyed), so a handle must not be used by two host threads at once -- create one
 * sampler per thread (handles are cheap; the potential may be shared).  release_workspace frees the cached buffers
 * (synchronises the device); the next host-buffer call allocates them again. */
int pdmpflux_sampler_release_workspace(pdmpflux_sampler_t s);
/* the config after constructor rewrites */
int pdmpflux_sampler_get_config(pdmpflux_sampler_t s, pdmpflux_config* out);

/* replaces sample_skeleton(sampler, n_sk, xinit, vinit; seed) (src/sample.jl:253-284) for n_chains chains:
 * column 0 = initial state (t=0, horizon=tmax, ar=0), columns 1..n_sk-1 = successive accepted events
 * (init_state AbstractPDMP.jl:93-153 + get_event_state! SamplingLoopInplace.jl:27-217 + record!
 * Composites.jl:239-260).  xinit/vinit: d x n_chains column-major (host, or device when hist->on_device).
 * hist->n_cols must be >= n_sk.  Global chain id = chain_offset + c (multi-GPU sharding).
 * Returns PDMPFLUX_ERR_CHAIN if any chain stopped (outputs of healthy chains are still valid). */
int pdmpflux_sample_skeleton(pdmpflux_sampler_t s, int64_t n_chains, int64_t n_sk, const double* xinit,
                             const double* vinit, uint64_t seed, int64_t chain_offset,
                             const pdmpflux_tape* tape_or_null, const pdmpflux_history* hist, void* cuda_stream);

/* Same, continuing from a saved PDMPState instead of init_state: x/v as xinit/vinit, per-chain t0 and
 * horizon0 (NULL -> 0 / tmax) and the number of events already generated (Philox event index offset).
 * The last column of a previous history (X, V, t, horizon) is a complete checkpoint: the reference keeps
 * the final state in `sampler.state` (src/sample.jl:281) but offers no resume call. */
int pdmpflux_sample_skeleton_resume(pdmpflux_sampler_t s, int64_t n_chains, int64_t n_sk, const double* xinit,
                                    const double* vinit, const double* t0, const double* horizon0, int64_t event0,
                                    uint64_t seed, int64_t chain_offset, const pdmpflux_tape* tape_or_null,
                                    const pdmpflux_history* hist, void* cuda_stream);

/* replaces sample_skeleton(sampler, T::Float64, xinit, vinit; seed, init_capacity) (src/sample.jl:323-439): every
 * chain advances until time T; events with t <= T are recorded and the skeleton ends with the point at exactly
 * t = T reached by the deterministic flow (zeroed event statistics), so t[end] == T.  hist->n_cols >= capacity;
 * n_cols_out[c] = columns written for chain c (ragged).  Returns PDMPFLUX_ERR_CAPACITY when some chain has not
 * reached T within `capacity` columns (the first `capacity` columns of every chain are valid: grow and call again;
 * the reference grows its PDMPHistory by doubling, Composites.jl:172-191). */
int pdmpflux_sample_skeleton_until(pdmpflux_sampler_t s, int64_t n_chains, double T, int64_t capacity,
                                   const double* xinit, const double* vinit, uint64_t seed, int64_t chain_offset,
                                   const pdmpflux_tape* tape_or_null, const pdmpflux_history* hist,
                                   int64_t* n_cols_out, void* cuda_stream);

/* Streaming form of the same loop: device-resident PDMPState array (the analogue of `sampler.state`,
 * src/sample.jl:281) that can be advanced in slices; lets skeletons larger than HBM stream to the host.
 * Stream ordering: chains_create / set_state / enable_moments / get_* synchronise the device themselves (device
 * inputs produced on any stream are complete before they are read, and the set-up is complete before the call
 * returns), so chains_advance / chains_record may run on any stream, including cudaStreamNonBlocking ones. */
int pdmpflux_chains_create(pdmpflux_sampler_t s, int64_t n_chains, const double* xinit, const double* vinit,
                           int32_t init_on_device, uint64_t seed, int64_t chain_offset,
                           const pdmpflux_tape* tape_or_null, pdmpflux_chains_t* out);
/* overwrite / read the per-chain clock, horizon and event counter (resume, teacher-forced parity tests) */
int pdmpflux_chains_set_state(pdmpflux_chains_t ch, const double* t, const double* horizon, int64_t event0,
                              int32_t on_device);
int pdmpflux_chains_get_state(pdmpflux_chains_t ch, double* x, double* v, double* t, double* horizon,
                              int32_t on_device);
/* Fused moments (no reference equivalent; feeds moments / ESS without materialising a skeleton): after enabling,
 * every later chains_advance accumulates int x_i dt and int x_i^2 dt per chain and coordinate ([C][d]) inside the
 * flows (closed form per segment); chains_advance may then be called with a NULL history. */
int pdmpflux_chains_enable_moments(pdmpflux_chains_t ch);
int pdmpflux_chains_get_moments(pdmpflux_chains_t ch, double* m1, double* m2, int32_t on_device);
/* time-horizon mode for chains_advance: chains stop (status PDMPFLUX_CHAIN_DONE) at exactly t = T; NaN disables */
int pdmpflux_chains_set_stop_time(pdmpflux_chains_t ch, double T);
/* columns recorded so far per chain (host pointer, [C]) */
int pdmpflux_chains_get_ncols(pdmpflux_chains_t ch, int64_t* ncols);
/* generate n_events more events per chain; column j of this call goes to hist column col0 + j (device view) */
int pdmpflux_chains_advance(pdmpflux_chains_t ch, int64_t n_events, const pdmpflux_history* device_hist,
                            int64_t col0, void* cuda_stream);
/* write the current state as one history column (used for column 0) */
int pdmpflux_chains_record(pdmpflux_chains_t ch, const pdmpflux_history* device_hist, int64_t col,
                           void* cuda_stream);
/* copy per-chain status / tape positions / counters out (host pointers, any may be NULL); returns
 * PDMPFLUX_ERR_CHAIN if any status != 0 */
int pdmpflux_chains_status(pdmpflux_chains_t ch, int32_t* status, int64_t* tape_pos, int64_t* counters);
int pdmpflux_chains_destroy(pdmpflux_chains_t ch);

/* replaces sample_from_skeleton(sampler, N, history; discard_vt) (src/sample.jl:475-513), per chain:
 * out is [C][N][d] (or [C][N][2d+1]); flow_kind 0 = linear (ZigZag/BPS/FECMC), 1 = rotation (Boomerang),
 * 2 = the Speed-Up Zig-Zag flow (SpeedUpZigZagSamplers.jl:71-79). */
int pdmpflux_sample_from_skeleton(int flow_kind, int dim, int64_t n_sk, int64_t n_chains, const double* X,
                                  const double* V, const double* t, int64_t N, int32_t discard_vt, double* out,
                                  int32_t on_device, void* cuda_stream);

/* replaces sample_from_skeleton(sampler, dt::Float64, history) (src/sample.jl:573-646): samples at times j*dt,
 * j = 1..n_out with n_out = floor(t[end]/dt) computed by the caller; and, with n_sk < ld_sk, the (N, dt) method
 * (src/sample.jl:649-682) that only uses the first n_sk columns of slabs whose leading dimension is ld_sk.
 * All chains must share n_out (pass chains one at a time for ragged skeletons). */
/* replaces sample_from_skeleton(sampler::StickyPDMP, N, history) (src/sample.jl:516-561): the reconstructed velocity of
 * a frozen coordinate is zero.  is_active: [C][n_sk][d] bytes as written by the sticky skeleton (NULL: all active). */
int pdmpflux_sample_from_skeleton_sticky(int dim, int64_t n_sk, int64_t n_chains, const double* X, const double* V,
                                         const double* t, const uint8_t* is_active, int64_t N, int32_t discard_vt,
                                         double* out, int32_t on_device, void* cuda_stream);

int pdmpflux_sample_from_skeleton_dt(int flow_kind, int dim, int64_t n_sk, int64_t ld_sk, int64_t n_chains,
                                     const double* X, const double* V, const double* t, double dt, int64_t n_out,
                                     int32_t discard_vt, double* out, int32_t on_device, void* cuda_stream);

/* Closed-form time integrals over each chain's skeleton (no reference equivalent; feeds moments / ESS,
 * SURVEY.md 8d): m1[C][d] = int x_i dt, m2[C][d] = int x_i^2 dt over [t[col_begin], t[n_sk-1]], T[C] = length. */
int pdmpflux_skeleton_moments(int flow_kind, int dim, int64_t n_sk, int64_t n_chains, int64_t col_begin,
                              const double* X, const double* V, const double* t, double* m1, double* m2,
                              double* T, int32_t on_device, void* cuda_stream);

/* Cross-chain sufficient statistics of the per-chain time integrals (one fused kernel; SURVEY.md 8d/8e -- the
 * reference has no ESS estimator): with m_c = m1[c] / T[c] and s_c = m2[c] / T[c] (T == NULL: already time averages),
 * sums[0][i] = sum_c m_c[i], sums[1][i] = sum_c m_c[i]^2, sums[2][i] = sum_c s_c[i], sums[3][i] = n_chains.
 * Summation order is fixed (bitwise reproducible).  Pooled mean / variance and the cross-chain ESS follow from the
 * sums after they have been added over ranks: ESS_i = C Var_pi(x_i) / Var_c(m_c[i]). */
int pdmpflux_moments_reduce(int dim, int64_t n_chains, const double* m1, const double* m2, const double* T,
                            double* sums /* [4][dim] */, int32_t on_device, void* cuda_stream);

/* The only collective of the path: sum the moment statistics over the GPUs of a job (NCCL over NVLink).  The library
 * owns the communicator; the host only moves the 128-byte unique id from rank 0 to the other ranks (MPI / sockets /
 * torch.distributed -- any transport).  NCCL is bound at run time (libnccl.so.2); without it comm_create with
 * n_ranks > 1 returns PDMPFLUX_ERR_UNSUPPORTED.  n_ranks == 1 needs no NCCL and allreduce is a no-op. */
#define PDMPFLUX_COMM_ID_BYTES 128
typedef struct pdmpflux_comm_s* pdmpflux_comm_t;
int pdmpflux_comm_unique_id(void* id_out, size_t bytes);           /* rank 0: ncclGetUniqueId */
int pdmpflux_comm_create(const void* unique_id, int n_ranks, int rank, pdmpflux_comm_t* out); /* after set_device */
int pdmpflux_comm_destroy(pdmpflux_comm_t comm);
/* in-place sum over ranks of `n` doubles in device memory, enqueued on cuda_stream */
int pdmpflux_moments_allreduce(pdmpflux_comm_t comm, double* device_sums, int64_t n, void* cuda_stream);

/* replaces RV_diagnostic(history, U; B) (src/diagnostic.jl:37-75) for a batch of skeletons: rv[c] = sum over B blocks
 * of (U(x(t_b)) - U(x(t_{b-1})))^2 / t[end], positions by the linear interpolation of _history_position_linear!
 * (src/diagnostic.jl:23-35) when flow_kind = 0; flow_kind = 1 interpolates with the Boomerang rotation, which is what
 * the online sample_skeleton_with_diagnostic (src/sample.jl:75-236) accumulates through sampler.flow.  U is the value
 * plugin of `pot` (Gaussians, banana, logistic regression).  X, V: [C][ld_sk][d],
 * t: [C][ld_sk]; chain c uses its first ncols[c] columns (ncols == NULL: n_sk for all).  B = 0 -> floor(sqrt(n)) like
 * the reference, B < 0 -> PDMPFLUX_ERR_ARGUMENT (the reference's ArgumentError).  A chain whose t[end] is negative or
 * not finite gets rv = NaN (the binding raises the reference's ArgumentError). */
int pdmpflux_rv_diagnostic(pdmpflux_potential_t pot, int flow_kind, int64_t n_sk, int64_t ld_sk, int64_t n_chains,
                           const int64_t* ncols, int64_t B, const double* X, const double* V, const double* t,
                           double* rv, int32_t on_device, void* cuda_stream);

/* pinned host memory for the host-buffer (end-to-end) path */
int pdmpflux_host_alloc(void** ptr, size_t bytes);
int pdmpflux_host_free(void* ptr);

/* number of kernel launches issued by this library in this process (bench.py's gpu_launches) */
int64_t pdmpflux_launch_count(void);
/* number of NVRTC compiles of source potentials in this process (contract checks and kernels; cached ones not counted) */
int64_t pdmpflux_jit_compile_count(void);

/* bytes that crossed PCIe in the last host-buffer sample_skeleton call of this process (initial states in; history
 * out -- for Zig-Zag the V rows travel as sign bits and are rebuilt on the host, so this is less than the size of
 * the history).  bench.py's e2e.{h2d,d2h}_bytes_per_step. */
int pdmpflux_last_transfer_bytes(int64_t* h2d, int64_t* d2h);
#endif /* __CUDACC_RTC__ */

#ifdef __cplusplus
}
#endif
#endif /* PDMPFLUX_CUDA_H */
