// C ABI of libpdmpflux_cuda.so (see include/pdmpflux_cuda.h).  Host orchestration only: handles, argument
// validation mirroring the reference constructors / drivers, kernel dispatch, and the host-buffer pipeline
// (device double buffering + pinned D2H copies overlapped with the next slice of events).
//
// There is no CPU fallback anywhere in this file: without a usable CUDA device every compute entry point
// returns PDMPFLUX_ERR_CUDA.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <thread>
#include <vector>
#if defined(__linux__)
#include <sched.h>
#endif
#if defined(__x86_64__)
#include <emmintrin.h>
#endif

#include "common.cuh"
#include "jit.cuh"
#include "launch.cuh"

using namespace pdmpflux;

namespace {

thread_local std::string g_err;
std::atomic<int64_t> g_launches{0};
std::atomic<int64_t> g_h2d_bytes{0}, g_d2h_bytes{0};  // PCIe bytes of the last host-buffer sample_skeleton call

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
#define CUDA_TRY(expr)                                                                            \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess)                                                                    \
            return fail(PDMPFLUX_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));   \
    } while (0)

struct DevBuf {  // RAII device allocation
    void* p = nullptr;
    size_t bytes = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t n) {
        if (p) { cudaFree(p); p = nullptr; }
        bytes = n;
        if (n == 0) return cudaSuccess;
        return cudaMalloc(&p, n);
    }
    template <class T> T* as() const { return static_cast<T*>(p); }
};

}  // namespace

// used by the other translation units (reduce.cu)
int pdmpflux_fail_(int code, const std::string& msg) { return fail(code, msg); }
void pdmpflux_count_launch_() { g_launches.fetch_add(1); }

struct pdmpflux_potential_s {
    int kind = 0, dim = 0;
    PotParams pp{};
    DevBuf params;
    std::string source;  // PDMPFLUX_SOURCE: the user's CUDA text (jit.cu)
    SourceTraits traits; // PDMPFLUX_SOURCE: the line model it declares (read by the contract check)
};

// Device slabs of the host-buffer pipeline, cached in the sampler handle so that repeated sample_skeleton calls do
// not pay cudaMalloc / cudaFree (which also synchronise the device) every time.
struct Slab {
    DevBuf X, V, t, horizon, ar, eva, eb, rej, hh;
    pdmpflux_history view{};
    cudaEvent_t done = nullptr, copied = nullptr;
    ~Slab() {
        if (done) cudaEventDestroy(done);
        if (copied) cudaEventDestroy(copied);
    }
};
struct Workspace {
    Slab slab[2];
    Slab scal;  // full-length scalar columns (t, horizon, ar, error_value_ar, counters) of the host pipeline
    cudaStream_t copy_stream = nullptr;
    // Zig-Zag host path: sign bits of every V row of the run, [slice][chain][column in slice][words], device + pinned host
    DevBuf vbits;
    uint32_t* vbits_host = nullptr;
    size_t vbits_host_bytes = 0;
    std::vector<cudaEvent_t> slice_copied;  // one event per slice: its sign bits have reached the host
    DevBuf zflags;                          // per slice: errored_bound (hence error_value_ar) has a non-zero entry
    int* zflags_host = nullptr;
    size_t zflags_host_n = 0;
    ~Workspace() {
        if (copy_stream) cudaStreamDestroy(copy_stream);
        if (vbits_host) cudaFreeHost(vbits_host);
        if (zflags_host) cudaFreeHost(zflags_host);
        for (cudaEvent_t e : slice_copied) cudaEventDestroy(e);
    }
};

struct pdmpflux_sampler_s {
    int kind = 0, dim = 0;
    pdmpflux_config cfg{};
    pdmpflux_potential_s* pot = nullptr;
    DevBuf kappa;  // Sticky Zig-Zag: thawing rates [dim]
    Workspace ws;
};

struct pdmpflux_chains_s {
    pdmpflux_sampler_s* s = nullptr;
    int64_t n_chains = 0, chain_offset = 0, event0 = 0;
    uint64_t seed = 0;
    int team = 32, n_own = 0, scratch_in_smem = 1, path = 0, vec_elems = 0, dpad = 0;
    int brent_nw = kLineShared;   // Zig-Zag x Brent line model (brent_line_model), fixed when the chains are created
    size_t smem = 0;
    unsigned grid = 0;
    int64_t n_groups = 0;   // groups of chains (one block's worth); grid < n_groups: persistent blocks walk over the groups
    DevBuf x, v, t, horizon, ar, tape_pos, status, counters, scratch, ncols, m1, m2, wq, act;
    int moments = 0;
    double t_stop = 0.0;
    int use_t_stop = 0;
    // draws
    int draw_mode = 1;
    DevBuf tE, tU, tN;  // owned device copies when the tape was given on the host
    const double *dE = nullptr, *dU = nullptr, *dN = nullptr;
    int64_t nE = 0, nU = 0, nN = 0;
};

namespace {

// Team widths built: 1, 8, 32 (launch.cuh: launch_for_sampler).
int default_team(int d, int64_t n_chains, bool zz_brent_fast);
int pick_team(int d, int64_t n_chains, bool zz_brent_fast) {
    if (const char* e = std::getenv("PDMPFLUX_TEAM")) {
        // only a width with a kernel for this shape: thread-per-chain Zig-Zag x Brent packs coordinate indices into 6
        // bits (chain.cuh: classify_line), so it is built for d <= 64 (widen_team's shared-memory budget already widens
        // it above d = 55; this check does not depend on that budget)
        const int t = std::atoi(e);
        if (t == 8 || t == 32 || (t == 1 && !(zz_brent_fast && d > 64))) return t;
    }
    return default_team(d, n_chains, zz_brent_fast);
}
int default_team(int d, int64_t n_chains, bool zz_brent_fast) {
    // Measured on B200 (profiles/): thread-per-chain wins for small d once there are enough chains to occupy the
    // SMs; 8 lanes per chain win for d up to a few hundred (fewer shuffle stages than a full warp, 4 chains share a
    // warp's instruction stream); a warp per chain beyond that (and whenever the shared-memory state would not fit).
    if (d <= 16) return n_chains >= 8192 ? 1 : 8;
    // Zig-Zag x Brent: the rate function is compressed per bracket to one line plus the few sign-changing coordinates
    // (chain.cuh: classify_line).  With a chain per thread the serial Brent recurrence runs without any cross-lane
    // reduction and 32 chains share every instruction: 4.9e8 events/s at 16384 chains, 9e8 at 65536 (banana d = 50).
    // Below ~10k chains there are too few warps for that, and teams of 8 running the transposed search (each lane its
    // own iterations, one pass per bound) are ahead: 3.1e8 at 4096 and at 8192 chains against 2.5e8 thread-per-chain
    // at 8192.
    if (zz_brent_fast && d <= 64 && n_chains >= 10240) return 1;
    // (A chain per thread does NOT pay for BPS / Boomerang at d ~ 100 -- measured 1.1e8 events/s against 3.4e8 with
    // teams of 8 on BASELINE config 3: a refresh draws d normals, and with 32 chains per warp some lane refreshes in
    // almost every event, so the whole warp pays the d-normal pass every time.)
    if (d <= 256) return 8;
    return 32;
}

// widen the team until the per-thread-owned shared-memory columns of a block (x, v, Zig-Zag x Brent A / B, moments,
// sticky flags; ForwardECMC scratch goes to global memory when it is large) leave room for a second block
int widen_team(int team, int sampler, int path, int d) {
    auto vectors_bytes = [&](int team) {
        const int bt_ = block_threads_rt(team, sampler, path);
        const int n_own = (d + team - 1) / team;
        const size_t nv = state_vectors(sampler, path, team, brent_line_model(sampler, path, team, n_own));
        return (nv + 2 /* fused moments may be enabled later */ + (sampler == PDMPFLUX_STICKY_ZIGZAG ? 1 : 0)) *
               (size_t)n_own * bt_ * sizeof(double);
    };
    while (team < 32 && vectors_bytes(team) > 110 * 1024) team = team < 8 ? 8 : 32;
    return team;
}

// the line-model traits select_path sees for this sampler: a built-in kind's Pot<> traits, a source's declared ones.
// Boomerang keeps a source on the generic kernel: its fast path takes <grad U(x), x> as <P x, x>, which holds only when
// grad U(0) = 0 -- true of every built-in, not promised by an affine declaration (a Gaussian with a non-zero mean).
LineTraits line_traits(int sampler, const pdmpflux_potential_s* pot) {
    if (pot->kind != PDMPFLUX_SOURCE) return builtin_line_traits(pot->kind);
    if (sampler == PDMPFLUX_BOOMERANG) return {};
    return {pot->traits.affine, pot->traits.special};
}

// The kernel variant that n_chains chains of a sampler run: path, team width and Zig-Zag x Brent line model.
// with_env: honour PDMPFLUX_FORCE_GENERIC and PDMPFLUX_TEAM (pdmpflux_chains_create); without: the default policy,
// which is what sampler creation compiles ahead for a source potential.
struct Variant { int path, team, n_own, nw; };
Variant chain_variant(int kind, int dim, const pdmpflux_config& cfg, const pdmpflux_potential_s* pot, int64_t n_chains,
                      bool with_env) {
    Variant v{};
    v.path = select_path(kind, line_traits(kind, pot), cfg.grid_size, cfg.vectorized_bound, cfg.deriv_mode);
    if (const char* e = with_env ? std::getenv("PDMPFLUX_FORCE_GENERIC") : nullptr) { if (std::atoi(e)) v.path = kPathGeneric; }
    const bool zz_brent_fast = kind == PDMPFLUX_ZIGZAG && v.path == kPathFastBrent && pot->kind != PDMPFLUX_LOGREG;
    const int team = with_env ? pick_team(dim, n_chains, zz_brent_fast) : default_team(dim, n_chains, zz_brent_fast);
    v.team = widen_team(team, kind, v.path, dim);
    v.n_own = (dim + v.team - 1) / v.team;
    v.nw = brent_line_model(kind, v.path, v.team, v.n_own);
    return v;
}

// `rows`: optional separate placement of the X / V rows (host pipeline: rows go through narrow double-buffered
// slabs while the scalar columns accumulate in full-length device buffers)
struct RowsView { double *X, *V; int64_t ld, col0; };

int launch(pdmpflux_chains_s* ch, int64_t n_events, const pdmpflux_history* h, int64_t col0, cudaStream_t stream,
           const RowsView* rows = nullptr) {
    const pdmpflux_sampler_s* s = ch->s;
    const pdmpflux_config& c = s->cfg;
    KernelParams p{};
    p.d = s->dim; p.G = c.grid_size; p.vectorized = c.vectorized_bound; p.signed_bound = c.signed_bound;
    p.adaptive = c.adaptive; p.deriv_mode = c.deriv_mode; p.gaussian_velocity = c.gaussian_velocity;
    p.ran_p = c.ran_p; p.switch_ = c.switch_; p.positive = c.positive;
    p.max_steps = c.max_steps > 0 ? c.max_steps : 100000;
    p.tmax = c.tmax; p.refresh_rate = c.refresh_rate;
    p.bound_refresh = c.signed_bound ? c.refresh_rate : 0.0;  // AbstractPDMP.jl:104-112
    p.mix_p = c.mix_p; p.speed_factor = c.speed_factor;
    p.inv_gm1 = c.grid_size > 1 ? 1.0 / (double)(c.grid_size - 1) : 0.0;
    p.pot = s->pot->pp;
    p.n_chains = ch->n_chains; p.chain_offset = ch->chain_offset; p.seed = ch->seed;
    p.n_groups = ch->n_groups;
    p.event0 = ch->event0; p.n_events = n_events;
    p.sx = ch->x.as<double>(); p.sv = ch->v.as<double>(); p.st = ch->t.as<double>();
    p.shorizon = ch->horizon.as<double>(); p.sar = ch->ar.as<double>();
    p.tape_pos = ch->tape_pos.as<int64_t>(); p.status = ch->status.as<int32_t>();
    p.counters = ch->counters.as<int64_t>();
    p.ncols = ch->ncols.as<int64_t>();
    p.use_t_stop = ch->use_t_stop; p.t_stop = ch->t_stop;
    p.accumulate_moments = ch->moments; p.M1 = ch->m1.as<double>(); p.M2 = ch->m2.as<double>();
    p.draw_mode = ch->draw_mode; p.tE = ch->dE; p.tU = ch->dU; p.tN = ch->dN;
    p.nE = ch->nE; p.nU = ch->nU; p.nN = ch->nN;
    if (h) {
        p.X = h->X; p.V = h->V; p.T = h->t; p.H = h->horizon; p.AR = h->ar; p.EVA = h->error_value_ar;
        p.EB = h->errored_bound; p.REJ = h->rejected; p.HH = h->hitting_horizon;
        p.ld_cols = h->n_cols;
        p.ld_rows = h->n_cols; p.col0_rows = col0;
        if (rows) { p.X = rows->X; p.V = rows->V; p.ld_rows = rows->ld; p.col0_rows = rows->col0; }
    }
    p.col0 = col0;
    p.kappa = s->kappa.as<double>(); p.sact = ch->act.as<uint8_t>(); p.ACT = h ? h->is_active : nullptr;
    p.scratch = ch->scratch.as<double>(); p.scratch_in_smem = ch->scratch_in_smem; p.n_own = ch->n_own;
    p.brent_nw = ch->brent_nw;
    p.vec_elems = ch->vec_elems; p.dpad = ch->dpad;
    if (h) {
        auto al = [](const void* q, uintptr_t a) { return q == nullptr || (reinterpret_cast<uintptr_t>(q) % a) == 0; };
        p.vec32 = al(p.X, 32) && al(p.V, 32) && al(h->t, 32) && al(h->horizon, 32) && al(h->ar, 32);
        p.bulk_rows = ch->team > 1 && (s->dim % 2 == 0) && al(p.X, 16) && al(p.V, 16);
        if (const char* e = std::getenv("PDMPFLUX_NO_BULK")) { if (std::atoi(e)) { p.bulk_rows = 0; p.vec32 = 0; } }
        // Diagnostic columns that are almost always zero are zero-filled here (one strided fill each) and the
        // kernel writes only their non-zero entries.
        p.sparse_cols = 1;
        const int64_t ncols = n_events > 0 ? n_events : 1;
        auto fill = [&](void* base, size_t elem) -> cudaError_t {
            if (!base) return cudaSuccess;
            char* q = static_cast<char*>(base) + (size_t)col0 * elem;
            if (ncols == h->n_cols) return cudaMemsetAsync(q, 0, (size_t)ch->n_chains * ncols * elem, stream);
            return cudaMemset2DAsync(q, (size_t)h->n_cols * elem, 0, (size_t)ncols * elem, (size_t)ch->n_chains, stream);
        };
        cudaError_t fe = fill(h->error_value_ar, 5 * sizeof(double));
        if (fe == cudaSuccess) fe = fill(h->errored_bound, sizeof(int32_t));
        if (fe == cudaSuccess) fe = fill(h->rejected, sizeof(int32_t));
        if (fe == cudaSuccess) fe = fill(h->hitting_horizon, sizeof(int32_t));
        if (fe != cudaSuccess) return fail(PDMPFLUX_ERR_CUDA, std::string("zero-fill of diagnostic columns: ") + cudaGetErrorString(fe));
    }
    cudaError_t e;
    const size_t smem_launch = ch->smem + (ch->moments ? 2 * (size_t)ch->vec_elems * sizeof(double) : 0);
    if (smem_launch > 227 * 1024) return fail(PDMPFLUX_ERR_UNSUPPORTED, "fused moments: shared memory exhausted for this dimension");
    if (s->pot->kind == PDMPFLUX_SOURCE) {
        const int rc = jit_launch(s->pot->source, s->kind, ch->team, ch->path, ch->brent_nw, p, ch->grid, smem_launch, stream);
        if (rc != PDMPFLUX_OK) return rc;
        e = cudaSuccess;
    } else if (s->pot->kind == PDMPFLUX_LOGREG) {
        p.vec32 = 0; p.bulk_rows = 0;
        // One CTA per SM (384 threads, 168 registers): with more CTAs of four chains than SMs, the first wave starts on
        // chains 0 .. 4 grid - 1 and every warp pulls its next chain from a work queue when its own is done.
        unsigned grid = ch->grid;
        p.work_counter = nullptr; p.work_start = 0;
        if (n_events > 0 && ch->wq.p) {
            static int n_sm = 0;
            if (n_sm == 0) {
                int dev = 0;
                cudaGetDevice(&dev);
                if (cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n_sm <= 0) n_sm = 148;
            }
            grid = std::min<unsigned>(grid, (unsigned)n_sm);
            p.work_counter = ch->wq.as<int64_t>();
            p.work_start = (int64_t)grid * logreg_chains_per_block();
            CUDA_TRY(cudaMemsetAsync(ch->wq.p, 0, sizeof(int64_t), stream));
        }
        e = launch_logreg_zigzag(p, grid, ch->smem, stream);
    } else
    switch (s->kind) {
    case PDMPFLUX_ZIGZAG: e = launch_skeleton_zigzag(ch->team, s->pot->kind, ch->path, p, ch->grid, smem_launch, stream); break;
    case PDMPFLUX_BPS: e = launch_skeleton_bps(ch->team, s->pot->kind, ch->path, p, ch->grid, smem_launch, stream); break;
    case PDMPFLUX_FECMC: e = launch_skeleton_fecmc(ch->team, s->pot->kind, ch->path, p, ch->grid, smem_launch, stream); break;
    case PDMPFLUX_BOOMERANG: e = launch_skeleton_boomerang(ch->team, s->pot->kind, ch->path, p, ch->grid, smem_launch, stream); break;
    case PDMPFLUX_STICKY_ZIGZAG: e = launch_skeleton_sticky(ch->team, s->pot->kind, ch->path, p, ch->grid, smem_launch, stream); break;
    case PDMPFLUX_SPEEDUP_ZIGZAG: e = launch_skeleton_speedup(ch->team, s->pot->kind, ch->path, p, ch->grid, smem_launch, stream); break;
    default: e = cudaErrorInvalidValue;
    }
    if (e != cudaSuccess) return fail(PDMPFLUX_ERR_CUDA, std::string("skeleton kernel launch: ") + cudaGetErrorString(e));
    g_launches.fetch_add(1);
    return PDMPFLUX_OK;
}

// errored_bound is zero for (almost) every event, and error_value_ar is zero wherever it is: one flag per slice tells the
// host path that both columns of the slice are all zero, so they need not cross PCIe (the host zero-fills its rows).
__global__ void __launch_bounds__(256) flag_nonzero_kernel(const int32_t* __restrict__ eb, int64_t n_chains, int64_t ld,
                                                           int64_t k0, int64_t n, int* __restrict__ flag) {
    bool any = false;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n_chains * n; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t c = e / n, k = e - c * n;
        any |= eb[c * ld + k0 + k] != 0;
    }
    if (__any_sync(0xffffffffu, any) && (threadIdx.x & 31) == 0) atomicOr(flag, 1);
}

// Zig-Zag velocities never change magnitude (ZigZagSamplers.jl:101-107 only flips signs), so on the host-buffer path a
// V row of d doubles crosses PCIe as d sign bits and is rebuilt bit-exactly on the host as copysign(|vinit_i|, bit).
// One warp per (chain, column) row: coalesced reads, one ballot per 32 coordinates.  bits: [chain][slab column][words].
__global__ void __launch_bounds__(256) pack_signs_kernel(const double* __restrict__ V, int d, int64_t n_chains, int64_t n,
                                                         int64_t ld, int words, uint32_t* __restrict__ bits) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp0; r < n_chains * n; r += nwarps) {
        const int64_t c = r / n, k = r - c * n;
        const double* row = V + (c * ld + k) * d;
        for (int wd = 0; wd < words; ++wd) {
            const int i = 32 * wd + lane;
            const bool neg = i < d && (__double2hiint(row[i]) < 0);
            const uint32_t m = __ballot_sync(0xffffffffu, neg);
            if (lane == 0) bits[(c * ld + k) * words + wd] = m;
        }
    }
}

// ---- sample_from_skeleton (src/sample.jl:475-513) -------------------------------------------------------
// One thread per output element (sample j, coordinate a) of one chain; neighbouring threads share j, so the
// binary search over the chain's event times is a broadcast and X/V/out accesses are coalesced.
// `dt_fixed > 0`: the dt method (src/sample.jl:573-646), sample times j * dt_fixed; otherwise dt = t[end] / N (:475-513).
// `ld_sk` is the leading dimension of the history slabs (>= n_sk: the (N, dt) method uses the first n_sk columns).
__global__ void __launch_bounds__(256) interp_kernel(int flow_kind, int d, int64_t n_sk, int64_t ld_sk, int64_t N,
                                                     int discard_vt, double dt_fixed, const double* __restrict__ X,
                                                     const double* __restrict__ V, const double* __restrict__ T,
                                                     const uint8_t* __restrict__ act, const double* __restrict__ su,
                                                     double* __restrict__ out) {
    const int64_t c = blockIdx.x;  // chains on grid.x (up to 2^31 - 1), output elements grid-strided over grid.y
    const double* t = T + c * ld_sk;
    const double dt = dt_fixed > 0.0 ? dt_fixed : t[n_sk - 1] / (double)N;
    const int ld = discard_vt ? d : 2 * d + 1;
    const int64_t total = N * (int64_t)ld;
    for (int64_t e = (int64_t)blockIdx.y * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.y * blockDim.x) {
        const int64_t j = e / ld;
        const int a = (int)(e - j * ld);
        const double tm = (double)(j + 1) * dt;
        // largest i with t[i] <= tm (the reference's monotone pointer walk `while t[i+1] <= tm`)
        int64_t lo = 0, hi = n_sk - 1;
        while (lo < hi) {
            const int64_t mid = (lo + hi + 1) >> 1;
            if (t[mid] <= tm) lo = mid; else hi = mid - 1;
        }
        const double tau = tm - t[lo];
        const double* x0 = X + (c * ld_sk + lo) * d;
        const double* v0 = V + (c * ld_sk + lo) * d;
        double r;
        if (a == 2 * d) r = tm;
        else {
            const int b = a < d ? a : a - d;
            // Sticky samplers (src/sample.jl:516-561): the reconstructed velocity of a frozen coordinate is zero
            const double xi = x0[b], vi = (act && !act[(c * ld_sk + lo) * d + b]) ? 0.0 : v0[b];
            if (flow_kind == 1) {
                double s, co;
                sincos(tau, &s, &co);
                r = a < d ? xi * co + vi * s : -xi * s + vi * co;
            } else if (flow_kind == 2) {  // SpeedUpZigZagSamplers.jl:71-79 from the segment scalars (speedup_scalars_kernel)
                const double* sc = su + (c * ld_sk + lo) * 4;   // <y,y>, <y,v>, v1 x1, v1
                const double dd = (double)d, vx1 = sc[2], v1 = sc[3], cc = v1 * sc[1];
                const double aa = (1 + sc[0]) / dd - (cc * cc) / (dd * dd), Y0 = v1 * vx1 + cc / dd;   // x1 = v1 (v1 x1)
                const double bt = (Y0 + sqrt(Y0 * Y0 + aa)) * exp(sqrt(dd) * v1 * tau);
                const double X1 = (bt * bt - aa) / (2 * bt) - cc / dd;
                r = a < d ? (xi - vx1 * vi) + v1 * X1 * vi : vi;
            } else r = a < d ? xi + vi * tau : vi;
        }
        out[(c * N + j) * ld + a] = r;
    }
}

// Speed-Up Zig-Zag: the four scalars of a skeleton point that fix its flow (y = x - v1 x1 v): <y,y>, <y,v>, v1 x1, v1.
// One warp per (chain, column).
__global__ void __launch_bounds__(256) speedup_scalars_kernel(int d, int64_t n_rows, const double* __restrict__ X,
                                                              const double* __restrict__ V, double* __restrict__ su) {
    const int lane = threadIdx.x & 31;
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= n_rows) return;
    const double* x = X + r * d;
    const double* v = V + r * d;
    const double v1 = v[0], vx1 = v[0] * x[0];
    double yy = 0.0, yv = 0.0;
    for (int i = lane; i < d; i += 32) {
        const double y = x[i] - vx1 * v[i];
        yy += y * y; yv += y * v[i];
    }
    for (int o = 16; o > 0; o >>= 1) { yy += __shfl_xor_sync(0xffffffffu, yy, o); yv += __shfl_xor_sync(0xffffffffu, yv, o); }
    if (lane == 0) { su[r * 4] = yy; su[r * 4 + 1] = yv; su[r * 4 + 2] = vx1; su[r * 4 + 3] = v1; }
}

// Closed-form time integrals of x_i and x_i^2 along each chain's piecewise flow (feeds moments / ESS).
// One thread per (chain, coordinate) sums its segments in event order.  The pass streams X and V once (3.3 GB at
// the bench shape), so what bounds it is the bytes in flight: the event loop is unrolled by kMomU and the loads of a
// whole batch are issued before its arithmetic, and the linear flow keeps 6 blocks per SM (40 registers) so the
// 800 blocks of the bench shape (4096 chains x d = 50) fit in one wave instead of leaving a 60-block tail (the
// rotation flow's sincos needs more registers: 4 blocks).
constexpr int kMomU = 4;
template <int FLOW>
__device__ __forceinline__ void moment_segment(double tau, double x, double v, double& s1, double& s2) {
    if constexpr (FLOW == 1) {
        double s, co;
        sincos(tau, &s, &co);
        const double s2t = 2.0 * s * co;  // sin(2 tau)
        s1 += x * s + v * (1.0 - co);
        s2 += x * x * (0.5 * tau + 0.25 * s2t) + v * v * (0.5 * tau - 0.25 * s2t) + x * v * s * s;
    } else {
        s1 += tau * (x + 0.5 * v * tau);
        s2 += tau * (x * x + tau * (x * v + v * v * tau * (1.0 / 3.0)));
    }
}
template <int FLOW>
__global__ void __launch_bounds__(256, FLOW == 1 ? 4 : 6) moments_kernel(int d, int64_t n_sk, int64_t n_chains, int64_t col_begin,
                                                         const double* __restrict__ X, const double* __restrict__ V,
                                                         const double* __restrict__ T, double* __restrict__ m1,
                                                         double* __restrict__ m2, double* __restrict__ Tlen) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_chains * d) return;
    const int64_t c = e / d;
    const int a = (int)(e - c * d);
    const double* t = T + c * n_sk;
    const double* tp = t + col_begin;
    const double* xp = X + (c * n_sk + col_begin) * d + a;
    const double* vp = V + (c * n_sk + col_begin) * d + a;
    double s1 = 0.0, s2 = 0.0;
    int64_t n = n_sk - 1 - col_begin;   // segments left
    for (; n >= kMomU; n -= kMomU, tp += kMomU, xp += kMomU * d, vp += kMomU * d) {
        double tk[kMomU + 1], x[kMomU], v[kMomU];
#pragma unroll
        for (int i = 0; i <= kMomU; ++i) tk[i] = tp[i];
#pragma unroll
        for (int i = 0; i < kMomU; ++i) { x[i] = xp[i * d]; v[i] = vp[i * d]; }
#pragma unroll
        for (int i = 0; i < kMomU; ++i) moment_segment<FLOW>(tk[i + 1] - tk[i], x[i], v[i], s1, s2);
    }
    for (; n > 0; --n, ++tp, xp += d, vp += d) moment_segment<FLOW>(tp[1] - tp[0], *xp, *vp, s1, s2);
    m1[e] = s1;
    m2[e] = s2;
    if (a == 0 && Tlen) Tlen[c] = t[n_sk - 1] - t[col_begin];
}

int normalise_config(int kind, int dim, pdmpflux_config& c) {
    // constructor rewrites: ZigZagSamplers.jl:73-78, BouncyParticleSamplers.jl:29-37,
    // ForwardEventChainMonteCarlo.jl:306-323, BoomerangSamplers.jl:27-36
    if (c.tmax == 0.0) { c.tmax = 1.0; c.adaptive = 1; }
    if (kind == PDMPFLUX_ZIGZAG || kind == PDMPFLUX_STICKY_ZIGZAG || kind == PDMPFLUX_SPEEDUP_ZIGZAG) {
        if (c.signed_bound && !c.vectorized_bound) c.signed_bound = 0;
    } else c.vectorized_bound = 0;
    if (kind == PDMPFLUX_FECMC) {
        c.refresh_rate = 0.0;
        if (dim == 2) c.mix_p = 0.0;
    }
    return 0;
}

}  // namespace

extern "C" {
#pragma GCC visibility push(default)

int pdmpflux_version(void) { return PDMPFLUX_VERSION; }
const char* pdmpflux_last_error(void) { return g_err.c_str(); }
int64_t pdmpflux_launch_count(void) { return g_launches.load(); }
int64_t pdmpflux_jit_compile_count(void) { return jit_compile_count(); }
int pdmpflux_last_transfer_bytes(int64_t* h2d, int64_t* d2h) {
    if (h2d) *h2d = g_h2d_bytes.load();
    if (d2h) *d2h = g_d2h_bytes.load();
    return PDMPFLUX_OK;
}

int pdmpflux_device_count(int* count) {
    if (!count) return fail(PDMPFLUX_ERR_ARGUMENT, "count is NULL");
    *count = 0;
    CUDA_TRY(cudaGetDeviceCount(count));
    return PDMPFLUX_OK;
}
int pdmpflux_set_device(int device) {
    CUDA_TRY(cudaSetDevice(device));
    return PDMPFLUX_OK;
}

int pdmpflux_potential_create(int kind, int dim, const double* params, int64_t n_params, pdmpflux_potential_t* out) {
    if (!out) return fail(PDMPFLUX_ERR_ARGUMENT, "out is NULL");
    *out = nullptr;
    if (dim <= 0) return fail(PDMPFLUX_ERR_ARGUMENT, "dimension dim must be positive. Current value: " + std::to_string(dim));
    auto pot = new pdmpflux_potential_s();
    pot->kind = kind; pot->dim = dim;
    auto need = [&](int64_t n) { return params != nullptr && n_params >= n; };
    int rc = PDMPFLUX_OK;
    switch (kind) {
    case PDMPFLUX_GAUSS_STD: break;
    case PDMPFLUX_BANANA:
    case PDMPFLUX_BANANA_README_SCALAR:
        if (dim < 2) rc = fail(PDMPFLUX_ERR_ARGUMENT, "banana potentials need dim >= 2");
        break;
    case PDMPFLUX_GAUSS_DIAG:
        if (!need(dim)) { rc = fail(PDMPFLUX_ERR_ARGUMENT, "GAUSS_DIAG needs dim precisions"); break; }
        if (pot->params.alloc(sizeof(double) * dim) != cudaSuccess ||
            cudaMemcpy(pot->params.p, params, sizeof(double) * dim, cudaMemcpyHostToDevice) != cudaSuccess)
            rc = fail(PDMPFLUX_ERR_CUDA, "GAUSS_DIAG parameter upload failed (is a CUDA device present?)");
        pot->pp.vec = pot->params.as<double>();
        break;
    case PDMPFLUX_GAUSS_EQUICORR: {
        if (!need(1)) { rc = fail(PDMPFLUX_ERR_ARGUMENT, "GAUSS_EQUICORR needs rho"); break; }
        const double rho = params[0];
        if (!(rho < 1.0) || !(1.0 - rho + dim * rho > 0.0)) { rc = fail(PDMPFLUX_ERR_ARGUMENT, "rho outside (-1/(d-1), 1)"); break; }
        pot->pp.alpha = 1.0 / (1.0 - rho);
        pot->pp.beta = rho / ((1.0 - rho) * (1.0 - rho + dim * rho));
    } break;
    case PDMPFLUX_LOGREG: {
        if (!need(2)) { rc = fail(PDMPFLUX_ERR_ARGUMENT, "LOGREG needs n, sigma0, X[n*d], y[n]"); break; }
        const int64_t n = (int64_t)params[0];
        const double s0 = params[1];
        if (n <= 0 || !(s0 > 0.0) || !need(2 + n * dim + n)) { rc = fail(PDMPFLUX_ERR_ARGUMENT, "LOGREG: bad n / sigma0 / parameter length"); break; }
        if (dim > 128) { rc = fail(PDMPFLUX_ERR_UNSUPPORTED, "LOGREG supports dim <= 128 on the device path"); break; }
        const size_t yoff = ((size_t)n * dim + 1) & ~size_t(1);  // y starts 16-byte aligned (TMA bulk source)
        // two zeroed doubles of padding: the TMA tile copies round odd tails up to 16 bytes (logreg.cu: issue)
        if (pot->params.alloc(sizeof(double) * (yoff + n + 2)) != cudaSuccess ||
            cudaMemset(pot->params.p, 0, sizeof(double) * (yoff + n + 2)) != cudaSuccess ||
            cudaMemcpy(pot->params.p, params + 2, sizeof(double) * (size_t)n * dim, cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaMemcpy(pot->params.as<double>() + yoff, params + 2 + (size_t)n * dim, sizeof(double) * n, cudaMemcpyHostToDevice) != cudaSuccess) {
            rc = fail(PDMPFLUX_ERR_CUDA, "LOGREG design-matrix upload failed (is a CUDA device present?)");
            break;
        }
        pot->pp.vec = pot->params.as<double>();
        pot->pp.vec2 = pot->pp.vec + yoff;
        pot->pp.n = n;
        pot->pp.inv_s2 = 1.0 / (s0 * s0);
    } break;
    case PDMPFLUX_SOURCE:
        rc = fail(PDMPFLUX_ERR_ARGUMENT, "PDMPFLUX_SOURCE potentials carry CUDA source: create them with pdmpflux_potential_create_source");
        break;
    default: rc = fail(PDMPFLUX_ERR_ARGUMENT, "unknown potential kind " + std::to_string(kind));
    }
    if (rc != PDMPFLUX_OK) { delete pot; return rc; }
    *out = pot;
    return PDMPFLUX_OK;
}

int pdmpflux_potential_create_source(int dim, const char* source, const double* params, int64_t n_params,
                                     pdmpflux_potential_t* out) {
    if (!out) return fail(PDMPFLUX_ERR_ARGUMENT, "out is NULL");
    *out = nullptr;
    if (dim <= 0) return fail(PDMPFLUX_ERR_ARGUMENT, "dimension dim must be positive. Current value: " + std::to_string(dim));
    if (!source) return fail(PDMPFLUX_ERR_ARGUMENT, "source is NULL");
    if (n_params < 0 || (n_params > 0 && !params)) return fail(PDMPFLUX_ERR_ARGUMENT, "params must hold n_params >= 0 doubles");
    auto pot = std::make_unique<pdmpflux_potential_s>();
    pot->kind = PDMPFLUX_SOURCE; pot->dim = dim; pot->source = source;
    // the contract check runs before any CUDA call: bad source fails here, with or without a device
    const int rc = jit_check_source(pot->source, &pot->traits);
    if (rc != PDMPFLUX_OK) return rc;
    if (n_params > 0) {
        if (pot->params.alloc(sizeof(double) * (size_t)n_params) != cudaSuccess ||
            cudaMemcpy(pot->params.p, params, sizeof(double) * (size_t)n_params, cudaMemcpyHostToDevice) != cudaSuccess)
            return fail(PDMPFLUX_ERR_CUDA, "source potential parameter upload failed (is a CUDA device present?)");
        pot->pp.vec = pot->params.as<double>();
    }
    pot->pp.n = n_params;
    *out = pot.release();
    return PDMPFLUX_OK;
}
int pdmpflux_potential_destroy(pdmpflux_potential_t pot) { delete pot; return PDMPFLUX_OK; }

static int sampler_create_impl(int kind, int dim, pdmpflux_potential_t pot, const pdmpflux_config* cfg, const double* kappa,
                               pdmpflux_sampler_t* out);

int pdmpflux_sampler_create(int kind, int dim, pdmpflux_potential_t pot, const pdmpflux_config* cfg, pdmpflux_sampler_t* out) {
    if (kind == PDMPFLUX_STICKY_ZIGZAG)
        return fail(PDMPFLUX_ERR_ARGUMENT, "StickyZigZag needs the thawing rates kappa: use pdmpflux_sampler_create_sticky");
    return sampler_create_impl(kind, dim, pot, cfg, nullptr, out);
}

int pdmpflux_sampler_create_sticky(int dim, pdmpflux_potential_t pot, const pdmpflux_config* cfg, const double* kappa,
                                   pdmpflux_sampler_t* out) {
    if (!kappa) return fail(PDMPFLUX_ERR_ARGUMENT, "kappa is NULL");
    return sampler_create_impl(PDMPFLUX_STICKY_ZIGZAG, dim, pot, cfg, kappa, out);
}

static int sampler_create_impl(int kind, int dim, pdmpflux_potential_t pot, const pdmpflux_config* cfg, const double* kappa,
                               pdmpflux_sampler_t* out) {
    if (!out) return fail(PDMPFLUX_ERR_ARGUMENT, "out is NULL");
    *out = nullptr;
    if (!pot || !cfg) return fail(PDMPFLUX_ERR_ARGUMENT, "potential / config is NULL");
    if (kind < PDMPFLUX_ZIGZAG || kind > PDMPFLUX_SPEEDUP_ZIGZAG)
        return fail(PDMPFLUX_ERR_UNSUPPORTED, "sampler kind outside the device path (Sticky/SpeedUp/RHMC are not ported; no CPU fallback)");
    if (dim <= 0) return fail(PDMPFLUX_ERR_ARGUMENT, "dimension dim must be positive. Current value: " + std::to_string(dim));
    if (dim != pot->dim) return fail(PDMPFLUX_ERR_DIMENSION_MISMATCH, "potential dim " + std::to_string(pot->dim) + " != sampler dim " + std::to_string(dim));
    if (cfg->grid_size < 0) return fail(PDMPFLUX_ERR_ARGUMENT, "grid_size must be non-negative. Current value: " + std::to_string(cfg->grid_size));
    if (cfg->grid_size == 1) return fail(PDMPFLUX_ERR_ARGUMENT, "grid_size == 1 is invalid upstream (t[2] out of bounds, UpperBound.jl:95,205); use 0 or >= 2");
    if (cfg->grid_size > kMaxGrid) return fail(PDMPFLUX_ERR_UNSUPPORTED, "grid_size > " + std::to_string(kMaxGrid) + " not supported on the device path");
    if (kind == PDMPFLUX_FECMC && dim < 2)
        return fail(PDMPFLUX_ERR_ARGUMENT, "The dimension must be at least 2 to use the ForwardEventChain. Got dimension " + std::to_string(dim));
    if (!(cfg->tmax >= 0.0) || !std::isfinite(cfg->tmax)) return fail(PDMPFLUX_ERR_ARGUMENT, "tmax must be finite and >= 0");
    pdmpflux_config ncfg = *cfg;
    normalise_config(kind, dim, ncfg);
    if (pot->kind == PDMPFLUX_SOURCE) {
        // compile every kernel variant the default policy can pick for this sampler (the team widths chosen at one
        // chain and at any number of chains) before any CUDA call, so that source errors surface here even without a
        // device
        for (int64_t n_chains : {int64_t(1), INT64_MAX}) {
            const Variant v = chain_variant(kind, dim, ncfg, pot, n_chains, false);
            const int rc = jit_prepare(pot->source, kind, v.team, v.path, v.nw);
            if (rc != PDMPFLUX_OK) return rc;
        }
    }
    auto s = new pdmpflux_sampler_s();
    s->kind = kind; s->dim = dim; s->cfg = ncfg; s->pot = pot;
    if (kind == PDMPFLUX_STICKY_ZIGZAG) {
        for (int i = 0; i < dim; ++i)
            if (!(kappa[i] >= 0.0) || !std::isfinite(kappa[i])) { delete s; return fail(PDMPFLUX_ERR_ARGUMENT, "kappa must be finite and non-negative"); }
        if (s->kappa.alloc(sizeof(double) * dim) != cudaSuccess ||
            cudaMemcpy(s->kappa.p, kappa, sizeof(double) * dim, cudaMemcpyHostToDevice) != cudaSuccess) {
            delete s;
            return fail(PDMPFLUX_ERR_CUDA, "kappa upload failed (is a CUDA device present?)");
        }
    }
    if (pot->kind == PDMPFLUX_LOGREG) {
        const pdmpflux_config& c = s->cfg;
        if (kind != PDMPFLUX_ZIGZAG || !c.vectorized_bound || c.grid_size < 2 || c.grid_size > 12 ||
            c.deriv_mode != PDMPFLUX_DERIV_JVP) {
            delete s;
            return fail(PDMPFLUX_ERR_UNSUPPORTED, "LOGREG runs on the device with ZigZag, vectorized_bound=true, 2 <= grid_size <= 12 "
                                                  "and an exact AD_backend (no CPU fallback)");
        }
    }
    *out = s;
    return PDMPFLUX_OK;
}
int pdmpflux_sampler_destroy(pdmpflux_sampler_t s) { delete s; return PDMPFLUX_OK; }
int pdmpflux_sampler_release_workspace(pdmpflux_sampler_t s) {
    if (!s) return fail(PDMPFLUX_ERR_ARGUMENT, "sampler is NULL");
    CUDA_TRY(cudaDeviceSynchronize());
    s->ws.~Workspace();
    new (&s->ws) Workspace();
    return PDMPFLUX_OK;
}
int pdmpflux_sampler_get_config(pdmpflux_sampler_t s, pdmpflux_config* out) {
    if (!s || !out) return fail(PDMPFLUX_ERR_ARGUMENT, "NULL argument");
    *out = s->cfg;
    return PDMPFLUX_OK;
}

int pdmpflux_chains_create(pdmpflux_sampler_t s, int64_t n_chains, const double* xinit, const double* vinit,
                           int32_t init_on_device, uint64_t seed, int64_t chain_offset,
                           const pdmpflux_tape* tape, pdmpflux_chains_t* out) {
    if (!out) return fail(PDMPFLUX_ERR_ARGUMENT, "out is NULL");
    *out = nullptr;
    if (!s || !xinit || !vinit) return fail(PDMPFLUX_ERR_ARGUMENT, "NULL argument");
    if (n_chains <= 0) return fail(PDMPFLUX_ERR_ARGUMENT, "n_chains must be positive");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(PDMPFLUX_ERR_CUDA, "no CUDA device: libpdmpflux_cuda has no CPU fallback");
    auto ch = new pdmpflux_chains_s();
    struct Guard { pdmpflux_chains_s* c; ~Guard() { delete c; } } guard{ch};
    ch->s = s; ch->n_chains = n_chains; ch->chain_offset = chain_offset; ch->seed = seed;
    const int d = s->dim;
    const bool logreg = s->pot->kind == PDMPFLUX_LOGREG;
    const Variant var = chain_variant(s->kind, d, s->cfg, s->pot, n_chains, true);
    ch->path = var.path; ch->team = var.team; ch->n_own = var.n_own; ch->brent_nw = var.nw;
    if (s->pot->kind == PDMPFLUX_SOURCE) {  // a variant sampler_create did not compile (PDMPFLUX_TEAM / _FORCE_GENERIC)
        const int rc = jit_prepare(s->pot->source, s->kind, ch->team, ch->path, ch->brent_nw);
        if (rc != PDMPFLUX_OK) return rc;
    }
    const int bt = block_threads_rt(ch->team, s->kind, ch->path);   // threads per block of the kernel that will run
    const int cpb = bt / ch->team;
    ch->grid = (unsigned)((n_chains + cpb - 1) / cpb);
    ch->n_groups = ch->grid;
    if (ch->team == 1) { ch->dpad = 0; ch->vec_elems = ch->n_own * bt; }
    else {
        ch->dpad = (ch->n_own * ch->team + 7) / 8 * 8;                  // 64-byte aligned chain slots (TMA source)
        if (ch->team < 32 && ch->dpad % 16 != 8) ch->dpad += 8;         // chains of a warp land on distinct bank halves
        ch->vec_elems = cpb * ch->dpad;
    }
    const size_t vec_bytes = (size_t)ch->vec_elems * sizeof(double);
    const size_t nvec = state_vectors(s->kind, ch->path, ch->team, ch->brent_nw);
    ch->smem = (nvec + (s->kind == PDMPFLUX_STICKY_ZIGZAG ? 1 : 0)) * vec_bytes;
    const size_t list_slack = ch->brent_nw == kLineTransposed ? 16 * sizeof(double) : 0;   // transposed Brent: unconditional reads of the 12-slot list
    if (s->kind == PDMPFLUX_FECMC) {
        if ((nvec + 3) * vec_bytes <= 64 * 1024) { ch->scratch_in_smem = 1; ch->smem = (nvec + 3) * vec_bytes; }
        else {
            // Scratch vectors in global memory: run a persistent grid (one block per resident slot: the kernel is built
            // for 3 blocks of a warp-per-chain team per SM) so that the scratch is indexed by the resident block, fits
            // the L2 (a few tens of MB) and is rewritten in place.
            ch->scratch_in_smem = 0;
            int dev = 0, n_sm = 148;
            cudaGetDevice(&dev);
            if (cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n_sm <= 0) n_sm = 148;
            ch->grid = (unsigned)std::min<int64_t>(ch->n_groups, (int64_t)(ch->team == 32 ? 3 : 4) * n_sm);
            CUDA_TRY(ch->scratch.alloc((size_t)ch->grid * 3 * vec_bytes));
        }
    }
    if (ch->team == 1) ch->smem += 6 * (size_t)bt * sizeof(double);  // row carry slots (record())
    {
        const size_t gb = s->cfg.grid_size > 2 ? s->cfg.grid_size : 2;      // box_max / cum_sum, one copy per chain
        ch->smem += (ch->team == 1 ? (size_t)bt : (size_t)cpb) * 2 * gb * sizeof(double);
    }
    ch->smem += list_slack;
    if (logreg) {  // logreg_chains_per_block() chains per CTA, one warp each
        const int lcpb = logreg_chains_per_block();
        ch->grid = (unsigned)((n_chains + lcpb - 1) / lcpb);
        ch->smem = logreg_smem_bytes(d, s->cfg.grid_size);
        // (z, w) = (X x, X v) cache, [chain][32-row tile][row][2] (logreg.cu: lr_produce).  Optional: when it does not
        // fit (or PDMPFLUX_LOGREG_NO_ZW_CACHE=1) the kernel recomputes z, w in every pass.
        const int64_t ntiles = (s->pot->pp.n + 31) / 32;
        const size_t zw_bytes = (size_t)n_chains * (size_t)ntiles * 64 * sizeof(double);
        const char* off = getenv("PDMPFLUX_LOGREG_NO_ZW_CACHE");
        if (!(off && off[0] == '1') && zw_bytes <= ((size_t)32 << 30) && ch->scratch.alloc(zw_bytes) != cudaSuccess)
            (void)cudaGetLastError();  // out of memory: run without the cache
        CUDA_TRY(ch->wq.alloc(sizeof(int64_t)));  // work-queue counter of the persistent launch
    }
    if (ch->smem > 227 * 1024) return fail(PDMPFLUX_ERR_UNSUPPORTED, "dimension too large for the shared-memory state layout");
    CUDA_TRY(ch->x.alloc(sizeof(double) * d * n_chains));
    CUDA_TRY(ch->v.alloc(sizeof(double) * d * n_chains));
    CUDA_TRY(ch->t.alloc(sizeof(double) * n_chains));
    CUDA_TRY(ch->horizon.alloc(sizeof(double) * n_chains));
    CUDA_TRY(ch->ar.alloc(sizeof(double) * n_chains));
    CUDA_TRY(ch->tape_pos.alloc(sizeof(int64_t) * 3 * n_chains));
    CUDA_TRY(ch->status.alloc(sizeof(int32_t) * n_chains));
    CUDA_TRY(ch->counters.alloc(sizeof(int64_t) * 2 * n_chains));
    CUDA_TRY(ch->ncols.alloc(sizeof(int64_t) * n_chains));
    // Stream ordering: the set-up below runs on the legacy default stream, the kernels later run on the caller's stream
    // (possibly cudaStreamNonBlocking).  Device inputs may still be in flight on the caller's stream, so wait for the
    // device first; the stream is drained again before returning, so every later launch sees initialised state.
    if (init_on_device || (tape && tape->on_device)) CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemset(ch->ncols.p, 0, sizeof(int64_t) * n_chains));
    if (s->kind == PDMPFLUX_STICKY_ZIGZAG) {  // PDMPState ctor: is_active = trues(d) (Composites.jl:95-99)
        CUDA_TRY(ch->act.alloc((size_t)d * n_chains));
        CUDA_TRY(cudaMemset(ch->act.p, 1, (size_t)d * n_chains));
    }
    const cudaMemcpyKind k = init_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    CUDA_TRY(cudaMemcpy(ch->x.p, xinit, sizeof(double) * d * n_chains, k));
    CUDA_TRY(cudaMemcpy(ch->v.p, vinit, sizeof(double) * d * n_chains, k));
    CUDA_TRY(cudaMemset(ch->t.p, 0, sizeof(double) * n_chains));
    CUDA_TRY(cudaMemset(ch->ar.p, 0, sizeof(double) * n_chains));
    CUDA_TRY(cudaMemset(ch->tape_pos.p, 0, sizeof(int64_t) * 3 * n_chains));
    CUDA_TRY(cudaMemset(ch->status.p, 0, sizeof(int32_t) * n_chains));
    CUDA_TRY(cudaMemset(ch->counters.p, 0, sizeof(int64_t) * 2 * n_chains));
    {
        std::vector<double> h0((size_t)n_chains, s->cfg.tmax);  // init_state: horizon = tmax (AbstractPDMP.jl:141-149)
        CUDA_TRY(cudaMemcpy(ch->horizon.p, h0.data(), sizeof(double) * n_chains, cudaMemcpyHostToDevice));
    }
    if (tape) {
        if (!tape->E || !tape->U || !tape->N || tape->nE <= 0 || tape->nU <= 0 || tape->nN <= 0)
            return fail(PDMPFLUX_ERR_ARGUMENT, "tape streams must be non-empty");
        ch->draw_mode = 0; ch->nE = tape->nE; ch->nU = tape->nU; ch->nN = tape->nN;
        if (tape->on_device) { ch->dE = tape->E; ch->dU = tape->U; ch->dN = tape->N; }
        else {
            CUDA_TRY(ch->tE.alloc(sizeof(double) * tape->nE * n_chains));
            CUDA_TRY(ch->tU.alloc(sizeof(double) * tape->nU * n_chains));
            CUDA_TRY(ch->tN.alloc(sizeof(double) * tape->nN * n_chains));
            CUDA_TRY(cudaMemcpy(ch->tE.p, tape->E, ch->tE.bytes, cudaMemcpyHostToDevice));
            CUDA_TRY(cudaMemcpy(ch->tU.p, tape->U, ch->tU.bytes, cudaMemcpyHostToDevice));
            CUDA_TRY(cudaMemcpy(ch->tN.p, tape->N, ch->tN.bytes, cudaMemcpyHostToDevice));
            ch->dE = ch->tE.as<double>(); ch->dU = ch->tU.as<double>(); ch->dN = ch->tN.as<double>();
        }
    }
    CUDA_TRY(cudaStreamSynchronize(cudaStreamLegacy));  // set-up complete before any launch on any stream
    guard.c = nullptr;
    *out = ch;
    return PDMPFLUX_OK;
}

int pdmpflux_chains_set_state(pdmpflux_chains_t ch, const double* t, const double* horizon, int64_t event0,
                              int32_t on_device) {
    if (!ch) return fail(PDMPFLUX_ERR_ARGUMENT, "chains is NULL");
    if (event0 < 0) return fail(PDMPFLUX_ERR_ARGUMENT, "event0 must be >= 0");
    const cudaMemcpyKind k = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    // earlier launches of these chains (any stream) and the producer of device inputs must be done; see chains_create
    if (t || horizon) CUDA_TRY(cudaDeviceSynchronize());
    if (t) CUDA_TRY(cudaMemcpy(ch->t.p, t, sizeof(double) * ch->n_chains, k));
    if (horizon) CUDA_TRY(cudaMemcpy(ch->horizon.p, horizon, sizeof(double) * ch->n_chains, k));
    if (t || horizon) CUDA_TRY(cudaStreamSynchronize(cudaStreamLegacy));
    ch->event0 = event0;
    return PDMPFLUX_OK;
}

int pdmpflux_chains_get_state(pdmpflux_chains_t ch, double* x, double* v, double* t, double* horizon, int32_t on_device) {
    if (!ch) return fail(PDMPFLUX_ERR_ARGUMENT, "chains is NULL");
    const cudaMemcpyKind k = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    const size_t nd = sizeof(double) * ch->s->dim * ch->n_chains;
    CUDA_TRY(cudaDeviceSynchronize());  // launches on a non-blocking stream are not ordered before legacy-stream copies
    if (x) CUDA_TRY(cudaMemcpy(x, ch->x.p, nd, k));
    if (v) CUDA_TRY(cudaMemcpy(v, ch->v.p, nd, k));
    if (t) CUDA_TRY(cudaMemcpy(t, ch->t.p, sizeof(double) * ch->n_chains, k));
    if (horizon) CUDA_TRY(cudaMemcpy(horizon, ch->horizon.p, sizeof(double) * ch->n_chains, k));
    return PDMPFLUX_OK;
}

int pdmpflux_chains_enable_moments(pdmpflux_chains_t ch) {
    if (!ch) return fail(PDMPFLUX_ERR_ARGUMENT, "chains is NULL");
    if (ch->s->pot->kind == PDMPFLUX_LOGREG) return fail(PDMPFLUX_ERR_UNSUPPORTED, "fused moments are not available for the logistic-regression kernel");
    if (ch->s->kind == PDMPFLUX_SPEEDUP_ZIGZAG) return fail(PDMPFLUX_ERR_UNSUPPORTED, "fused moments need closed-form segment integrals: not available for the Speed-Up Zig-Zag flow");
    if (ch->moments) return PDMPFLUX_OK;
    const size_t nd = sizeof(double) * ch->s->dim * ch->n_chains;
    CUDA_TRY(ch->m1.alloc(nd)); CUDA_TRY(ch->m2.alloc(nd));
    CUDA_TRY(cudaMemset(ch->m1.p, 0, nd)); CUDA_TRY(cudaMemset(ch->m2.p, 0, nd));
    CUDA_TRY(cudaStreamSynchronize(cudaStreamLegacy));  // zeroed before the next launch on the caller's stream
    ch->moments = 1;
    return PDMPFLUX_OK;
}

int pdmpflux_chains_get_moments(pdmpflux_chains_t ch, double* m1, double* m2, int32_t on_device) {
    if (!ch || !ch->moments) return fail(PDMPFLUX_ERR_ARGUMENT, "moments are not enabled on these chains");
    const cudaMemcpyKind k = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    const size_t nd = sizeof(double) * ch->s->dim * ch->n_chains;
    CUDA_TRY(cudaDeviceSynchronize());
    if (m1) CUDA_TRY(cudaMemcpy(m1, ch->m1.p, nd, k));
    if (m2) CUDA_TRY(cudaMemcpy(m2, ch->m2.p, nd, k));
    return PDMPFLUX_OK;
}

int pdmpflux_chains_set_stop_time(pdmpflux_chains_t ch, double T) {
    if (!ch) return fail(PDMPFLUX_ERR_ARGUMENT, "chains is NULL");
    if (T != T) { ch->use_t_stop = 0; return PDMPFLUX_OK; }
    if (!std::isfinite(T) || T < 0) return fail(PDMPFLUX_ERR_ARGUMENT, "T must be finite and non-negative. Current value: " + std::to_string(T));
    ch->use_t_stop = 1; ch->t_stop = T;
    return PDMPFLUX_OK;
}

int pdmpflux_chains_get_ncols(pdmpflux_chains_t ch, int64_t* ncols) {
    if (!ch || !ncols) return fail(PDMPFLUX_ERR_ARGUMENT, "NULL argument");
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(ncols, ch->ncols.p, sizeof(int64_t) * ch->n_chains, cudaMemcpyDeviceToHost));
    return PDMPFLUX_OK;
}

int pdmpflux_chains_advance(pdmpflux_chains_t ch, int64_t n_events, const pdmpflux_history* h, int64_t col0, void* stream) {
    if (!ch) return fail(PDMPFLUX_ERR_ARGUMENT, "chains is NULL");
    if (n_events <= 0) return fail(PDMPFLUX_ERR_ARGUMENT, "n_events must be positive");
    if (h && (!h->on_device || col0 < 0 || col0 + n_events > h->n_cols))
        return fail(PDMPFLUX_ERR_ARGUMENT, "chains_advance needs a device history view with col0 + n_events <= n_cols");
    const int rc = launch(ch, n_events, h, col0, static_cast<cudaStream_t>(stream));
    if (rc == PDMPFLUX_OK) ch->event0 += n_events;
    return rc;
}

int pdmpflux_chains_record(pdmpflux_chains_t ch, const pdmpflux_history* h, int64_t col, void* stream) {
    if (!ch || !h) return fail(PDMPFLUX_ERR_ARGUMENT, "NULL argument");
    if (!h->on_device || col < 0 || col >= h->n_cols) return fail(PDMPFLUX_ERR_ARGUMENT, "chains_record needs a device view and a valid column");
    return launch(ch, 0, h, col, static_cast<cudaStream_t>(stream));
}

int pdmpflux_chains_status(pdmpflux_chains_t ch, int32_t* status, int64_t* tape_pos, int64_t* counters) {
    if (!ch) return fail(PDMPFLUX_ERR_ARGUMENT, "chains is NULL");
    std::vector<int32_t> st((size_t)ch->n_chains);
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(st.data(), ch->status.p, sizeof(int32_t) * ch->n_chains, cudaMemcpyDeviceToHost));
    if (status) std::memcpy(status, st.data(), sizeof(int32_t) * ch->n_chains);
    if (tape_pos) CUDA_TRY(cudaMemcpy(tape_pos, ch->tape_pos.p, sizeof(int64_t) * 3 * ch->n_chains, cudaMemcpyDeviceToHost));
    if (counters) CUDA_TRY(cudaMemcpy(counters, ch->counters.p, sizeof(int64_t) * 2 * ch->n_chains, cudaMemcpyDeviceToHost));
    int64_t bad = 0, first = -1;
    for (int64_t c = 0; c < ch->n_chains; ++c)
        if (st[c] != 0 && st[c] != PDMPFLUX_CHAIN_DONE) { if (first < 0) first = c; ++bad; }
    if (bad) return fail(PDMPFLUX_ERR_CHAIN, std::to_string(bad) + " chain(s) stopped; first: chain " + std::to_string(first) + " status " + std::to_string(st[first]));
    return PDMPFLUX_OK;
}

int pdmpflux_chains_destroy(pdmpflux_chains_t ch) { delete ch; return PDMPFLUX_OK; }

int pdmpflux_sample_skeleton(pdmpflux_sampler_t s, int64_t n_chains, int64_t n_sk, const double* xinit,
                             const double* vinit, uint64_t seed, int64_t chain_offset, const pdmpflux_tape* tape,
                             const pdmpflux_history* hist, void* stream_) {
    return pdmpflux_sample_skeleton_resume(s, n_chains, n_sk, xinit, vinit, nullptr, nullptr, 0, seed, chain_offset,
                                           tape, hist, stream_);
}

static int run_skeleton(pdmpflux_sampler_t s, int64_t n_chains, int64_t n_sk, const double* xinit, const double* vinit,
                        const double* t0, const double* horizon0, int64_t event0, uint64_t seed, int64_t chain_offset,
                        const pdmpflux_tape* tape, const pdmpflux_history* hist, void* stream_, const double* t_stop,
                        int64_t* n_cols_out);

int pdmpflux_sample_skeleton_resume(pdmpflux_sampler_t s, int64_t n_chains, int64_t n_sk, const double* xinit,
                                    const double* vinit, const double* t0, const double* horizon0, int64_t event0,
                                    uint64_t seed, int64_t chain_offset, const pdmpflux_tape* tape,
                                    const pdmpflux_history* hist, void* stream_) {
    return run_skeleton(s, n_chains, n_sk, xinit, vinit, t0, horizon0, event0, seed, chain_offset, tape, hist, stream_,
                        nullptr, nullptr);
}

int pdmpflux_sample_skeleton_until(pdmpflux_sampler_t s, int64_t n_chains, double T, int64_t capacity,
                                   const double* xinit, const double* vinit, uint64_t seed, int64_t chain_offset,
                                   const pdmpflux_tape* tape, const pdmpflux_history* hist, int64_t* n_cols_out,
                                   void* stream_) {
    if (!std::isfinite(T) || T < 0) return fail(PDMPFLUX_ERR_ARGUMENT, "T must be finite and non-negative. Current value: " + std::to_string(T));
    if (capacity <= 0 || !n_cols_out) return fail(PDMPFLUX_ERR_ARGUMENT, "capacity must be positive and n_cols_out non-NULL");
    return run_skeleton(s, n_chains, capacity, xinit, vinit, nullptr, nullptr, 0, seed, chain_offset, tape, hist, stream_,
                        &T, n_cols_out);
}

static int run_skeleton(pdmpflux_sampler_t s, int64_t n_chains, int64_t n_sk, const double* xinit, const double* vinit,
                        const double* t0, const double* horizon0, int64_t event0, uint64_t seed, int64_t chain_offset,
                        const pdmpflux_tape* tape, const pdmpflux_history* hist, void* stream_, const double* t_stop,
                        int64_t* n_cols_out) {
    if (!s || !hist) return fail(PDMPFLUX_ERR_ARGUMENT, "NULL argument");
    if (n_sk <= 0) return fail(PDMPFLUX_ERR_ARGUMENT, "n_sk must be positive. Current value: " + std::to_string(n_sk));
    if (hist->n_cols < n_sk) return fail(PDMPFLUX_ERR_ARGUMENT, "history n_cols < n_sk");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    pdmpflux_chains_t ch = nullptr;
    int rc = pdmpflux_chains_create(s, n_chains, xinit, vinit, hist->on_device, seed, chain_offset, tape, &ch);
    if (rc != PDMPFLUX_OK) return rc;
    struct Guard { pdmpflux_chains_t c; ~Guard() { pdmpflux_chains_destroy(c); } } guard{ch};
    const int d = s->dim;
    if (t0 || horizon0 || event0) {
        rc = pdmpflux_chains_set_state(ch, t0, horizon0, event0, hist->on_device);
        if (rc != PDMPFLUX_OK) return rc;
    }
    if (t_stop) {
        if (s->kind == PDMPFLUX_STICKY_ZIGZAG)
            return fail(PDMPFLUX_ERR_UNSUPPORTED, "the time-horizon sample_skeleton is not available for StickyZigZag on the device path (no CPU fallback)");
        rc = pdmpflux_chains_set_stop_time(ch, *t_stop);
        if (rc != PDMPFLUX_OK) return rc;
    }
    // time-horizon variant: report ragged column counts; a chain that used the whole capacity without reaching T
    // makes the call return PDMPFLUX_ERR_CAPACITY (after the outputs have been delivered)
    auto finish = [&](int rc_status) -> int {
        if (!t_stop || (rc_status != PDMPFLUX_OK)) return rc_status;
        std::vector<int64_t> nc((size_t)n_chains);
        std::vector<int32_t> st((size_t)n_chains);
        if (cudaMemcpy(nc.data(), ch->ncols.p, sizeof(int64_t) * n_chains, cudaMemcpyDeviceToHost) != cudaSuccess ||
            cudaMemcpy(st.data(), ch->status.p, sizeof(int32_t) * n_chains, cudaMemcpyDeviceToHost) != cudaSuccess)
            return fail(PDMPFLUX_ERR_CUDA, "reading back column counts failed");
        int64_t unfinished = 0;
        for (int64_t c = 0; c < n_chains; ++c) {
            if (hist->on_device) { /* counts are always returned on the host */ }
            n_cols_out[c] = nc[c];
            if (st[c] != PDMPFLUX_CHAIN_DONE) ++unfinished;
        }
        if (unfinished) return fail(PDMPFLUX_ERR_CAPACITY, std::to_string(unfinished) + " chain(s) need more than " + std::to_string(n_sk) + " columns to reach T");
        return PDMPFLUX_OK;
    };

    if (hist->on_device) {
        pdmpflux_history h = *hist;
        rc = pdmpflux_chains_record(ch, &h, 0, stream);
        if (rc == PDMPFLUX_OK && n_sk > 1) rc = pdmpflux_chains_advance(ch, n_sk - 1, &h, 1, stream);
        if (rc != PDMPFLUX_OK) return rc;
        CUDA_TRY(cudaStreamSynchronize(stream));
        if (hist->status) CUDA_TRY(cudaMemcpy(hist->status, ch->status.p, sizeof(int32_t) * n_chains, cudaMemcpyDeviceToDevice));
        if (hist->tape_pos) CUDA_TRY(cudaMemcpy(hist->tape_pos, ch->tape_pos.p, sizeof(int64_t) * 3 * n_chains, cudaMemcpyDeviceToDevice));
        if (hist->counters) CUDA_TRY(cudaMemcpy(hist->counters, ch->counters.p, sizeof(int64_t) * 2 * n_chains, cudaMemcpyDeviceToDevice));
        return finish(pdmpflux_chains_status(ch, nullptr, nullptr, nullptr));
    }

    if (s->kind == PDMPFLUX_STICKY_ZIGZAG) {
        // Sticky Zig-Zag with host buffers: the whole history is produced in device memory and copied once (this is the
        // row after the hot path; the sliced, overlapped pipeline below serves the four samplers of the hot path).
        const size_t nc = (size_t)n_chains * n_sk;
        DevBuf dX, dV, dt, dh, da, de, deb, drj, dhh, dact;
        pdmpflux_history hv{};
        hv.n_cols = n_sk; hv.on_device = 1;
        auto want = [&](DevBuf& b, const void* host, size_t bytes) -> void* {
            if (!host) return nullptr;
            return b.alloc(bytes) == cudaSuccess ? b.p : nullptr;
        };
        hv.X = (double*)want(dX, hist->X, nc * d * 8); hv.V = (double*)want(dV, hist->V, nc * d * 8);
        hv.t = (double*)want(dt, hist->t, nc * 8); hv.horizon = (double*)want(dh, hist->horizon, nc * 8);
        hv.ar = (double*)want(da, hist->ar, nc * 8); hv.error_value_ar = (double*)want(de, hist->error_value_ar, nc * 40);
        hv.errored_bound = (int32_t*)want(deb, hist->errored_bound, nc * 4); hv.rejected = (int32_t*)want(drj, hist->rejected, nc * 4);
        hv.hitting_horizon = (int32_t*)want(dhh, hist->hitting_horizon, nc * 4);
        hv.is_active = (uint8_t*)want(dact, hist->is_active, nc * d);
        if ((hist->X && !hv.X) || (hist->V && !hv.V) || (hist->t && !hv.t) || (hist->is_active && !hv.is_active))
            return fail(PDMPFLUX_ERR_CUDA, "device allocation for the sticky history failed");
        rc = pdmpflux_chains_record(ch, &hv, 0, stream);
        if (rc == PDMPFLUX_OK && n_sk > 1) rc = pdmpflux_chains_advance(ch, n_sk - 1, &hv, 1, stream);
        if (rc != PDMPFLUX_OK) return rc;
        CUDA_TRY(cudaStreamSynchronize(stream));
        auto back = [&](void* host, const void* dev, size_t elem) -> cudaError_t {
            if (!host) return cudaSuccess;
            return cudaMemcpy2D(host, (size_t)hist->n_cols * elem, dev, (size_t)n_sk * elem, (size_t)n_sk * elem, (size_t)n_chains,
                                cudaMemcpyDeviceToHost);
        };
        CUDA_TRY(back(hist->X, hv.X, 8 * (size_t)d)); CUDA_TRY(back(hist->V, hv.V, 8 * (size_t)d));
        CUDA_TRY(back(hist->t, hv.t, 8)); CUDA_TRY(back(hist->horizon, hv.horizon, 8)); CUDA_TRY(back(hist->ar, hv.ar, 8));
        CUDA_TRY(back(hist->error_value_ar, hv.error_value_ar, 40)); CUDA_TRY(back(hist->errored_bound, hv.errored_bound, 4));
        CUDA_TRY(back(hist->rejected, hv.rejected, 4)); CUDA_TRY(back(hist->hitting_horizon, hv.hitting_horizon, 4));
        CUDA_TRY(back(hist->is_active, hv.is_active, (size_t)d));
        return pdmpflux_chains_status(ch, hist->status, hist->tape_pos, hist->counters);
    }

    // ---- host-buffer path: slices of columns, two device slabs, D2H of slice i overlaps the kernel of slice i+1
    const size_t per_col = (size_t)n_chains * ((hist->X ? 8 * d : 0) + (hist->V ? 8 * d : 0) + (hist->t ? 8 : 0) +
                                               (hist->horizon ? 8 : 0) + (hist->ar ? 8 : 0) + (hist->error_value_ar ? 40 : 0) +
                                               (hist->errored_bound ? 4 : 0) + (hist->rejected ? 4 : 0) + (hist->hitting_horizon ? 4 : 0));
    size_t budget = 1ull << 30;  // bytes per device slab
    if (const char* e = std::getenv("PDMPFLUX_SLAB_BYTES")) budget = std::max<size_t>(1 << 16, std::strtoull(e, nullptr, 10));
    int64_t slice = per_col ? (int64_t)std::max<size_t>(1, budget / per_col) : n_sk;
    slice = std::min<int64_t>(slice, n_sk);
    // enough slices for the copies to overlap the kernels, but slices long enough to amortise launches
    int64_t want_slices = 16;
    if (const char* e = std::getenv("PDMPFLUX_SLICES")) want_slices = std::max<int64_t>(1, std::atoll(e));
    if (n_sk >= 64) slice = std::min<int64_t>(slice, std::max<int64_t>(16, (n_sk + want_slices - 1) / want_slices));
    slice = std::max<int64_t>(slice, 1);
    slice = (slice + 3) & ~int64_t(3);  // keeps every slab column 32-byte aligned for the 256-bit store path

    Workspace& ws = s->ws;
    Slab* slab = ws.slab;
    if (!ws.copy_stream) CUDA_TRY(cudaStreamCreateWithFlags(&ws.copy_stream, cudaStreamNonBlocking));
    cudaStream_t copy_stream = ws.copy_stream;
    const int n_slabs = slice < n_sk ? 2 : 1;
    auto ensure = [](DevBuf& b, bool want, size_t bytes) -> cudaError_t {
        if (!want) return cudaSuccess;
        if (b.bytes >= bytes && b.p) return cudaSuccess;
        return b.alloc(bytes);
    };
    // Scalar columns (76 of the 16d+76 bytes per event) accumulate in full-length device buffers and go to the host
    // in a few wide chunks; only the X / V rows are double-buffered through the narrow slabs.  (Slicing the scalar
    // columns like the rows would mean n_chains x n_slices x 7 strided host rows of a few hundred bytes each.)
    const int64_t ldS = (n_sk + 3) & ~int64_t(3);
    const bool full_scalars = (size_t)n_chains * ldS * 76 <= (8ull << 30);
    Slab& sc = ws.scal;
    if (full_scalars) {
        CUDA_TRY(ensure(sc.t, hist->t, sizeof(double) * n_chains * ldS));
        CUDA_TRY(ensure(sc.horizon, hist->horizon, sizeof(double) * n_chains * ldS));
        CUDA_TRY(ensure(sc.ar, hist->ar, sizeof(double) * n_chains * ldS));
        CUDA_TRY(ensure(sc.eva, hist->error_value_ar, sizeof(double) * 5 * n_chains * ldS));
        CUDA_TRY(ensure(sc.eb, hist->errored_bound, sizeof(int32_t) * n_chains * ldS));
        CUDA_TRY(ensure(sc.rej, hist->rejected, sizeof(int32_t) * n_chains * ldS));
        CUDA_TRY(ensure(sc.hh, hist->hitting_horizon, sizeof(int32_t) * n_chains * ldS));
        sc.view = pdmpflux_history{};
        sc.view.t = hist->t ? sc.t.as<double>() : nullptr; sc.view.horizon = hist->horizon ? sc.horizon.as<double>() : nullptr;
        sc.view.ar = hist->ar ? sc.ar.as<double>() : nullptr;
        sc.view.error_value_ar = hist->error_value_ar ? sc.eva.as<double>() : nullptr;
        sc.view.errored_bound = hist->errored_bound ? sc.eb.as<int32_t>() : nullptr;
        sc.view.rejected = hist->rejected ? sc.rej.as<int32_t>() : nullptr;
        sc.view.hitting_horizon = hist->hitting_horizon ? sc.hh.as<int32_t>() : nullptr;
        sc.view.n_cols = ldS; sc.view.on_device = 1;
    }
    // Zig-Zag: V rows travel as sign bits (pack_signs_kernel) and are rebuilt on the host by worker threads while the
    // later slices still run; everything else (and PDMPFLUX_NO_VBITS=1) copies the V rows as they are.
    // Rebuilding 8 d bytes per event on the host only pays when enough CPUs are free for it (measured: 16 threads beat
    // the plain copy by 1.2-1.3x on a PCIe Gen5 host, 8 threads lose), so it needs >= 12 usable CPUs unless
    // PDMPFLUX_VBITS=1 forces it; PDMPFLUX_NO_VBITS=1 (or PDMPFLUX_VBITS=0) turns it off.
    unsigned avail_cpus = std::max<unsigned>(1, std::thread::hardware_concurrency());
#if defined(__linux__)
    {
        cpu_set_t set;
        if (sched_getaffinity(0, sizeof(set), &set) == 0) avail_cpus = std::max(1, CPU_COUNT(&set));
    }
#endif
    const char* no_vbits = std::getenv("PDMPFLUX_NO_VBITS");
    const char* force_vbits = std::getenv("PDMPFLUX_VBITS");
    bool vbits = hist->V && s->kind == PDMPFLUX_ZIGZAG && avail_cpus >= 12;
    if (force_vbits) vbits = hist->V && s->kind == PDMPFLUX_ZIGZAG && force_vbits[0] == '1';
    if (no_vbits && no_vbits[0] == '1') vbits = false;
    const int vwords = (d + 31) / 32;
    const int64_t n_slices = (n_sk + slice - 1) / slice;
    const size_t vstride = (size_t)n_chains * slice * vwords;  // words per slice
    std::vector<double> absv;
    int n_threads = 1;
    if (vbits) {
        absv.resize((size_t)n_chains * d);
        for (size_t e = 0; e < absv.size(); ++e) absv[e] = std::fabs(vinit[e]);
        n_threads = (int)std::min<unsigned>(16, avail_cpus);
        if (const char* e = std::getenv("PDMPFLUX_HOST_THREADS")) n_threads = std::max(1, std::atoi(e));
        n_threads = (int)std::min<int64_t>(n_threads, n_chains);
        const size_t vb = sizeof(uint32_t) * vstride * (size_t)n_slices;
        CUDA_TRY(ensure(ws.vbits, true, vb));
        if (ws.vbits_host_bytes < vb) {
            if (ws.vbits_host) { cudaFreeHost(ws.vbits_host); ws.vbits_host = nullptr; ws.vbits_host_bytes = 0; }
            CUDA_TRY(cudaHostAlloc(reinterpret_cast<void**>(&ws.vbits_host), vb, cudaHostAllocDefault));
            ws.vbits_host_bytes = vb;
        }
        while ((int64_t)ws.slice_copied.size() < n_slices) {
            cudaEvent_t e;
            CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            ws.slice_copied.push_back(e);
        }
    }
    // all-zero slices of errored_bound / error_value_ar stay on the device (flag_nonzero_kernel); the workers zero-fill
    const bool zskip = vbits && full_scalars && hist->errored_bound && hist->error_value_ar;
    if (zskip) {
        CUDA_TRY(ensure(ws.zflags, true, sizeof(int) * (size_t)n_slices));
        if (ws.zflags_host_n < (size_t)n_slices) {
            if (ws.zflags_host) { cudaFreeHost(ws.zflags_host); ws.zflags_host = nullptr; ws.zflags_host_n = 0; }
            CUDA_TRY(cudaHostAlloc(reinterpret_cast<void**>(&ws.zflags_host), sizeof(int) * (size_t)n_slices, cudaHostAllocDefault));
            ws.zflags_host_n = (size_t)n_slices;
        }
        CUDA_TRY(cudaMemsetAsync(ws.zflags.p, 0, sizeof(int) * (size_t)n_slices, stream));
    }
    // worker t rebuilds the V rows of chains [c0, c1) slice by slice, as soon as each slice's bits are on the host
    std::atomic<int64_t> enqueued{0};
    std::atomic<bool> abort_workers{false};
    int cur_dev = 0;
    cudaGetDevice(&cur_dev);
    auto worker = [&](int64_t c0, int64_t c1) {
        cudaSetDevice(cur_dev);
        for (int64_t it = 0; it < n_slices; ++it) {
            while (enqueued.load(std::memory_order_acquire) <= it) {
                if (abort_workers.load(std::memory_order_relaxed)) return;
                std::this_thread::yield();
            }
            if (cudaEventSynchronize(ws.slice_copied[(size_t)it]) != cudaSuccess) return;
            const int64_t k0 = it * slice, n = std::min<int64_t>(slice, n_sk - k0);
            if (zskip && ws.zflags_host[it] == 0)
                for (int64_t c = c0; c < c1; ++c) {
                    std::memset(hist->error_value_ar + ((size_t)c * hist->n_cols + k0) * 5, 0, sizeof(double) * 5 * (size_t)n);
                    std::memset(hist->errored_bound + (size_t)c * hist->n_cols + k0, 0, sizeof(int32_t) * (size_t)n);
                }
            const uint32_t* bits = ws.vbits_host + (size_t)it * vstride;
            for (int64_t c = c0; c < c1; ++c) {
                const uint64_t* au = reinterpret_cast<const uint64_t*>(absv.data() + (size_t)c * d);  // |v| >= 0: OR the sign in
                for (int64_t k = 0; k < n; ++k) {
                    const uint32_t* w = bits + ((size_t)c * slice + k) * vwords;
                    uint64_t* ou = reinterpret_cast<uint64_t*>(hist->V + ((size_t)c * hist->n_cols + k0 + k) * d);
                    int i = 0;
#if defined(__x86_64__)
                    if ((reinterpret_cast<uintptr_t>(ou) & 15) == 0) {  // two coordinates per streaming (write-combining) store
                        alignas(16) static const uint64_t kMask[4][2] = {{0, 0}, {1ull << 63, 0}, {0, 1ull << 63}, {1ull << 63, 1ull << 63}};
                        for (; i + 2 <= d; i += 2) {
                            const uint32_t two = (w[i >> 5] >> (i & 31)) & 3u;
                            const __m128i m = _mm_load_si128(reinterpret_cast<const __m128i*>(kMask[two]));
                            const __m128i av = _mm_loadu_si128(reinterpret_cast<const __m128i*>(au + i));
                            _mm_stream_si128(reinterpret_cast<__m128i*>(ou + i), _mm_or_si128(av, m));
                        }
                    }
#endif
                    for (; i < d; ++i) ou[i] = au[i] | ((uint64_t)((w[i >> 5] >> (i & 31)) & 1u) << 63);
                }
            }
#if defined(__x86_64__)
            _mm_sfence();
#endif
        }
    };
    struct Workers {  // joined on every exit path
        std::vector<std::thread> pool;
        std::atomic<bool>* abort_flag;
        bool finished = false;
        void finish() { for (auto& th : pool) th.join(); pool.clear(); finished = true; }
        ~Workers() { if (!finished) { abort_flag->store(true); finish(); } }
    } workers{{}, &abort_workers};
    if (vbits)
        for (int t = 0; t < n_threads; ++t) workers.pool.emplace_back(worker, n_chains * t / n_threads, n_chains * (t + 1) / n_threads);
    for (int i = 0; i < n_slabs; ++i) {
        Slab& b = slab[i];
        CUDA_TRY(ensure(b.X, hist->X, sizeof(double) * d * n_chains * slice));
        CUDA_TRY(ensure(b.V, hist->V, sizeof(double) * d * n_chains * slice));
        b.view = pdmpflux_history{};
        b.view.X = hist->X ? b.X.as<double>() : nullptr; b.view.V = hist->V ? b.V.as<double>() : nullptr;
        if (!full_scalars) {
            CUDA_TRY(ensure(b.t, hist->t, sizeof(double) * n_chains * slice));
            CUDA_TRY(ensure(b.horizon, hist->horizon, sizeof(double) * n_chains * slice));
            CUDA_TRY(ensure(b.ar, hist->ar, sizeof(double) * n_chains * slice));
            CUDA_TRY(ensure(b.eva, hist->error_value_ar, sizeof(double) * 5 * n_chains * slice));
            CUDA_TRY(ensure(b.eb, hist->errored_bound, sizeof(int32_t) * n_chains * slice));
            CUDA_TRY(ensure(b.rej, hist->rejected, sizeof(int32_t) * n_chains * slice));
            CUDA_TRY(ensure(b.hh, hist->hitting_horizon, sizeof(int32_t) * n_chains * slice));
            b.view.t = hist->t ? b.t.as<double>() : nullptr; b.view.horizon = hist->horizon ? b.horizon.as<double>() : nullptr;
            b.view.ar = hist->ar ? b.ar.as<double>() : nullptr;
            b.view.error_value_ar = hist->error_value_ar ? b.eva.as<double>() : nullptr;
            b.view.errored_bound = hist->errored_bound ? b.eb.as<int32_t>() : nullptr;
            b.view.rejected = hist->rejected ? b.rej.as<int32_t>() : nullptr;
            b.view.hitting_horizon = hist->hitting_horizon ? b.hh.as<int32_t>() : nullptr;
        }
        b.view.n_cols = slice; b.view.on_device = 1;
        if (!b.done) CUDA_TRY(cudaEventCreateWithFlags(&b.done, cudaEventDisableTiming));
        if (!b.copied) CUDA_TRY(cudaEventCreateWithFlags(&b.copied, cudaEventDisableTiming));
    }
    // chain c: host dst + (c*n_cols + k0)*elem  <-  device src + c*src_ld*elem, n*elem bytes
    auto copy2d = [&](void* dst, const void* src, size_t elem, int64_t src_ld, int64_t k0, int64_t n) -> cudaError_t {
        return cudaMemcpy2DAsync(static_cast<char*>(dst) + (size_t)k0 * elem, (size_t)hist->n_cols * elem, src,
                                 (size_t)src_ld * elem, (size_t)n * elem, (size_t)n_chains, cudaMemcpyDeviceToHost, copy_stream);
    };
    int64_t k0 = 0, sc_copied = 0;
    int it = 0;
    while (k0 < n_sk) {
        Slab& b = slab[it % n_slabs];
        const int64_t n = std::min<int64_t>(slice, n_sk - k0);
        if (it >= n_slabs) CUDA_TRY(cudaStreamWaitEvent(stream, b.copied, 0));  // slab free again
        // columns [k0, k0+n): column 0 of the whole run is the initial state, the others are events
        const pdmpflux_history* hv = full_scalars ? &sc.view : &b.view;
        const int64_t hcol = full_scalars ? k0 : 0;
        RowsView rows{b.view.X, b.view.V, slice, 0};
        int64_t first = 0, nev = n;
        if (k0 == 0) {
            rc = launch(ch, 0, hv, hcol, stream, &rows);
            if (rc != PDMPFLUX_OK) return rc;
            first = 1; nev = n - 1;
        }
        if (nev > 0) {
            RowsView rows2{b.view.X, b.view.V, slice, first};
            rc = launch(ch, nev, hv, hcol + first, stream, &rows2);
            if (rc != PDMPFLUX_OK) return rc;
            ch->event0 += nev;
        }
        CUDA_TRY(cudaEventRecord(b.done, stream));
        CUDA_TRY(cudaStreamWaitEvent(copy_stream, b.done, 0));
        if (vbits) {
            pack_signs_kernel<<<592, 256, 0, stream>>>(b.view.V, d, n_chains, n, slice, vwords,
                                                       ws.vbits.as<uint32_t>() + (size_t)it * vstride);
            CUDA_TRY(cudaGetLastError());
            g_launches.fetch_add(1);
            if (zskip) {
                flag_nonzero_kernel<<<296, 256, 0, stream>>>(sc.view.errored_bound, n_chains, ldS, k0, n, ws.zflags.as<int>() + it);
                CUDA_TRY(cudaGetLastError());
                g_launches.fetch_add(1);
            }
            CUDA_TRY(cudaEventRecord(b.done, stream));
            CUDA_TRY(cudaStreamWaitEvent(copy_stream, b.done, 0));
        }
        if (hist->X) CUDA_TRY(copy2d(hist->X, b.view.X, sizeof(double) * d, slice, k0, n));
        if (vbits) {
            CUDA_TRY(cudaMemcpyAsync(ws.vbits_host + (size_t)it * vstride, ws.vbits.as<uint32_t>() + (size_t)it * vstride,
                                     sizeof(uint32_t) * vstride, cudaMemcpyDeviceToHost, copy_stream));
            if (zskip) CUDA_TRY(cudaMemcpyAsync(ws.zflags_host + it, ws.zflags.as<int>() + it, sizeof(int), cudaMemcpyDeviceToHost, copy_stream));
            CUDA_TRY(cudaEventRecord(ws.slice_copied[(size_t)it], copy_stream));
            enqueued.store(it + 1, std::memory_order_release);
        } else if (hist->V) CUDA_TRY(copy2d(hist->V, b.view.V, sizeof(double) * d, slice, k0, n));
        if (!full_scalars) {
            if (hist->t) CUDA_TRY(copy2d(hist->t, b.view.t, sizeof(double), slice, k0, n));
            if (hist->horizon) CUDA_TRY(copy2d(hist->horizon, b.view.horizon, sizeof(double), slice, k0, n));
            if (hist->ar) CUDA_TRY(copy2d(hist->ar, b.view.ar, sizeof(double), slice, k0, n));
            if (hist->error_value_ar) CUDA_TRY(copy2d(hist->error_value_ar, b.view.error_value_ar, sizeof(double) * 5, slice, k0, n));
            if (hist->errored_bound) CUDA_TRY(copy2d(hist->errored_bound, b.view.errored_bound, sizeof(int32_t), slice, k0, n));
            if (hist->rejected) CUDA_TRY(copy2d(hist->rejected, b.view.rejected, sizeof(int32_t), slice, k0, n));
            if (hist->hitting_horizon) CUDA_TRY(copy2d(hist->hitting_horizon, b.view.hitting_horizon, sizeof(int32_t), slice, k0, n));
        }
        CUDA_TRY(cudaEventRecord(b.copied, copy_stream));
        k0 += n;
        ++it;
        // The scalar columns follow in a few wide chunks (rows of >= 256 columns) behind the X rows on the copy stream
        // (which already waits for this slice's kernel), so that only the last chunk is left after the last kernel.
        if (full_scalars && (k0 == n_sk || k0 - sc_copied >= 256)) {
            const int64_t a = sc_copied, m = k0 - sc_copied;
            auto src = [&](auto* base, size_t elems) { return base + (size_t)a * elems; };
            if (hist->t) CUDA_TRY(copy2d(hist->t, src(sc.view.t, 1), sizeof(double), ldS, a, m));
            if (hist->horizon) CUDA_TRY(copy2d(hist->horizon, src(sc.view.horizon, 1), sizeof(double), ldS, a, m));
            if (hist->ar) CUDA_TRY(copy2d(hist->ar, src(sc.view.ar, 1), sizeof(double), ldS, a, m));
            if (hist->error_value_ar && !zskip) CUDA_TRY(copy2d(hist->error_value_ar, src(sc.view.error_value_ar, 5), sizeof(double) * 5, ldS, a, m));
            if (hist->errored_bound && !zskip) CUDA_TRY(copy2d(hist->errored_bound, src(sc.view.errored_bound, 1), sizeof(int32_t), ldS, a, m));
            if (hist->rejected) CUDA_TRY(copy2d(hist->rejected, src(sc.view.rejected, 1), sizeof(int32_t), ldS, a, m));
            if (hist->hitting_horizon) CUDA_TRY(copy2d(hist->hitting_horizon, src(sc.view.hitting_horizon, 1), sizeof(int32_t), ldS, a, m));
            sc_copied = k0;
        }
    }
    CUDA_TRY(cudaStreamSynchronize(stream));
    CUDA_TRY(cudaStreamSynchronize(copy_stream));
    workers.finish();  // the V rows of the last slices
    int64_t z_copied_cols = 0;
    if (zskip) {  // the rare slices with a non-zero errored_bound: copy their two columns after all
        for (int64_t i = 0; i < n_slices; ++i)
            if (ws.zflags_host[i] != 0) {
                const int64_t a = i * slice, m = std::min<int64_t>(slice, n_sk - a);
                CUDA_TRY(copy2d(hist->error_value_ar, sc.view.error_value_ar + (size_t)a * 5, sizeof(double) * 5, ldS, a, m));
                CUDA_TRY(copy2d(hist->errored_bound, sc.view.errored_bound + (size_t)a, sizeof(int32_t), ldS, a, m));
                z_copied_cols += m;
            }
        CUDA_TRY(cudaStreamSynchronize(copy_stream));
    }
    {   // what actually crossed PCIe (bench.py reports it next to the end-to-end number)
        const int64_t cols = n_chains * n_sk;
        int64_t out = cols * ((hist->X ? 8 * d : 0) + (hist->t ? 8 : 0) + (hist->horizon ? 8 : 0) + (hist->ar ? 8 : 0) +
                              (hist->error_value_ar ? 40 : 0) + (hist->errored_bound ? 4 : 0) + (hist->rejected ? 4 : 0) +
                              (hist->hitting_horizon ? 4 : 0));
        if (vbits) out += (int64_t)(sizeof(uint32_t) * vstride * (size_t)n_slices);
        else if (hist->V) out += cols * 8 * d;
        if (zskip) out += n_slices * 4 - (n_sk - z_copied_cols) * n_chains * 44;
        g_d2h_bytes.store(out);
        g_h2d_bytes.store(2 * 8 * (int64_t)d * n_chains);
    }
    return finish(pdmpflux_chains_status(ch, hist->status, hist->tape_pos, hist->counters));
}

static int interp_impl(int flow_kind, int dim, int64_t n_sk, int64_t ld_sk, int64_t n_chains, const double* X,
                       const double* V, const double* t, int64_t N, double dt_fixed, int32_t discard_vt, double* out,
                       int32_t on_device, void* stream_, const uint8_t* act = nullptr);

int pdmpflux_sample_from_skeleton_sticky(int dim, int64_t n_sk, int64_t n_chains, const double* X, const double* V,
                                         const double* t, const uint8_t* is_active, int64_t N, int32_t discard_vt,
                                         double* out, int32_t on_device, void* stream_) {
    if (N <= 0) return fail(PDMPFLUX_ERR_ARGUMENT, "N must be positive. Current value: " + std::to_string(N));
    return interp_impl(0, dim, n_sk, n_sk, n_chains, X, V, t, N, 0.0, discard_vt, out, on_device, stream_, is_active);
}

int pdmpflux_sample_from_skeleton(int flow_kind, int dim, int64_t n_sk, int64_t n_chains, const double* X,
                                  const double* V, const double* t, int64_t N, int32_t discard_vt, double* out,
                                  int32_t on_device, void* stream_) {
    if (N <= 0) return fail(PDMPFLUX_ERR_ARGUMENT, "N must be positive. Current value: " + std::to_string(N));
    return interp_impl(flow_kind, dim, n_sk, n_sk, n_chains, X, V, t, N, 0.0, discard_vt, out, on_device, stream_);
}

int pdmpflux_sample_from_skeleton_dt(int flow_kind, int dim, int64_t n_sk, int64_t ld_sk, int64_t n_chains,
                                     const double* X, const double* V, const double* t, double dt, int64_t n_out,
                                     int32_t discard_vt, double* out, int32_t on_device, void* stream_) {
    if (!(dt > 0.0) || !std::isfinite(dt)) return fail(PDMPFLUX_ERR_ARGUMENT, "dt must be positive and finite");
    if (n_out <= 0 || ld_sk < n_sk) return fail(PDMPFLUX_ERR_ARGUMENT, "n_out must be positive and ld_sk >= n_sk");
    return interp_impl(flow_kind, dim, n_sk, ld_sk, n_chains, X, V, t, n_out, dt, discard_vt, out, on_device, stream_);
}

static int interp_impl(int flow_kind, int dim, int64_t n_sk, int64_t ld_sk, int64_t n_chains, const double* X,
                       const double* V, const double* t, int64_t N, double dt_fixed, int32_t discard_vt, double* out,
                       int32_t on_device, void* stream_, const uint8_t* act) {
    if (!X || !V || !t || !out || dim <= 0 || n_sk <= 0 || n_chains <= 0) return fail(PDMPFLUX_ERR_ARGUMENT, "invalid argument");
    if (flow_kind < 0 || flow_kind > 2) return fail(PDMPFLUX_ERR_ARGUMENT, "flow_kind must be 0 (linear), 1 (rotation) or 2 (Speed-Up Zig-Zag)");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const int ld = discard_vt ? dim : 2 * dim + 1;
    DevBuf dX, dV, dt, dout, dact, dsu;
    const double *pX = X, *pV = V, *pt = t;
    const uint8_t* pact = act;
    double* po = out;
    if (!on_device) {
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(PDMPFLUX_ERR_CUDA, "no CUDA device: no CPU fallback");
        const size_t nx = sizeof(double) * dim * ld_sk * n_chains;
        if (act) {
            CUDA_TRY(dact.alloc((size_t)dim * ld_sk * n_chains));
            CUDA_TRY(cudaMemcpyAsync(dact.p, act, (size_t)dim * ld_sk * n_chains, cudaMemcpyHostToDevice, stream));
            pact = dact.as<uint8_t>();
        }
        CUDA_TRY(dX.alloc(nx)); CUDA_TRY(dV.alloc(nx)); CUDA_TRY(dt.alloc(sizeof(double) * ld_sk * n_chains));
        CUDA_TRY(dout.alloc(sizeof(double) * ld * N * n_chains));
        CUDA_TRY(cudaMemcpyAsync(dX.p, X, nx, cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemcpyAsync(dV.p, V, nx, cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemcpyAsync(dt.p, t, sizeof(double) * ld_sk * n_chains, cudaMemcpyHostToDevice, stream));
        pX = dX.as<double>(); pV = dV.as<double>(); pt = dt.as<double>(); po = dout.as<double>();
    }
    const int64_t total = N * (int64_t)ld;
    if (flow_kind == 2) {
        const int64_t rows = n_chains * ld_sk;
        CUDA_TRY(dsu.alloc(sizeof(double) * 4 * (size_t)rows));
        speedup_scalars_kernel<<<(unsigned)((rows * 32 + 255) / 256), 256, 0, stream>>>(dim, rows, pX, pV, dsu.as<double>());
        CUDA_TRY(cudaGetLastError());
        g_launches.fetch_add(1);
    }
    dim3 grid((unsigned)n_chains, (unsigned)std::min<int64_t>((total + 255) / 256, 65535));
    interp_kernel<<<grid, 256, 0, stream>>>(flow_kind, dim, n_sk, ld_sk, N, discard_vt, dt_fixed, pX, pV, pt, pact, dsu.as<double>(), po);
    CUDA_TRY(cudaGetLastError());
    g_launches.fetch_add(1);
    if (!on_device) {
        CUDA_TRY(cudaMemcpyAsync(out, po, sizeof(double) * ld * N * n_chains, cudaMemcpyDeviceToHost, stream));
        CUDA_TRY(cudaStreamSynchronize(stream));
    } else if (flow_kind == 2) CUDA_TRY(cudaStreamSynchronize(stream));  // the segment scalars are freed on return
    return PDMPFLUX_OK;
}

int pdmpflux_skeleton_moments(int flow_kind, int dim, int64_t n_sk, int64_t n_chains, int64_t col_begin,
                              const double* X, const double* V, const double* t, double* m1, double* m2, double* T,
                              int32_t on_device, void* stream_) {
    if (!X || !V || !t || !m1 || !m2 || dim <= 0 || n_sk <= 1 || n_chains <= 0 || col_begin < 0 || col_begin >= n_sk - 1)
        return fail(PDMPFLUX_ERR_ARGUMENT, "invalid argument");
    if (flow_kind != 0 && flow_kind != 1) return fail(PDMPFLUX_ERR_UNSUPPORTED, "closed-form segment integrals exist for the linear and rotation flows only");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    DevBuf dX, dV, dt, d1, d2, dT;
    const double *pX = X, *pV = V, *pt = t;
    double *p1 = m1, *p2 = m2, *pT = T;
    if (!on_device) {
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(PDMPFLUX_ERR_CUDA, "no CUDA device: no CPU fallback");
        const size_t nx = sizeof(double) * dim * n_sk * n_chains;
        CUDA_TRY(dX.alloc(nx)); CUDA_TRY(dV.alloc(nx)); CUDA_TRY(dt.alloc(sizeof(double) * n_sk * n_chains));
        CUDA_TRY(d1.alloc(sizeof(double) * dim * n_chains)); CUDA_TRY(d2.alloc(sizeof(double) * dim * n_chains));
        CUDA_TRY(dT.alloc(sizeof(double) * n_chains));
        CUDA_TRY(cudaMemcpyAsync(dX.p, X, nx, cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemcpyAsync(dV.p, V, nx, cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemcpyAsync(dt.p, t, sizeof(double) * n_sk * n_chains, cudaMemcpyHostToDevice, stream));
        pX = dX.as<double>(); pV = dV.as<double>(); pt = dt.as<double>();
        p1 = d1.as<double>(); p2 = d2.as<double>(); pT = dT.as<double>();
    }
    const int64_t total = n_chains * dim;
    auto kern = flow_kind == 1 ? moments_kernel<1> : moments_kernel<0>;
    kern<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(dim, n_sk, n_chains, col_begin, pX, pV, pt, p1, p2, pT);
    CUDA_TRY(cudaGetLastError());
    g_launches.fetch_add(1);
    if (!on_device) {
        CUDA_TRY(cudaMemcpyAsync(m1, p1, sizeof(double) * dim * n_chains, cudaMemcpyDeviceToHost, stream));
        CUDA_TRY(cudaMemcpyAsync(m2, p2, sizeof(double) * dim * n_chains, cudaMemcpyDeviceToHost, stream));
        if (T) CUDA_TRY(cudaMemcpyAsync(T, pT, sizeof(double) * n_chains, cudaMemcpyDeviceToHost, stream));
        CUDA_TRY(cudaStreamSynchronize(stream));
    }
    return PDMPFLUX_OK;
}

int pdmpflux_rv_diagnostic(pdmpflux_potential_t pot, int flow_kind, int64_t n_sk, int64_t ld_sk, int64_t n_chains,
                           const int64_t* ncols, int64_t B, const double* X, const double* V, const double* t,
                           double* rv, int32_t on_device, void* stream_) {
    if (!pot || !X || !V || !t || !rv || n_sk <= 0 || ld_sk < n_sk || n_chains <= 0)
        return fail(PDMPFLUX_ERR_ARGUMENT, "invalid argument");
    if (pot->kind == PDMPFLUX_SOURCE)
        return fail(PDMPFLUX_ERR_UNSUPPORTED, "RV_diagnostic needs U(x), which a source potential does not define (it gives grad U only)");
    if (B < 0) return fail(PDMPFLUX_ERR_ARGUMENT, "B must be non-negative");  // diagnostic.jl:49-51
    if (flow_kind != 0 && flow_kind != 1) return fail(PDMPFLUX_ERR_ARGUMENT, "flow_kind must be 0 (linear) or 1 (rotation)");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(PDMPFLUX_ERR_CUDA, "no CUDA device: no CPU fallback");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const int dim = pot->dim;
    const int64_t ld_u = (B > 0 ? B : (int64_t)std::floor(std::sqrt((double)n_sk)) + 1) + 1;
    DevBuf dX, dV, dt, dn, du, drv;
    const double *pX = X, *pV = V, *pt = t;
    const int64_t* pn = ncols;
    double* prv = rv;
    CUDA_TRY(du.alloc(sizeof(double) * ld_u * n_chains));
    if (!on_device) {
        const size_t nx = sizeof(double) * dim * ld_sk * n_chains;
        CUDA_TRY(dX.alloc(nx)); CUDA_TRY(dV.alloc(nx)); CUDA_TRY(dt.alloc(sizeof(double) * ld_sk * n_chains));
        CUDA_TRY(drv.alloc(sizeof(double) * n_chains));
        CUDA_TRY(cudaMemcpyAsync(dX.p, X, nx, cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemcpyAsync(dV.p, V, nx, cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemcpyAsync(dt.p, t, sizeof(double) * ld_sk * n_chains, cudaMemcpyHostToDevice, stream));
        if (ncols) {
            CUDA_TRY(dn.alloc(sizeof(int64_t) * n_chains));
            CUDA_TRY(cudaMemcpyAsync(dn.p, ncols, sizeof(int64_t) * n_chains, cudaMemcpyHostToDevice, stream));
            pn = dn.as<int64_t>();
        }
        pX = dX.as<double>(); pV = dV.as<double>(); pt = dt.as<double>(); prv = drv.as<double>();
    }
    CUDA_TRY(launch_rv_diagnostic(pot->kind, pot->pp, flow_kind, dim, ld_sk, n_sk, n_chains, pn, B, pX, pV, pt,
                                  du.as<double>(), ld_u, prv, stream));
    g_launches.fetch_add(1);
    if (!on_device) CUDA_TRY(cudaMemcpyAsync(rv, prv, sizeof(double) * n_chains, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));  // the scratch row is freed on return
    return PDMPFLUX_OK;
}

int pdmpflux_host_alloc(void** ptr, size_t bytes) {
    if (!ptr) return fail(PDMPFLUX_ERR_ARGUMENT, "ptr is NULL");
    CUDA_TRY(cudaHostAlloc(ptr, bytes, cudaHostAllocDefault));
    return PDMPFLUX_OK;
}
int pdmpflux_host_free(void* ptr) {
    CUDA_TRY(cudaFreeHost(ptr));
    return PDMPFLUX_OK;
}

#pragma GCC visibility pop
}  // extern "C"
