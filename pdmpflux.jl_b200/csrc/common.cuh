// Shared declarations for the thinning kernels: launch parameters, team (sub-warp) collectives.
#pragma once
#ifdef __CUDACC_RTC__  // run-time compiled (jit.cu): NVRTC has the CUDA built-ins but no C++ library headers
typedef unsigned char uint8_t;
typedef int int32_t;
typedef unsigned int uint32_t;
typedef long int64_t;            // LP64, as <cstdint> on the Linux hosts the library is built on
typedef unsigned long uint64_t;
#else
#include <cstdint>
#include <cuda_runtime.h>
#endif
#include <math_constants.h>

#include "../../include/pdmpflux_cuda.h"

namespace pdmpflux {

constexpr int kBlockThreads = 128;   // threads per block of every kernel except the one below

// PATH of a skeleton kernel (chain.cuh)
enum { kPathGeneric = 0, kPathFastBrent = 1, kPathFastGrid = 2 };

// Zig-Zag x Brent on a team of lanes: where the kernel keeps the line model (A_j, B_j) of the owned coordinates.  The
// value is the NW template argument of skeleton_kernel (launch.cuh: brent_line_model picks it).
constexpr int kLineShared = 0;       // shared-memory A / B vectors (also every kernel that has no Zig-Zag x Brent line model)
constexpr int kLineTransposed = -1;  // transposed Brent search: every lane keeps the chain's compressed model (chain.cuh)
constexpr int kLineRegs = 16;        // registers: at most kLineRegs owned coordinates per lane, one team reduction per rate

// shared-memory state vectors of a block before the scratch / flags / moments: x, v and, where the line model keeps
// them there, A and B
__host__ __device__ constexpr int state_vectors(int sampler, int path, int team, int line) {
    return sampler == PDMPFLUX_ZIGZAG && path == kPathFastBrent && team > 1 && line != kLineRegs ? 4 : 2;
}

// Thread-per-chain Zig-Zag x Brent is limited by the shared memory its chains' x and v take (16 d bytes per chain):
// blocks of 64 threads pack the SM with four blocks (8 warps) where blocks of 128 leave room for one or two.
// The same holds for thread-per-chain BPS / Boomerang / ForwardECMC at d ~ 100 (1.8 kB of state per chain): blocks of
// one warp.  (Thread-per-chain Zig-Zag with a grid bound is used at small d only and keeps 128.)
__host__ __device__ constexpr int block_threads_rt(int team, int sampler, int path) {
    if (team != 1) return kBlockThreads;
    if (sampler == PDMPFLUX_ZIGZAG) return path == kPathFastBrent ? 64 : kBlockThreads;
    if (sampler == PDMPFLUX_BPS || sampler == PDMPFLUX_FECMC || sampler == PDMPFLUX_BOOMERANG) return 32;
    return kBlockThreads;
}
constexpr int kMaxGrid = 64;        // largest supported grid_size (per-thread local arrays)
constexpr int kChunk = 8;           // grid nodes / cells processed per register chunk
constexpr double kSqrtEps = 1.4901161193847656e-08;
constexpr double kEps = 2.220446049250313e-16;

// Device-side potential parameters (owned by pdmpflux_potential_s).
struct PotParams {
    const double* vec;   // GAUSS_DIAG: p[d]; LOGREG: X[n*d]
    const double* vec2;  // LOGREG: y[n]
    double alpha, beta;  // GAUSS_EQUICORR
    double inv_s2;       // LOGREG prior precision
    int64_t n;           // LOGREG rows
};

// Everything a skeleton launch needs; passed by value (constant bank).
struct KernelParams {
    // sampler config after constructor rewrites
    int d, G, vectorized, signed_bound, adaptive, deriv_mode;
    int gaussian_velocity, ran_p, switch_, positive, max_steps;
    double tmax, refresh_rate, bound_refresh, mix_p, speed_factor;
    double inv_gm1;  // 1 / (grid_size - 1)
    PotParams pot;
    // chains
    int64_t n_chains, chain_offset;
    int64_t n_groups;  // groups of (kBlockThreads / TEAM) chains; > gridDim.x for a persistent grid
    uint64_t seed;
    int64_t event0;    // events already generated per chain (the next event has index event0+1)
    int64_t n_events;  // events to generate in this launch
    // PDMPState arrays (in/out)
    double* sx;        // [C][d]
    double* sv;        // [C][d]
    double* st;        // [C]
    double* shorizon;  // [C]
    double* sar;       // [C] last acceptance ratio (recorded in column 0 as 0)
    int64_t* tape_pos; // [C][3]
    int32_t* status;   // [C]
    int64_t* counters; // [C][2]
    int64_t* ncols;    // [C] history columns recorded so far (time-horizon variant)
    // logistic-regression kernel: chains beyond the first gridDim.x * 4 are pulled from a work queue (logreg.cu)
    int64_t* work_counter;  // device counter, zeroed before the launch (nullptr: no queue)
    int64_t work_start;     // index of the first queued chain
    // fused moments (no reference equivalent; SURVEY.md 8f.2): running time integrals of x_i and x_i^2 per chain,
    // accumulated segment by segment inside the flows, so moments / ESS need no stored skeleton
    int accumulate_moments;
    double* M1;        // [C][d] int x_i dt
    double* M2;        // [C][d] int x_i^2 dt
    // time-horizon variant (src/sample.jl:323-439): stop each chain at exactly t_stop
    int use_t_stop;
    double t_stop;
    // draws
    int draw_mode;  // 0 tape, 1 philox
    const double *tE, *tU, *tN;
    int64_t nE, nU, nN;
    // outputs (any may be null)
    double *X, *V, *T, *H, *AR, *EVA;
    int32_t *EB, *REJ, *HH;
    int64_t ld_cols, col0;        // scalar columns: leading dimension / first column of this launch
    int64_t ld_rows, col0_rows;   // X, V rows (may live in a narrower slab than the scalar columns)
    // Sticky Zig-Zag (StickySamplingLoop.jl): thawing rates, per-chain activity flags (state, in/out), is_active output
    const double* kappa;   // [d]
    uint8_t* sact;         // [C][d]
    uint8_t* ACT;          // [C][n_cols][d] (may be null)
    // per-block scratch vectors in global memory (used when they do not fit in shared memory)
    double* scratch;
    int scratch_in_smem;
    int n_own;      // ceil(d / TEAM)
    int brent_nw;   // Zig-Zag x Brent: the line model chosen at chains_create (kLine*, launch.cuh: brent_line_model)
    int vec_elems;  // doubles per shared-memory state vector of a block (x, v, A, B, scratch each take one)
    int dpad;       // TEAM > 1: doubles reserved per chain inside a state vector (chain-contiguous layout)
    // output path
    int sparse_cols;  // error_value_ar / errored_bound / rejected / hitting_horizon were zero-filled by the host:
                      // the kernel only writes their non-zero entries
    int vec32;        // X, V, t, horizon, ar are 32-byte aligned: 256-bit (one full sector) stores are legal
    int bulk_rows;    // TEAM > 1: X / V rows go out as TMA bulk copies straight from the shared-memory state
};

// ---- Blackwell store primitives ---------------------------------------------------------------------------
// 256-bit store: one full 32-byte DRAM sector per lane in a single request (SASS: STG.E.ENL2.256)
__device__ __forceinline__ void st256(double* g, double a, double b, double c, double d) {
    asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(g), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}
// TMA bulk copy shared -> global (SASS: UBLKCP.G.S); size and both addresses are multiples of 16 bytes
// History rows are written once and never read by the kernel: the L2 evict-first policy keeps them from displacing the
// per-block scratch vectors (and the chains' state) that live in the L2.
__device__ __forceinline__ void bulk_store(void* gdst, const void* ssrc, uint32_t bytes) {
    const uint32_t s = (uint32_t)__cvta_generic_to_shared(ssrc);
    uint64_t policy;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(gdst), "r"(s), "r"(bytes),
                 "l"(policy)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }


// ---- team collectives: TEAM consecutive lanes of a warp cooperate on one chain --------------------------
template <int TEAM>
__device__ __forceinline__ unsigned team_mask() {
    if constexpr (TEAM == 32) return 0xffffffffu;
    else {
        const unsigned lane = threadIdx.x & 31u;
        return ((1u << TEAM) - 1u) << (lane & ~(unsigned)(TEAM - 1));
    }
}

template <int TEAM>
__device__ __forceinline__ double team_sum(double v, unsigned mask) {
#pragma unroll
    for (int o = TEAM / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o);
    return v;  // butterfly: bitwise identical in every lane of the team
}

template <int TEAM, int N>
__device__ __forceinline__ void team_sum_n(double (&v)[N], unsigned mask) {
    if constexpr (TEAM > 1) {
#pragma unroll
        for (int o = TEAM / 2; o > 0; o >>= 1) {
#pragma unroll
            for (int i = 0; i < N; ++i) v[i] += __shfl_xor_sync(mask, v[i], o);
        }
    }
}

// inclusive scan over the team's lanes (in lane order)
template <int TEAM>
__device__ __forceinline__ double team_scan_incl(double v, unsigned mask, int tl) {
#pragma unroll
    for (int o = 1; o < TEAM; o <<= 1) {
        const double u = __shfl_up_sync(mask, v, o, TEAM);
        if (tl >= o) v += u;
    }
    return v;
}

// Team vote without vote.sync: a ballot whose member mask differs between the teams of a warp is compiled into a loop
// over the distinct masks (MATCH.ANY + REDUX + one VOTE per team: ~100 extra warp instructions per event and a fifth
// of the stall samples on the Zig-Zag x Brent kernel); an OR butterfly over the team's lanes is three shuffles.
template <int TEAM>
__device__ __forceinline__ unsigned team_or(unsigned v, unsigned mask) {
#pragma unroll
    for (int o = TEAM / 2; o > 0; o >>= 1) v |= __shfl_xor_sync(mask, v, o);
    return v;
}
template <int TEAM>
__device__ __forceinline__ unsigned long long team_or64(unsigned long long v, unsigned mask) {
#pragma unroll
    for (int o = TEAM / 2; o > 0; o >>= 1) v |= __shfl_xor_sync(mask, v, o);
    return v;
}
// bit tl of the result = pred of team lane tl (what ballot >> team shift gives)
template <int TEAM>
__device__ __forceinline__ unsigned team_ballot(bool pred, int tl, unsigned mask) {
    if constexpr (TEAM == 1) return pred ? 1u : 0u;
    else if constexpr (TEAM == 32) return __ballot_sync(0xffffffffu, pred);   // one mask for the whole warp: a plain VOTE
    else return team_or<TEAM>(pred ? (1u << tl) : 0u, mask);
}

template <int TEAM>
__device__ __forceinline__ double team_bcast(double v, int src_tl, unsigned mask) {
    if constexpr (TEAM == 1) return v;
    else return __shfl_sync(mask, v, src_tl, TEAM);
}

}  // namespace pdmpflux
