// Host-side dispatch from (team width, potential kind) to a kernel instantiation.
#pragma once
#include "chain.cuh"

namespace pdmpflux {

// Zig-Zag + Brent on a team of lanes: which line model the kernel keeps (the NW template argument, common.cuh).
//   kLineTransposed  teams of 8 with at most 8 owned coordinates per lane (d <= 64) -- every lane keeps the chain's
//                    compressed model and takes its own iterations of the search (chain.cuh, build_bound_brent)
//   kLineRegs        teams of 8 with at most 16 owned coordinates per lane (d <= 128): register-resident (A_j, B_j),
//                    team reduction per rate evaluation
//   kLineShared      the shared-memory A/B arrays (every other team and sampler)
// launch_for_pot instantiates exactly these; api.cu sizes the shared memory with it.
inline int brent_line_model(int sampler, int path, int team, int n_own) {
    if (sampler != PDMPFLUX_ZIGZAG || path != kPathFastBrent || team != 8) return kLineShared;
    if (n_own <= 8) return kLineTransposed;
    return n_own <= kLineRegs ? kLineRegs : kLineShared;
}

// whether a sampler has a fast path (kPathFastBrent / kPathFastGrid) for a potential with these traits
constexpr bool has_fast_path(int sampler, bool affine, int n_special) {
    return affine && sampler != PDMPFLUX_STICKY_ZIGZAG   // masked velocities: per-node evaluation only
           && sampler != PDMPFLUX_SPEEDUP_ZIGZAG         // nonlinear flow: no affine line model
           && !(sampler == PDMPFLUX_BOOMERANG && n_special > 0);
}
template <int POT>
constexpr bool has_fast_path(int sampler) { return has_fast_path(sampler, Pot<POT>::kAffine, Pot<POT>::kSpecial); }

template <int TEAM, int SAMPLER, int POT, int PATH, int NW = kLineShared>
cudaError_t launch_one(const KernelParams& p, unsigned grid, size_t smem, cudaStream_t stream) {
    // no fast-path kernel is built where select_path never picks one
    constexpr bool ok = PATH == kPathGeneric || has_fast_path<POT>(SAMPLER);
    if constexpr (!ok) return cudaErrorInvalidValue;
    else {
        auto kern = skeleton_kernel<TEAM, SAMPLER, POT, PATH, NW>;
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        kern<<<grid, block_threads_rt(TEAM, SAMPLER, PATH), smem, stream>>>(p);
        return cudaGetLastError();
    }
}

template <int TEAM, int SAMPLER, int POT>
cudaError_t launch_for_pot(int path, const KernelParams& p, unsigned grid, size_t smem, cudaStream_t stream) {
    switch (path) {
    case kPathGeneric: return launch_one<TEAM, SAMPLER, POT, kPathGeneric>(p, grid, smem, stream);
    case kPathFastBrent:
        if constexpr (TEAM == 8 && SAMPLER == PDMPFLUX_ZIGZAG && Pot<POT>::kAffine) {
            switch (p.brent_nw) {
            case kLineTransposed: return launch_one<TEAM, SAMPLER, POT, kPathFastBrent, kLineTransposed>(p, grid, smem, stream);
            case kLineRegs: return launch_one<TEAM, SAMPLER, POT, kPathFastBrent, kLineRegs>(p, grid, smem, stream);
            }
        }
        return launch_one<TEAM, SAMPLER, POT, kPathFastBrent>(p, grid, smem, stream);
    case kPathFastGrid: return launch_one<TEAM, SAMPLER, POT, kPathFastGrid>(p, grid, smem, stream);
    default: return cudaErrorInvalidValue;
    }
}

template <int TEAM, int SAMPLER>
cudaError_t launch_for_team(int pot, int path, const KernelParams& p, unsigned grid, size_t smem, cudaStream_t stream) {
    switch (pot) {
    case PDMPFLUX_GAUSS_STD: return launch_for_pot<TEAM, SAMPLER, PDMPFLUX_GAUSS_STD>(path, p, grid, smem, stream);
    case PDMPFLUX_GAUSS_DIAG: return launch_for_pot<TEAM, SAMPLER, PDMPFLUX_GAUSS_DIAG>(path, p, grid, smem, stream);
    case PDMPFLUX_GAUSS_EQUICORR: return launch_for_pot<TEAM, SAMPLER, PDMPFLUX_GAUSS_EQUICORR>(path, p, grid, smem, stream);
    case PDMPFLUX_BANANA: return launch_for_pot<TEAM, SAMPLER, PDMPFLUX_BANANA>(path, p, grid, smem, stream);
    case PDMPFLUX_BANANA_README_SCALAR:
        return launch_for_pot<TEAM, SAMPLER, PDMPFLUX_BANANA_README_SCALAR>(path, p, grid, smem, stream);
    default: return cudaErrorInvalidValue;
    }
}

template <int SAMPLER>
cudaError_t launch_for_sampler(int team, int pot, int path, const KernelParams& p, unsigned grid, size_t smem,
                               cudaStream_t stream) {
    switch (team) {
    case 1: return launch_for_team<1, SAMPLER>(pot, path, p, grid, smem, stream);
    case 8: return launch_for_team<8, SAMPLER>(pot, path, p, grid, smem, stream);
    case 32: return launch_for_team<32, SAMPLER>(pot, path, p, grid, smem, stream);
    default: return cudaErrorInvalidValue;
    }
}

// the line-model traits (kAffine, kSpecial) of a built-in potential kind (potentials.cuh); none for the others
struct LineTraits { bool affine = false; int special = 0; };
inline LineTraits builtin_line_traits(int pot) {
    switch (pot) {
    case PDMPFLUX_GAUSS_STD: return {Pot<PDMPFLUX_GAUSS_STD>::kAffine, Pot<PDMPFLUX_GAUSS_STD>::kSpecial};
    case PDMPFLUX_GAUSS_DIAG: return {Pot<PDMPFLUX_GAUSS_DIAG>::kAffine, Pot<PDMPFLUX_GAUSS_DIAG>::kSpecial};
    case PDMPFLUX_GAUSS_EQUICORR: return {Pot<PDMPFLUX_GAUSS_EQUICORR>::kAffine, Pot<PDMPFLUX_GAUSS_EQUICORR>::kSpecial};
    case PDMPFLUX_BANANA: return {Pot<PDMPFLUX_BANANA>::kAffine, Pot<PDMPFLUX_BANANA>::kSpecial};
    case PDMPFLUX_BANANA_README_SCALAR:
        return {Pot<PDMPFLUX_BANANA_README_SCALAR>::kAffine, Pot<PDMPFLUX_BANANA_README_SCALAR>::kSpecial};
    default: return {};
    }
}

// which path a (sampler, potential traits, config) combination runs on: a fast path exactly where launch_one builds one
inline int select_path(int sampler, LineTraits pt, int grid_size, int vectorized, int deriv_mode) {
    if (!has_fast_path(sampler, pt.affine, pt.special)) return kPathGeneric;
    if (grid_size == 0) return kPathFastBrent;
    if (sampler == PDMPFLUX_ZIGZAG) {
        // vectorised bound with analytic derivatives only: with finite differences the reference's cell maximum
        // depends on the O(sqrt(eps)) derivative noise, which the affine shortcut does not reproduce
        if (!vectorized || deriv_mode != PDMPFLUX_DERIV_JVP) return kPathGeneric;
    }
    return kPathFastGrid;  // BPS / FECMC / Boomerang: closed-form nodes, analytic or finite-difference derivative
}

// logreg.cu: Zig-Zag x logistic regression, four chains per CTA sharing each pass over X, FP64 DMMA
cudaError_t launch_logreg_zigzag(const KernelParams& p, unsigned grid, size_t smem, cudaStream_t stream);
size_t logreg_smem_bytes(int d, int G);
int logreg_chains_per_block();

// diagnostic.cu: RV_diagnostic (src/diagnostic.jl:37-75) over a batch of skeletons; uval is a [C][ld_u >= B+1] scratch
cudaError_t launch_rv_diagnostic(int kind, const PotParams& pp, int flow_kind, int d, int64_t ld_sk, int64_t n_sk,
                                 int64_t n_chains, const int64_t* ncols, int64_t B, const double* X, const double* V,
                                 const double* t, double* uval, int64_t ld_u, double* rv, cudaStream_t stream);

cudaError_t launch_skeleton_zigzag(int team, int pot, int path, const KernelParams& p, unsigned grid, size_t smem, cudaStream_t stream);
cudaError_t launch_skeleton_bps(int team, int pot, int path, const KernelParams& p, unsigned grid, size_t smem, cudaStream_t stream);
cudaError_t launch_skeleton_fecmc(int team, int pot, int path, const KernelParams& p, unsigned grid, size_t smem, cudaStream_t stream);
cudaError_t launch_skeleton_boomerang(int team, int pot, int path, const KernelParams& p, unsigned grid, size_t smem, cudaStream_t stream);
cudaError_t launch_skeleton_sticky(int team, int pot, int path, const KernelParams& p, unsigned grid, size_t smem, cudaStream_t stream);
cudaError_t launch_skeleton_speedup(int team, int pot, int path, const KernelParams& p, unsigned grid, size_t smem, cudaStream_t stream);

}  // namespace pdmpflux
