// Counter-based draws for the thinning loop (device side).
//
// Philox4x32-10 keyed by (seed, global chain id, event index), as BASELINE.json's north_star asks
// (the reference installs MersenneTwister(seed), AbstractPDMP.jl:100-101, whose stream no test pins).
//   key     = (seed lo32, seed hi32)
//   counter = (call index, event index, chain lo32, stream | chain hi bits << 8)
//   stream 0 = E (randexp), 1 = U (rand), 2 = N (randn); slot counters restart at every event.
//   E slot s : -log((k52 + 0.5) * 2^-52)            k52 = top 52 bits of (r1:r0)
//   U slot s : k53 * 2^-53                           k53 = top 53 bits of (r1:r0)
//   N slot j : call j>>1, Box-Muller: sqrt(-2 log u1) * (j&1 ? sin : cos)(2 pi u2)
// The same specification is restated for the CPU in oracle/pdmp_draws.h (test infrastructure).
#pragma once
#ifdef __CUDACC_RTC__
#include "common.cuh"  // fixed-width types
#else
#include <cstdint>
#endif

namespace pdmpflux {

__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t (&out)[4]) {
    constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t h0 = __umulhi(M0, c0), l0 = M0 * c0;
        const uint32_t h1 = __umulhi(M1, c2), l1 = M1 * c2;
        const uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
        c0 = n0; c1 = l1; c2 = n2; c3 = l0;
        k0 += W0; k1 += W1;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__device__ __forceinline__ double u53(uint32_t lo, uint32_t hi) {
    const uint64_t k = ((static_cast<uint64_t>(hi) << 32) | lo) >> 11;
    return static_cast<double>(k) * 0x1.0p-53;
}
__device__ __forceinline__ double u52_open(uint32_t lo, uint32_t hi) {
    const uint64_t k = ((static_cast<uint64_t>(hi) << 32) | lo) >> 12;
    return (static_cast<double>(k) + 0.5) * 0x1.0p-52;
}

struct DrawKey {
    uint32_t k0, k1, chain_lo, chain_hi8;
    uint32_t event;
};

__device__ __forceinline__ void draw_call(const DrawKey& k, uint32_t stream, uint32_t call, uint32_t (&r)[4]) {
    philox4x32_10(call, k.event, k.chain_lo, stream | k.chain_hi8, k.k0, k.k1, r);
}
__device__ __forceinline__ double draw_exp(const DrawKey& k, uint32_t slot) {
    uint32_t r[4];
    draw_call(k, 0u, slot, r);
    return -log(u52_open(r[0], r[1]));
}
__device__ __forceinline__ double draw_uniform(const DrawKey& k, uint32_t slot) {
    uint32_t r[4];
    draw_call(k, 1u, slot, r);
    return u53(r[0], r[1]);
}
// Both normals of Box-Muller pair `pair` (slots 2*pair and 2*pair+1): one Philox call, one log, one sincospi.
// cos/sin(2 pi u) are evaluated as sincospi(2u): no range reduction, and exact at the quadrant boundaries.
__device__ __forceinline__ void draw_normal_pair(const DrawKey& k, uint32_t pair, double& n_even, double& n_odd) {
    uint32_t r[4];
    draw_call(k, 2u, pair, r);
    const double rad = sqrt(-2.0 * log(u52_open(r[0], r[1])));
    double s, c;
    sincospi(2.0 * u53(r[2], r[3]), &s, &c);
    n_even = rad * c;
    n_odd = rad * s;
}
__device__ __forceinline__ double draw_normal(const DrawKey& k, uint32_t slot) {
    double a, b;
    draw_normal_pair(k, slot >> 1, a, b);
    return (slot & 1u) ? b : a;
}

}  // namespace pdmpflux
