// Instantiations of the thinning kernel for the zigzag sampler (one translation unit per sampler so the
// build parallelises).  See chain.cuh for the device logic and the reference lines it replaces.
#include "chain.cuh"
#include "launch.cuh"

namespace pdmpflux {
cudaError_t launch_skeleton_zigzag(int team, int pot, int path, const KernelParams& p, unsigned grid, size_t smem,
                                 cudaStream_t stream) {
    return launch_for_sampler<PDMPFLUX_ZIGZAG>(team, pot, path, p, grid, smem, stream);
}
}  // namespace pdmpflux

#ifdef PDMPFLUX_PHASE_CLOCK
// Phase-clock build only (tools/phase_clock.py): copies the Zig-Zag kernels' kPhases + 1 counters (lane cycles per
// phase, then lane events) to out[] and zeroes them.
extern "C" __attribute__((visibility("default"))) int pdmpflux_phase_clock(unsigned long long* out) {
    using namespace pdmpflux;
    cudaError_t e = cudaMemcpyFromSymbol(out, g_phase_clock, sizeof(g_phase_clock));
    const unsigned long long zero[kPhases + 1] = {};
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(g_phase_clock, zero, sizeof(zero));
    return (int)e;
}
#endif
