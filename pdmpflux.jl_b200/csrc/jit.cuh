// Source potentials (jit.cu): run-time compiled generic kernels for user-written potentials.  Every entry point
// returns a pdmpflux_error code and sets the thread-local error message.
#pragma once
#include <string>

#include "common.cuh"

namespace pdmpflux {

// compiles the contract check of a user source (no CUDA runtime call): PDMPFLUX_ERR_COMPILE with the NVRTC log
int jit_check_source(const std::string& source);
// compiles skeleton_kernel<team, sampler_kind, PDMPFLUX_SOURCE, kPathGeneric, 0> for the source (cached; no CUDA call)
int jit_prepare(const std::string& source, int sampler_kind, int team);
// launches that kernel (compiling it first if needed) with the same parameters as the built-in instantiations
int jit_launch(const std::string& source, int sampler_kind, int team, const KernelParams& p, unsigned grid, size_t smem,
               cudaStream_t stream);
// NVRTC compiles so far in this process
int64_t jit_compile_count();

}  // namespace pdmpflux
