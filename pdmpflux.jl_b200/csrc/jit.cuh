// Source potentials (jit.cu): run-time compiled kernels for user-written potentials.  Every entry point returns a
// pdmpflux_error code and sets the thread-local error message.
#pragma once
#include <string>

#include "common.cuh"

namespace pdmpflux {

// the traits of Pot<PDMPFLUX_SOURCE> (jit_source.cuh): what the source declares about its line model
struct SourceTraits {
    int K = 0;
    bool affine = false;
    int special = 0;
    bool split = false;
};

// compiles the contract check of a user source (no CUDA runtime call): PDMPFLUX_ERR_COMPILE with the NVRTC log; on
// success *traits (if not null) receives the declared traits
int jit_check_source(const std::string& source, SourceTraits* traits);
// compiles skeleton_kernel<team, sampler_kind, PDMPFLUX_SOURCE, path, nw> for the source (cached; no CUDA call)
int jit_prepare(const std::string& source, int sampler_kind, int team, int path, int nw);
// launches that kernel (compiling it first if needed) with the same parameters and block size as the built-in
// instantiations
int jit_launch(const std::string& source, int sampler_kind, int team, int path, int nw, const KernelParams& p,
               unsigned grid, size_t smem, cudaStream_t stream);
// NVRTC compiles so far in this process
int64_t jit_compile_count();

}  // namespace pdmpflux
