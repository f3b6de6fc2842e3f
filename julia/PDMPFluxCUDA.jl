# PDMPFluxCUDA.jl -- Julia `ccall` glue over libpdmpflux_cuda.so (include/pdmpflux_cuda.h, ABI version 200).
#
# UNTESTED IN THIS REPOSITORY'S CI: the build image has no Julia.  The tested binding of the same C ABI is the
# ctypes one in pdmpflux.jl_b200/_lib.py (every call below has a ctypes twin there, exercised by tests/); this file is
# what a PDMPFlux.jl maintainer would add (see INTEGRATION.md).  It extends the reference's own functions and
# constructor names with methods that dispatch on a device-potential descriptor, and returns real
# `PDMPFlux.PDMPHistory` objects, so `diagnostic`, `plot_traj`, `anim_traj` of the reference work unchanged.
module PDMPFluxCUDA

import PDMPFlux
import PDMPFlux: PDMPHistory, sample_skeleton, sample_from_skeleton, sample, RV_diagnostic,
                 sample_skeleton_with_diagnostic
export CuPotential, GaussStd, GaussDiag, GaussEquicorr, GaussDense, Banana, BananaReadmeScalar, LogReg, CudaPotential, CuPDMP, CuHistoryBatch,
       moments_reduce, CuComm, comm_unique_id, moments_allreduce!

const LIB = get(ENV, "PDMPFLUX_CUDA_LIB", joinpath(@__DIR__, "..", "pdmpflux.jl_b200", "lib", "libpdmpflux_cuda.so"))

# ---- C structs (layout must match include/pdmpflux_cuda.h) -----------------------------------------------------
struct CConfig
    grid_size::Int32; vectorized_bound::Int32; signed_bound::Int32; adaptive::Int32; deriv_mode::Int32
    gaussian_velocity::Int32; ran_p::Int32; switch_::Int32; positive::Int32; max_steps::Int32
    tmax::Float64; refresh_rate::Float64; mix_p::Float64; speed_factor::Float64
end
struct CHistory
    X::Ptr{Float64}; V::Ptr{Float64}; t::Ptr{Float64}; horizon::Ptr{Float64}; ar::Ptr{Float64}
    error_value_ar::Ptr{Float64}; errored_bound::Ptr{Int32}; rejected::Ptr{Int32}; hitting_horizon::Ptr{Int32}
    status::Ptr{Int32}; tape_pos::Ptr{Int64}; counters::Ptr{Int64}; n_cols::Int64; on_device::Int32
    is_active::Ptr{UInt8}          # appended in ABI 200 (Sticky Zig-Zag only; C_NULL otherwise)
end

last_error() = unsafe_string(ccall((:pdmpflux_last_error, LIB), Cstring, ()))
function check(rc::Integer)
    rc == 0 && return
    msg = last_error()
    rc == -1 && throw(ArgumentError(msg))          # PDMPFLUX_ERR_ARGUMENT
    rc == -2 && throw(DimensionMismatch(msg))      # PDMPFLUX_ERR_DIMENSION_MISMATCH
    rc == -7 && throw(ErrorException("CudaPotential did not compile:\n" * msg))   # PDMPFLUX_ERR_COMPILE (NVRTC log)
    error("libpdmpflux_cuda ($rc): $msg")          # unsupported / CUDA / chain failure: there is no CPU fallback
end
function __init__()
    v = ccall((:pdmpflux_version, LIB), Cint, ())
    v >= 200 || error("libpdmpflux_cuda.so is older (version $v) than this binding (200)")
end

# ---- device potentials: replace the `∇U` / `U` closure ----------------------------------------------------------
struct CuPotential
    kind::Int32
    params::Vector{Float64}
    source::Union{Nothing,String}   # kind 6 (PDMPFLUX_SOURCE): user CUDA source
end
CuPotential(kind::Integer, params::Vector{Float64}) = CuPotential(Int32(kind), params, nothing)
GaussStd() = CuPotential(0, Float64[])
GaussDiag(p::AbstractVector) = CuPotential(1, collect(Float64, p))
GaussEquicorr(rho::Real) = CuPotential(2, [Float64(rho)])
# U = (x - mu)' P (x - mu) / 2, P dense symmetric positive definite (checked by the library); Zig-Zag and BPS only
GaussDense(P::AbstractMatrix, mu::AbstractVector = zeros(size(P, 1))) =
    CuPotential(7, vcat(vec(permutedims(Float64.(P))), Float64.(mu)))
Banana() = CuPotential(3, Float64[])
BananaReadmeScalar() = CuPotential(4, Float64[])
"Bayesian logistic regression posterior: rows of `X` (n × d), labels `y` in {0, 1}, prior N(0, sigma0² I).  X is
passed row-major, i.e. as the memory of `permutedims(X)`."
LogReg(X::AbstractMatrix, y::AbstractVector, sigma0::Real) =
    CuPotential(5, vcat(Float64(size(X, 1)), Float64(sigma0), vec(permutedims(Matrix{Float64}(X))), Vector{Float64}(y)))
"""
    CudaPotential(source, params=Float64[])

A potential written in CUDA C++: `source` defines `struct UserPotential` (K linear functionals, `accum`, `grad`,
`eval`; the contract is stated in include/pdmpflux_cuda.h above `pdmpflux_potential_create_source`) and `params` are
`pp.vec[0 .. pp.n-1]` on the device.  Compiled at run time with NVRTC when the sampler is constructed.

The optional members `affine`, `special`, `eval_local` and `line_corr` declare the potential's line model (same header)
and put it on the fast-path kernels of Zig-Zag, BPS and ForwardECMC; without them it runs the generic kernel.  The
library cannot check that the potential has the declared structure: a wrong declaration samples the wrong target.
"""
CudaPotential(source::AbstractString, params::AbstractVector=Float64[]) =
    CuPotential(Int32(6), collect(Float64, params), String(source))

"A sampler living on the GPU: what the reference constructors return when the second argument is a `CuPotential`."
mutable struct CuPDMP
    kind::Int32; dim::Int; pot::Ptr{Cvoid}; handle::Ptr{Cvoid}; flow_kind::Int32
    sticky::Bool
    state::Any
end
deriv_mode(ad::String) = ad in ("", "Undefined", "FiniteDiff") ? Int32(1) :
    (ad in ("ForwardDiff", "Zygote", "ReverseDiff", "Enzyme", "PolyesterForwardDiff") ? Int32(0) :
     throw(ArgumentError("Unsupported AD_backend: $ad")))

function CuPDMP(kind, dim::Int, pot::CuPotential, cfg::CConfig; kappa::Union{Nothing,Vector{Float64}}=nothing)
    dim <= 0 && throw(ArgumentError("dimension dim must be positive. Current value: $dim"))
    hp = Ref{Ptr{Cvoid}}(C_NULL)
    if pot.source === nothing
        check(ccall((:pdmpflux_potential_create, LIB), Cint, (Cint, Cint, Ptr{Float64}, Int64, Ref{Ptr{Cvoid}}),
                    pot.kind, dim, pot.params, length(pot.params), hp))
    else
        check(ccall((:pdmpflux_potential_create_source, LIB), Cint, (Cint, Cstring, Ptr{Float64}, Int64, Ref{Ptr{Cvoid}}),
                    dim, pot.source, pot.params, length(pot.params), hp))
    end
    hs = Ref{Ptr{Cvoid}}(C_NULL)
    rc = if kappa === nothing
        ccall((:pdmpflux_sampler_create, LIB), Cint, (Cint, Cint, Ptr{Cvoid}, Ref{CConfig}, Ref{Ptr{Cvoid}}),
              kind, dim, hp[], Ref(cfg), hs)
    else
        length(kappa) == dim || throw(DimensionMismatch("kappa must have length dim ($dim)"))
        ccall((:pdmpflux_sampler_create_sticky, LIB), Cint, (Cint, Ptr{Cvoid}, Ref{CConfig}, Ptr{Float64}, Ref{Ptr{Cvoid}}),
              dim, hp[], Ref(cfg), kappa, hs)
    end
    if rc != 0
        ccall((:pdmpflux_potential_destroy, LIB), Cint, (Ptr{Cvoid},), hp[])
        check(rc)
    end
    s = CuPDMP(kind, dim, hp[], hs[], kind == 3 ? 1 : (kind == 5 ? 2 : 0), kappa !== nothing, nothing)   # flow_kind
    finalizer(s) do x
        ccall((:pdmpflux_sampler_destroy, LIB), Cint, (Ptr{Cvoid},), x.handle)
        ccall((:pdmpflux_potential_destroy, LIB), Cint, (Ptr{Cvoid},), x.pot)
    end
    return s
end

# ---- the reference's constructor names, dispatched on the potential type --------------------------------------
# (ZigZagSamplers.jl:58-60 / :118-126, BouncyParticleSamplers.jl:21-24 / :86-94, ForwardEventChainMonteCarlo.jl:301-303 /
#  :367-378, BoomerangSamplers.jl:21-23 / :79-87, StickyZigZagSamplers.jl:60-62 / :117-127; same keywords and defaults)
PDMPFlux.ZigZag(dim::Int, pot::CuPotential; grid_size::Int=10, tmax=2.0, refresh_rate::Float64=0.0,
                vectorized_bound::Bool=true, signed_bound::Bool=true, adaptive::Bool=true, AD_backend::String="FiniteDiff") =
    CuPDMP(0, dim, pot, CConfig(grid_size, vectorized_bound, signed_bound, adaptive, deriv_mode(AD_backend), 0, 0, 1, 1, 0,
                                Float64(tmax), refresh_rate, 0.5, 1.0))
PDMPFlux.ZigZagAD(dim::Int, pot::CuPotential; refresh_rate::Float64=0.0, grid_size::Int=10, tmax=2.0,
                  vectorized_bound::Bool=true, signed_bound::Bool=true, adaptive::Bool=true, AD_backend::String="ForwardDiff") =
    PDMPFlux.ZigZag(dim, pot; grid_size, tmax, refresh_rate, vectorized_bound, signed_bound, adaptive, AD_backend)
PDMPFlux.BPS(dim::Int, pot::CuPotential; grid_size::Int=10, tmax=1.0, refresh_rate::Float64=0.1, vectorized_bound::Bool=false,
             signed_bound::Bool=true, adaptive::Bool=true, AD_backend::String="ForwardDiff", Gaussian_velocity::Bool=false) =
    CuPDMP(1, dim, pot, CConfig(grid_size, 0, signed_bound, adaptive, deriv_mode(AD_backend), Gaussian_velocity, 0, 1, 1, 0,
                                Float64(tmax), refresh_rate, 0.5, 1.0))
PDMPFlux.BPSAD(dim::Int, pot::CuPotential; refresh_rate::Float64=0.0, grid_size::Int=10, tmax=2.0, vectorized_bound::Bool=true,
               signed_bound::Bool=true, adaptive::Bool=true, AD_backend::String="ForwardDiff") =
    PDMPFlux.BPS(dim, pot; grid_size, tmax, refresh_rate, signed_bound, adaptive, AD_backend)
function PDMPFlux.ForwardECMC(dim::Int, pot::CuPotential; grid_size::Int=10, tmax=2.0, signed_bound::Bool=true,
                              adaptive::Bool=true, ran_p::Bool=false, mix_p::Float64=0.5, switch::Bool=true,
                              positive::Bool=true, AD_backend::String="ForwardDiff", speed_factor::Float64=1.0,
                              normal::Bool=false)
    dim < 2 && throw(ArgumentError("The dimension must be at least 2 to use the ForwardEventChain. Got dimension $dim"))
    normal && error("ForwardECMC(normal=true) throws upstream (ForwardEventChainMonteCarlo.jl:227) and is not offered on the device")
    CuPDMP(2, dim, pot, CConfig(grid_size, 0, signed_bound, adaptive, deriv_mode(AD_backend), 0, ran_p, switch, positive, 0,
                                Float64(tmax), 0.0, mix_p, speed_factor))
end
PDMPFlux.ForwardECMCAD(dim::Int, pot::CuPotential; kw...) = PDMPFlux.ForwardECMC(dim, pot; AD_backend="ForwardDiff", kw...)
PDMPFlux.Boomerang(dim::Int, pot::CuPotential; grid_size::Int=10, tmax=1.0, refresh_rate::Float64=0.1,
                   vectorized_bound::Bool=false, signed_bound::Bool=true, adaptive::Bool=true, AD_backend::String="FiniteDiff") =
    CuPDMP(3, dim, pot, CConfig(grid_size, 0, signed_bound, adaptive, deriv_mode(AD_backend), 0, 0, 1, 1, 0,
                                Float64(tmax), refresh_rate, 0.5, 1.0))
PDMPFlux.BoomerangAD(dim::Int, pot::CuPotential; refresh_rate::Float64=0.0, grid_size::Int=10, tmax=2.0,
                     vectorized_bound::Bool=true, signed_bound::Bool=true, adaptive::Bool=true, AD_backend::String="ForwardDiff") =
    PDMPFlux.Boomerang(dim, pot; grid_size, tmax, refresh_rate, signed_bound, adaptive, AD_backend)
PDMPFlux.StickyZigZag(dim::Int, pot::CuPotential, κ::Vector{Float64}; refresh_rate::Float64=0.0, grid_size::Int=10, tmax=2.0,
                      vectorized_bound::Bool=true, signed_bound::Bool=true, adaptive::Bool=true, AD_backend::String="FiniteDiff") =
    CuPDMP(4, dim, pot, CConfig(grid_size, vectorized_bound, signed_bound, adaptive, deriv_mode(AD_backend), 0, 0, 1, 1, 0,
                                Float64(tmax), refresh_rate, 0.5, 1.0); kappa=κ)
PDMPFlux.StickyZigZagAD(dim::Int, pot::CuPotential, κ::Vector{Float64}; kw...) =
    PDMPFlux.StickyZigZag(dim, pot, κ; AD_backend="ForwardDiff", kw...)
# SpeedUpZigZagSamplers.jl:58-60 / :119-129
PDMPFlux.SpeedUpZigZag(dim::Int, pot::CuPotential; grid_size::Int=10, tmax=2.0, refresh_rate::Float64=0.0,
                       vectorized_bound::Bool=true, signed_bound::Bool=true, adaptive::Bool=true, AD_backend::String="FiniteDiff") =
    CuPDMP(5, dim, pot, CConfig(grid_size, vectorized_bound, signed_bound, adaptive, deriv_mode(AD_backend), 0, 0, 1, 1, 0,
                                Float64(tmax), refresh_rate, 0.5, 1.0))
PDMPFlux.SpeedUpZigZagAD(dim::Int, pot::CuPotential; kw...) = PDMPFlux.SpeedUpZigZag(dim, pot; AD_backend="ForwardDiff", kw...)

# ---- histories ---------------------------------------------------------------------------------------------------
"""
    CuHistoryBatch <: AbstractVector{PDMPHistory{Float64}}

The skeletons of C chains as the library wrote them: chain-major arrays (`X[:, :, c]` is chain c's d × n_sk matrix).
`batch[c]` is a `PDMPHistory` whose `X`, `V`, `t`, ... ALIAS those arrays (`unsafe_wrap`, no copy): it stays valid as
long as `batch` is reachable.  `copy(batch[c])`-style independence needs `deepcopy`.  (`is_active` is a fresh
`BitMatrix`: the library stores bytes.)
"""
struct CuHistoryBatch <: AbstractVector{PDMPHistory{Float64}}
    X::Array{Float64,3}; V::Array{Float64,3}; t::Matrix{Float64}; horizon::Matrix{Float64}; ar::Matrix{Float64}
    error_value_ar::Array{Float64,3}; errored_bound::Matrix{Int32}; rejected::Matrix{Int32}; hitting_horizon::Matrix{Int32}
    is_active::Union{Nothing,Array{UInt8,3}}
    ncols::Vector{Int}        # columns in use per chain (ragged for the time-horizon method)
end
Base.size(b::CuHistoryBatch) = (size(b.t, 2),)
function Base.getindex(b::CuHistoryBatch, c::Int)
    d, cap, _ = size(b.X)
    n = b.ncols[c]
    mat(A, r) = unsafe_wrap(Array, pointer(A, 1 + (c - 1) * r * cap), (r, n))      # leading columns of chain c's slab
    vec_(A) = unsafe_wrap(Array, pointer(A, 1 + (c - 1) * cap), (n,))
    act = b.is_active === nothing ? trues(d, n) : BitMatrix(view(b.is_active, :, 1:n, c) .!= 0x00)
    PDMPHistory{Float64}(mat(b.X, d), mat(b.V, d), vec_(b.t), act, vec_(b.horizon), vec_(b.ar), vec_(b.errored_bound),
                         mat(b.error_value_ar, 5), vec_(b.rejected), vec_(b.hitting_horizon))
end

function _alloc_batch(d, cap, C, sticky)
    CuHistoryBatch(Array{Float64}(undef, d, cap, C), Array{Float64}(undef, d, cap, C), Matrix{Float64}(undef, cap, C),
                   Matrix{Float64}(undef, cap, C), Matrix{Float64}(undef, cap, C), Array{Float64}(undef, 5, cap, C),
                   Matrix{Int32}(undef, cap, C), Matrix{Int32}(undef, cap, C), Matrix{Int32}(undef, cap, C),
                   sticky ? Array{UInt8}(undef, d, cap, C) : nothing, fill(cap, C))
end
_chist(b::CuHistoryBatch, status, cap) =
    CHistory(pointer(b.X), pointer(b.V), pointer(b.t), pointer(b.horizon), pointer(b.ar), pointer(b.error_value_ar),
             pointer(b.errored_bound), pointer(b.rejected), pointer(b.hitting_horizon), pointer(status), C_NULL, C_NULL,
             cap, 0, b.is_active === nothing ? Ptr{UInt8}(C_NULL) : pointer(b.is_active))

_check_init(s, xinit, vinit) = (size(xinit, 1) == s.dim && size(vinit) == size(xinit)) ||
    throw(DimensionMismatch("xinit and vinit must have the same dimension as pdmp.dim ($(s.dim)). Current dimensions: xinit ($(size(xinit, 1))), vinit ($(size(vinit, 1)))"))

"""
    sample_skeleton(sampler::CuPDMP, n_sk::Int, xinit::Vector, vinit::Vector; seed) -> PDMPHistory   (one chain, as upstream)
    sample_skeleton(sampler::CuPDMP, n_sk::Int, xinit::Matrix, vinit::Matrix; seed) -> CuHistoryBatch (d × C initial states)

Replaces `PDMPFlux.sample_skeleton` (src/sample.jl:253-284).  The library writes every chain's slab straight into the
Julia arrays (chain-major layout = Julia column-major `d × n_sk × C`); no copy is made afterwards.
"""
function sample_skeleton(s::CuPDMP, n_sk::Int, xinit::Matrix{Float64}, vinit::Matrix{Float64};
                         seed::Union{Int,Nothing}=nothing, verbose::Bool=true, chain_offset::Int=0)
    n_sk <= 0 && throw(ArgumentError("n_sk must be positive. Current value: $n_sk"))
    _check_init(s, xinit, vinit)
    C = size(xinit, 2)
    b = _alloc_batch(s.dim, n_sk, C, s.sticky)
    status = zeros(Int32, C)
    sd = seed === nothing ? rand(UInt64) : UInt64(seed)
    GC.@preserve b status xinit vinit begin
        check(ccall((:pdmpflux_sample_skeleton, LIB), Cint,
                    (Ptr{Cvoid}, Int64, Int64, Ptr{Float64}, Ptr{Float64}, UInt64, Int64, Ptr{Cvoid}, Ref{CHistory}, Ptr{Cvoid}),
                    s.handle, C, n_sk, xinit, vinit, sd, chain_offset, C_NULL, Ref(_chist(b, status, n_sk)), C_NULL))
    end
    s.state = status
    return b
end
function sample_skeleton(s::CuPDMP, n_sk::Int, xinit::Vector{Float64}, vinit::Vector{Float64}; kw...)
    b = sample_skeleton(s, n_sk, reshape(xinit, :, 1), reshape(vinit, :, 1); kw...)
    d = s.dim
    # one chain: the slab IS the history's storage.  `reshape` / `vec` of an Array share its memory and are GC-safe,
    # so the PDMPHistory below owns the very buffers the library wrote (zero copy, no unsafe_wrap).
    act = b.is_active === nothing ? trues(d, n_sk) : BitMatrix(reshape(b.is_active, d, n_sk) .!= 0x00)
    return PDMPHistory{Float64}(reshape(b.X, d, n_sk), reshape(b.V, d, n_sk), vec(b.t), act, vec(b.horizon), vec(b.ar),
                                vec(b.errored_bound), reshape(b.error_value_ar, 5, n_sk), vec(b.rejected), vec(b.hitting_horizon))
end
sample_skeleton(s::CuPDMP, n_sk::Int, xinit::Float64, vinit::Float64; kw...) = sample_skeleton(s, n_sk, [xinit], [vinit]; kw...)

"""
    sample_skeleton(sampler::CuPDMP, T::Float64, xinit, vinit; seed, init_capacity=1024)

Replaces the time-horizon method (src/sample.jl:323-439) for one chain (`Vector` inits -> `PDMPHistory`) or C chains
(`Matrix` inits -> `CuHistoryBatch` with ragged `ncols`): every skeleton ends with the point at exactly `t == T`.  The
number of events is not known in advance: like `_grow_history` (src/Composites.jl:172-191) the capacity doubles until
every chain fits (`PDMPFLUX_ERR_CAPACITY = -6`; the run is deterministic, so it is simply repeated).
"""
function sample_skeleton(s::CuPDMP, T::Float64, xinit::Matrix{Float64}, vinit::Matrix{Float64};
                         seed::Union{Int,Nothing}=nothing, verbose::Bool=true, init_capacity::Int=1024, chain_offset::Int=0)
    (isfinite(T) && T >= 0) || throw(ArgumentError("T must be finite and non-negative. Current value: $T"))
    _check_init(s, xinit, vinit)
    C = size(xinit, 2)
    sd = seed === nothing ? rand(UInt64) : UInt64(seed)
    cap = max(1, init_capacity)
    while true
        b = _alloc_batch(s.dim, cap, C, false)
        status = zeros(Int32, C); ncols = zeros(Int64, C)
        rc = GC.@preserve b status ncols xinit vinit begin
            ccall((:pdmpflux_sample_skeleton_until, LIB), Cint,
                  (Ptr{Cvoid}, Int64, Float64, Int64, Ptr{Float64}, Ptr{Float64}, UInt64, Int64, Ptr{Cvoid}, Ref{CHistory},
                   Ptr{Int64}, Ptr{Cvoid}),
                  s.handle, C, T, cap, xinit, vinit, sd, chain_offset, C_NULL, Ref(_chist(b, status, cap)), ncols, C_NULL)
        end
        if rc == -6      # PDMPFLUX_ERR_CAPACITY
            cap *= 2
            continue
        end
        check(rc)
        s.state = status
        b.ncols .= ncols
        return b
    end
end
function sample_skeleton(s::CuPDMP, T::Float64, xinit::Vector{Float64}, vinit::Vector{Float64}; kw...)
    b = sample_skeleton(s, T, reshape(xinit, :, 1), reshape(vinit, :, 1); kw...)
    return deepcopy(b[1])     # detach from the batch storage
end

"""
    sample_skeleton_with_diagnostic(sampler::CuPDMP, T, xinit, vinit[, pot]; B=1000, seed) -> (history, rv)

Replaces src/sample.jl:75-236.  The reference accumulates the realised volatility of `U` online through
`sampler.flow`; the sum telescopes to the per-boundary form, so it is evaluated here from the finished skeleton on the
device with the sampler's own flow (`U` is the value plugin of the sampler's potential).
"""
function sample_skeleton_with_diagnostic(s::CuPDMP, T::Float64, xinit::Vector{Float64}, vinit::Vector{Float64};
                                         B::Int64=10^3, seed::Union{Int,Nothing}=nothing, verbose::Bool=true,
                                         init_capacity::Int=1024)
    B <= 0 && throw(ArgumentError("B must be positive. Current value: $B"))
    h = sample_skeleton(s, T, xinit, vinit; seed, verbose, init_capacity)
    T == 0.0 && return h, 0.0
    return h, RV_diagnostic(h, s; B=B, online=true)
end

"Replaces `PDMPFlux.sample_from_skeleton(sampler, dt::Float64, history)` (src/sample.jl:573-646): samples at j*dt."
function sample_from_skeleton(s::CuPDMP, dt::Float64, h::PDMPHistory; discard_vt::Bool=true)
    (dt > 0 && isfinite(dt)) || throw(ArgumentError("dt must be positive. Current value: $dt"))
    d, n_sk = size(h.X)
    M = floor(Int, h.t[end] / dt)
    out = Matrix{Float64}(undef, discard_vt ? d : 2d + 1, M)
    M == 0 && return out
    check(ccall((:pdmpflux_sample_from_skeleton_dt, LIB), Cint,
                (Cint, Cint, Int64, Int64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Float64, Int64, Int32,
                 Ptr{Float64}, Int32, Ptr{Cvoid}),
                s.flow_kind, d, n_sk, n_sk, 1, h.X, h.V, h.t, dt, M, discard_vt, out, 0, C_NULL))
    return out
end

"Replaces `PDMPFlux.sample_from_skeleton` (src/sample.jl:475-513; :516-561 for Sticky samplers: frozen coordinates rest)."
function sample_from_skeleton(s::CuPDMP, N::Int, h::PDMPHistory; discard_vt::Bool=true)
    N <= 0 && throw(ArgumentError("N must be positive. Current value: $N"))
    d, n_sk = size(h.X)
    out = Matrix{Float64}(undef, discard_vt ? d : 2d + 1, N)
    if s.sticky
        act = Matrix{UInt8}(h.is_active)
        check(ccall((:pdmpflux_sample_from_skeleton_sticky, LIB), Cint,
                    (Cint, Int64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{UInt8}, Int64, Int32, Ptr{Float64}, Int32, Ptr{Cvoid}),
                    d, n_sk, 1, h.X, h.V, h.t, act, N, discard_vt, out, 0, C_NULL))
    else
        check(ccall((:pdmpflux_sample_from_skeleton, LIB), Cint,
                    (Cint, Cint, Int64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Int32, Ptr{Float64}, Int32, Ptr{Cvoid}),
                    s.flow_kind, d, n_sk, 1, h.X, h.V, h.t, N, discard_vt, out, 0, C_NULL))
    end
    return out
end

"""
Replaces `PDMPFlux.RV_diagnostic(history, U; B)` (src/diagnostic.jl:37-75): `U` is the value plugin of the sampler's
device potential.  `online=true` interpolates with the sampler's flow, i.e. the value
`sample_skeleton_with_diagnostic` (src/sample.jl:75-236) accumulates.
"""
function RV_diagnostic(h::PDMPHistory, s::CuPDMP; B::Int64=0, online::Bool=false)
    B < 0 && throw(ArgumentError("B must be non-negative. Current value: $B"))
    n_sk = length(h.t)
    n_sk == 0 && return 0.0
    T = h.t[end]
    (!isfinite(T) || T < 0.0) && throw(ArgumentError("history.t[end] must be finite and non-negative. Current value: $T"))
    rv = Ref{Float64}(0.0)
    check(ccall((:pdmpflux_rv_diagnostic, LIB), Cint,
                (Ptr{Cvoid}, Cint, Int64, Int64, Int64, Ptr{Int64}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                 Ref{Float64}, Int32, Ptr{Cvoid}),
                s.pot, online ? s.flow_kind : Int32(0), n_sk, n_sk, 1, C_NULL, B, h.X, h.V, h.t, rv, 0, C_NULL))
    return rv[]
end

sample(s::CuPDMP, N_sk::Int, N::Int, xinit::Vector{Float64}, vinit::Vector{Float64}; seed=nothing, discard_vt=true) =
    sample_from_skeleton(s, N, sample_skeleton(s, N_sk, xinit, vinit; seed=seed); discard_vt=discard_vt)

# ---- the final reduction (no reference equivalent; SURVEY.md 8d/8e) ------------------------------------------------
"""
    moments_reduce(m1, m2, T) -> sums (4 × d)

`m1`, `m2`: d × C time integrals of x and x² per chain, `T`: their time spans (C).  Rows of the result: Σ_c m_c,
Σ_c m_c², Σ_c s_c, C with m_c = m1[:, c] / T[c], s_c = m2[:, c] / T[c] (`pdmpflux_moments_reduce`, one fused kernel).
"""
function moments_reduce(m1::Matrix{Float64}, m2::Matrix{Float64}, T::Vector{Float64})
    d, C = size(m1)
    sums = Matrix{Float64}(undef, d, 4)     # the C side writes [4][d] row-major = d × 4 column-major
    check(ccall((:pdmpflux_moments_reduce, LIB), Cint,
                (Cint, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int32, Ptr{Cvoid}),
                d, C, m1, m2, T, sums, 0, C_NULL))
    return permutedims(sums)
end

"The library-owned NCCL communicator of this rank.  Move `comm_unique_id()` (128 bytes, from rank 0) to the other ranks
with any transport (MPI.jl, Distributed, a file), call `pdmpflux_set_device` first."
mutable struct CuComm
    handle::Ptr{Cvoid}
end
function comm_unique_id()
    id = Vector{UInt8}(undef, 128)
    check(ccall((:pdmpflux_comm_unique_id, LIB), Cint, (Ptr{UInt8}, Csize_t), id, 128))
    return id
end
function CuComm(id::Vector{UInt8}, n_ranks::Int, rank::Int)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:pdmpflux_comm_create, LIB), Cint, (Ptr{UInt8}, Cint, Cint, Ref{Ptr{Cvoid}}), id, n_ranks, rank, h))
    c = CuComm(h[])
    finalizer(x -> ccall((:pdmpflux_comm_destroy, LIB), Cint, (Ptr{Cvoid},), x.handle), c)
    return c
end
"In-place sum over the ranks of `n` doubles at the DEVICE pointer `dptr` (`pdmpflux_moments_allreduce`, ncclAllReduce)."
moments_allreduce!(c::CuComm, dptr::Ptr{Float64}, n::Int; stream::Ptr{Cvoid}=C_NULL) =
    check(ccall((:pdmpflux_moments_allreduce, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Cvoid}), c.handle, dptr, n, stream))

end # module
