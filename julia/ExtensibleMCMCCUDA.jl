# ExtensibleMCMCCUDA.jl -- reference-side binding of libextmcmc_cuda.so (ABI version 2).
#
# UNEXECUTED IN THIS ENVIRONMENT: Julia is not installed in the build image nor on the GPU box.
# The file is the `ccall` binding a maintainer of ExtensibleMCMC.jl would add; it is written against
# include/extmcmc.h and checked STATICALLY against it by tests/test_julia_shim_static.py (every
# ccall symbol exists in the header with the same number of arguments; every struct has the header's
# field order and types; every accessor of src/workspaces.jl:91-136,294-385 has a method here).  The
# Python mirror in extensiblemcmc.jl_b200/ drives the very same symbols through ctypes and is what
# the GPU tests exercise.
#
# Seam used: MCMCBackend (src/types.jl:107-117); MCMC(updates; backend=CUDAMCMCBackend(...))
# (src/mcmc.jl:39-48) makes init! dispatch init_global_workspace(::CUDAMCMCBackend, ...)
# (src/workspaces.jl:38-47) and run! dispatch create_workspace(::CUDAMCMCBackend, ...)
# (src/workspaces.jl:280-287); __run! gets a method for the CUDA workspace (src/run.jl:64).
#
# Shape of the workspaces.  The reference's callbacks read FIELDS, not accessors
# (src/callbacks.jl:246-256: ws.sub_ws.state_history[i][j], local_wss[j].sub_ws.ll_history[i],
# local_wss[j].sub_ws°.ll_history[i], local_wss[j].acceptance_history[i]; :306-319: accepted(lws, M),
# ll / ll° / llr(lws, M), state(lws), state°(lws)).  The CUDA workspaces therefore carry the very
# same fields with the reference's element types for ONE chain, the `report_chain` (default 1), so
# SavingCallback and REPLCallback run unchanged; all chains live next to them in chain-fastest
# arrays (`all_*`), and SavingCallback gets a method that writes one file per chain
# (`<name>_chain<c>.csv`, the rule of the Python mirror, callbacks.py:62-67) when n_chains > 1.
module ExtensibleMCMCCUDA

using ExtensibleMCMC
using Distributions
using LinearAlgebra
const eMCMC = ExtensibleMCMC
const LIB = "libextmcmc_cuda"
const ABI_VERSION = Int32(2)

# ---- POD structs of include/extmcmc.h (same field order and types) ------------------------------
struct Adapt                      # extmcmc_adapt_t
    kind::Int32
    adapt_every_k_steps::Int32
    target_accpt_rate::Float64
    scale::Float64
    min::Float64
    max::Float64
    offset::Float64
end
struct Update                     # extmcmc_update_t
    kernel::Int32
    n_coords::Int32
    coords::Ptr{Int32}
    step::Ptr{Float64}
    pos::Ptr{UInt8}
    prior::Int32
    n_prior_params::Int32
    prior_params::Ptr{Float64}
    adapt::Adapt
end
struct Step                       # extmcmc_step_t
    mcmciter::Int64
    prev_mcmciter::Int64
    pidx::Int32
    prev_pidx::Int32
end
struct Config                     # extmcmc_config_t
    abi_version::Int32
    device::Int32
    n_chains::Int64
    chain_offset::Int64
    n_params::Int32
    n_updates::Int32
    law::Int32
    obs_dim::Int32
    seed::UInt64
    shard_mode::Int32
    rank::Int32
    world_size::Int32
    history_window::Int32
    roll_window::Int32
    use_graphs::Int32
    instrument::Int32
    sweep_variant::Int32
    stats_mode::Int32
    reserved_::NTuple{3,Int32}
end

# enumerations of the header
const LAW_GSN_IID_1D, LAW_GSN_MV, LAW_LOGISTIC, LAW_HIER_NORMAL, LAW_USER = Int32(1), Int32(2), Int32(3), Int32(4), Int32(5)
const KERNEL_RW_UNIFORM, KERNEL_RW_GAUSS, KERNEL_RW_GAUSS_MIX, KERNEL_MALA = Int32(1), Int32(2), Int32(3), Int32(4)
const ADAPT_NONE, ADAPT_UNIF_RW, ADAPT_HAARIO, ADAPT_MALA = Int32(0), Int32(1), Int32(2), Int32(3)
const PRIOR_PRODUCT, PRIOR_MVNORMAL = Int32(5), Int32(11)
const USER_GRAD_NONE, USER_GRAD_HAND, USER_GRAD_FORWARD = Int32(0), Int32(1), Int32(2)
const USER_THETA_TERM = Int32(1)

# ---- backend, build-defined laws and the MALA update (an empty stub in the reference) ------------
struct CUDAMCMCBackend <: eMCMC.MCMCBackend
    n_chains::Int
    device::Int
    seed::UInt64
    block_len::Int
    report_chain::Int
    runs_started::Base.RefValue{Int}
end
CUDAMCMCBackend(; n_chains=1, device=0, seed=0, block_len=128, report_chain=1) =
    CUDAMCMCBackend(n_chains, device, UInt64(seed), block_len, report_chain, Ref(0))

"Bayesian logistic regression, theta = beta[d] (EXTMCMC_LAW_LOGISTIC); data = (P = LogisticLaw(d), obs = rows of X, y = responses)"
struct LogisticLaw; d::Int; end
"Hierarchical normal model, theta = [theta_1..G, mu, tau] (EXTMCMC_LAW_HIER_NORMAL); data = (P = HierNormalLaw(G), obs = y, groups = 1-based group of every observation, sorted)"
struct HierNormalLaw; G::Int; end

"""
    DeviceLaw(source::String, n_params, obs_dim; gradient=false, chunk=nothing, theta_term=false)

A user-defined law on the device (EXTMCMC_LAW_USER): the counterparts of `set_parameters!(P, θ)` and
one term of `loglikelihood(P, obs)`, written in CUDA C++ (`struct Law`, `set_parameters`, `logpdf`, and
`logpdf_grad` with `gradient = true`; contract in include/extmcmc.h and INTEGRATION.md).  With
`gradient = :forward` the law is written generic over its scalar (`template <class real> struct Law`,
`set_parameters`, `logpdf`) and the gradient is derived in forward mode, as ForwardDiff would (at most
16 parameters; with `chunk = :auto` or a chunk width, up to 64 in chunks of that many tangents, as
ForwardDiff's chunk mode: `law.chunk` is the width the library compiled).  With `theta_term = true` the
source also defines `logpdf_theta` (and `logpdf_theta_grad` with `gradient = true`), a term of θ only
that is added once to the log-likelihood, such as the hierarchical p(θ_g | μ, τ) of a multilevel model.
Compiled for sm_100a when constructed (no device needed); a source that does not
compile throws with the compiler's log.  data = (P = DeviceLaw(...), obs = rows of obs_dim values);
responses are columns of the rows.
"""
struct DeviceLaw
    source::String
    n_params::Int
    obs_dim::Int
    with_grad::Int32                                     # USER_GRAD_NONE / _HAND / _FORWARD
    chunk_arg::Int32                                     # -1: unchunked; 0: the library's width; K
    chunk::Int                                           # forward mode: the width compiled (0 otherwise)
    flags::Int32                                         # USER_THETA_TERM or 0
    log::String
    function DeviceLaw(source::String, n_params, obs_dim; gradient=false, chunk=nothing, theta_term=false)
        with_grad = gradient === :forward ? USER_GRAD_FORWARD :
                    gradient === true ? USER_GRAD_HAND :
                    gradient === false ? USER_GRAD_NONE :
                    throw(ArgumentError("gradient must be false, true or :forward, not $(repr(gradient))"))
        chunk === nothing || with_grad == USER_GRAD_FORWARD ||
            throw(ArgumentError("chunk needs gradient = :forward"))
        chunk_arg = chunk === nothing ? Int32(-1) : chunk === :auto ? Int32(0) :
                    chunk isa Integer && !(chunk isa Bool) && chunk >= 1 ? Int32(chunk) :
                    throw(ArgumentError("chunk must be nothing, :auto or a positive width, not $(repr(chunk))"))
        theta_term isa Bool || throw(ArgumentError("theta_term must be true or false, not $(repr(theta_term))"))
        flags = theta_term ? USER_THETA_TERM : Int32(0)
        buf = zeros(UInt8, 1 << 16)
        used = Ref{Int32}(with_grad == USER_GRAD_FORWARD ? n_params : 0)
        rc = if theta_term                               # chunk: nothing in forward mode is the width n_params
            GC.@preserve buf ccall((:extmcmc_user_law_check_ex, LIB), Int32,
                                   (Cstring, Int32, Int32, Int32, Int32, Int32, Ptr{Int32}, Ptr{UInt8}, Int64),
                                   source, n_params, obs_dim, with_grad, ex_chunk(with_grad, chunk_arg, n_params),
                                   flags, used, pointer(buf), length(buf))
        elseif chunk_arg < 0
            GC.@preserve buf ccall((:extmcmc_user_law_check, LIB), Int32,
                                   (Cstring, Int32, Int32, Int32, Ptr{UInt8}, Int64),
                                   source, n_params, obs_dim, with_grad, pointer(buf), length(buf))
        else
            GC.@preserve buf ccall((:extmcmc_user_law_check_chunked, LIB), Int32,
                                   (Cstring, Int32, Int32, Int32, Ptr{Int32}, Ptr{UInt8}, Int64),
                                   source, n_params, obs_dim, chunk_arg, used, pointer(buf), length(buf))
        end
        log = unsafe_string(pointer(buf))
        rc == 0 || throw(ArgumentError("the device law does not compile (status $rc):\n" * log))
        new(source, n_params, obs_dim, with_grad, chunk_arg, used[], flags, log)
    end
end
# chunk of the _ex entry points
ex_chunk(with_grad, chunk_arg, n_params) =
    chunk_arg >= 0 ? chunk_arg : with_grad == USER_GRAD_FORWARD ? Int32(n_params) : Int32(0)

"MALAUpdate(tau, coords; prior, adpt): theta° = theta + tau^2/2 grad(ll + log prior)(theta) + tau z (src/updates.jl:216-218 is an empty stub)"
struct CUDAMALAUpdate{TP,TA} <: eMCMC.MCMCGradientBasedUpdate
    tau::Float64
    coords::Vector{Int}
    prior::TP
    adpt::TA
end
CUDAMALAUpdate(tau, coords; prior=eMCMC.ImproperPrior(), adpt=eMCMC.NoAdaptation()) =
    CUDAMALAUpdate(Float64(tau), collect(Int, coords), prior, adpt)
"Acceptance-rate targeting of the MALA step with the +-delta rule of AdaptationUnifRW (adaptation.jl:312-329); target 0.574"
struct AdaptationMALA
    adapt_every_k_steps::Int
    target_accpt_rate::Float64
    scale::Float64
    min::Float64
    max::Float64
    offset::Float64
end
AdaptationMALA(; adapt_every_k_steps=100, target_accpt_rate=0.574, scale=1.0, min=1e-12, max=1e7, offset=1e2) =
    AdaptationMALA(adapt_every_k_steps, target_accpt_rate, scale, min, max, offset)

last_error(h) = unsafe_string(ccall((:extmcmc_last_error, LIB), Cstring, (Ptr{Cvoid},), h))
check(h, rc) = rc == 0 ? nothing : error("libextmcmc_cuda (", rc, "): ", last_error(h))

# Philox key of the run-th run of a backend: the reference advances a global RNG from run to run,
# a counter RNG restarts -- run 0 keeps the user's seed, later runs get a SplitMix64 mix of it.
function run_seed(seed::UInt64, run::Int)
    run == 0 && return seed
    z = seed + UInt64(run) * 0x9E3779B97F4A7C15
    z = (z ⊻ (z >> 30)) * 0xBF58476D1CE4E5B9
    z = (z ⊻ (z >> 27)) * 0x94D049BB133111EB
    z ⊻ (z >> 31)
end

# ---- priors (src/priors.jl:18-88) -> (EXTMCMC_PRIOR_* kind, parameters) -------------------------
# params(dist) of Distributions.jl returns exactly the parameter order the header documents.
const PRIOR_KIND = Dict(Normal => 2, Gamma => 3, Uniform => 4, Exponential => 6, InverseGamma => 7,
                        Beta => 8, LogNormal => 9, Cauchy => 10)
prior_abi(::eMCMC.ImproperPrior) = (Int32(0), Float64[])
prior_abi(::eMCMC.ImproperPosPrior) = (Int32(1), Float64[])
function prior_abi(pr::eMCMC.StandardPrior)
    if pr.dist isa AbstractMvNormal                       # joint prior: {mu[n], L[n*n] column-major}
        L = cholesky(Symmetric(Matrix(cov(pr.dist)))).L
        return (PRIOR_MVNORMAL, vcat(Float64.(mean(pr.dist)), vec(Matrix{Float64}(L))))
    end
    for (T, k) in PRIOR_KIND
        pr.dist isa T && return (Int32(k), Float64[params(pr.dist)...])
    end
    error("StandardPrior($(typeof(pr.dist))) not implemented on the GPU path")
end
function prior_abi(pr::eMCMC.ProductPrior)                  # {K, then per factor: kind, dim, p0, p1}
    out = Float64[length(pr.dists)]
    for (dist, idx) in zip(pr.dists, pr.idx)
        k, pp = prior_abi(dist isa eMCMC.Prior ? dist : eMCMC.StandardPrior(dist))
        (k == PRIOR_PRODUCT || k == PRIOR_MVNORMAL) && error("ProductPrior factors must be iid families on the GPU path")
        append!(out, (Float64(k), Float64(length(idx)), get(pp, 1, 0.0), get(pp, 2, 0.0)))
    end
    (PRIOR_PRODUCT, out)
end
prior_abi(pr) = error("prior $(typeof(pr)) not implemented on the GPU path")

# ---- laws ------------------------------------------------------------------------------------------
law_abi(P::eMCMC.GsnTargetLaw) = length(P.P.μ) == 1 ? (LAW_GSN_IID_1D, 1) : (LAW_GSN_MV, length(P.P.μ))
law_abi(P::LogisticLaw) = (LAW_LOGISTIC, P.d)
law_abi(P::HierNormalLaw) = (LAW_HIER_NORMAL, 1)
law_abi(P::DeviceLaw) = (LAW_USER, P.obs_dim)
law_abi(P) = error("target law $(typeof(P)) is not implemented on the GPU path (write it as a DeviceLaw: set_parameters / logpdf in CUDA C++)")

# ---- transition kernels and adaptations -> (kernel id, step vector, pos flags) --------------------
kernel_abi(rw::eMCMC.UniformRandomWalk) = (KERNEL_RW_UNIFORM, Float64.(collect(rw.ϵ)), UInt8.(collect(rw.pos)))
kernel_abi(rw::eMCMC.GaussianRandomWalk) = (KERNEL_RW_GAUSS, vec(Matrix{Float64}(rw.Σ)), UInt8.(collect(rw.pos)))
kernel_abi(rw::eMCMC.GaussianRandomWalkMix) =
    (KERNEL_RW_GAUSS_MIX, vcat(vec(Matrix{Float64}(rw.gsn_A.Σ)), vec(Matrix{Float64}(rw.gsn_B.Σ)), Float64(rw.λ)),
     UInt8.(collect(rw.gsn_A.pos)))
kernel_abi(rw) = error("transition kernel $(typeof(rw)) not implemented on the GPU path")

const NO_ADAPT = Adapt(ADAPT_NONE, 100, 0.234, 1.0, 1e-12, 1e7, 1e2)
adapt_abi(::eMCMC.NoAdaptation) = NO_ADAPT
adapt_abi(a::eMCMC.AdaptationUnifRW) =
    Adapt(ADAPT_UNIF_RW, a.adapt_every_k_steps, a.target_accpt_rate, a.scale, a.min, a.max, a.offset)
adapt_abi(a::eMCMC.HaarioTypeAdaptation) = Adapt(ADAPT_HAARIO, a.adapt_every_k_steps, 0.0, a.scale, 0.0, 0.0, 0.0)
adapt_abi(a::AdaptationMALA) =
    Adapt(ADAPT_MALA, a.adapt_every_k_steps, a.target_accpt_rate, a.scale, a.min, a.max, a.offset)
adapt_abi(a) = error("adaptation $(typeof(a)) not implemented on the GPU path")

# HaarioTypeAdaptation's weight schedule f(lambda, N, iter) (adaptation.jl:385,422-426): the library
# calls it back on the host, on the calling thread, once per readjustment.
function lambda_trampoline(lam::Cdouble, N::Int64, iter::Int64, user::Ptr{Cvoid})::Cdouble
    f = unsafe_pointer_to_objref(user)::Base.RefValue{Any}
    Cdouble(f[](lam, N, iter))
end

# ---- host mirrors with the reference's field names and element types (one chain) -----------------
mutable struct CUDAGlobalSub{T}            # StandardGlobalSubworkspace, src/workspaces.jl:157-180
    state::Vector{T}
    state_history::Vector{Vector{Vector{T}}}             # [M][NU][p]
    state_proposal_history::Vector{Vector{Vector{T}}}
    data
end
mutable struct CUDALocalSub{T}             # StandardLocalSubworkspace, src/workspaces.jl:413-431
    state::Vector{T}
    ll::Vector{Float64}
    ll_history::Vector{Vector{Float64}}                  # [M][1]
end

mutable struct CUDAGlobalWorkspace{T} <: eMCMC.GlobalWorkspace{T}
    handle::Ptr{Cvoid}
    sub_ws::CUDAGlobalSub{T}               # the report chain, reference-shaped
    report_chain::Int
    n_chains::Int
    all_state::Matrix{T}                   # [C, p]          chain fastest, as the ABI fills it
    all_state_history::Array{T,4}          # [C, p, NU, M]
    all_state_proposal_history::Array{T,4}
    all_ll_history::Array{Float64,3}       # [C, NU, M]
    all_llprop_history::Array{Float64,3}
    all_acceptance_history::Array{UInt8,3}
    block_len::Int
    n_local::Int                           # local workspaces created so far (their pidx)
    keep::Vector{Any}                      # closures handed to the library (kept alive)
end

struct CUDALocalWorkspace{T} <: eMCMC.LocalWorkspace{T}
    gws::CUDAGlobalWorkspace{T}
    pidx::Int
    coords::Vector{Int}
    sub_ws::CUDALocalSub{T}
    sub_ws°::CUDALocalSub{T}
    acceptance_history::Vector{Bool}       # [M]
    updt_name::String
end

# ---- init_global_workspace (src/workspaces.jl:38-47, 215-234) ----------------------------------------
function eMCMC.init_global_workspace(b::CUDAMCMCBackend, M, updates::Vector{<:eMCMC.MCMCUpdate},
                                     data, θinit::Vector{T}; kwargs...) where T
    p, NU, C = length(θinit), length(updates), b.n_chains
    law, d = law_abi(data.P)
    seed = run_seed(b.seed, b.runs_started[]); b.runs_started[] += 1
    cfg = Config(ABI_VERSION, b.device, C, 0, p, NU, law, d, seed, 0, 0, 1, 2b.block_len, 100, 1, 0, 0,
                 p <= 16 ? 0 : 1, (Int32(0), Int32(0), Int32(0)))
    h = Ref{Ptr{Cvoid}}(C_NULL)
    rc = ccall((:extmcmc_create, LIB), Int32, (Ref{Config}, Ref{Ptr{Cvoid}}), cfg, h)
    rc == 0 || error("extmcmc_create: ", last_error(C_NULL))
    if data.P isa DeviceLaw                              # compiled once per process (cached by the check)
        if data.P.flags != 0
            check(h[], ccall((:extmcmc_set_user_law_ex, LIB), Int32, (Ptr{Cvoid}, Cstring, Int32, Int32, Int32),
                             h[], data.P.source, data.P.with_grad,
                             ex_chunk(data.P.with_grad, data.P.chunk_arg, data.P.n_params), data.P.flags))
        elseif data.P.chunk_arg < 0
            check(h[], ccall((:extmcmc_set_user_law, LIB), Int32, (Ptr{Cvoid}, Cstring, Int32),
                             h[], data.P.source, data.P.with_grad))
        else
            check(h[], ccall((:extmcmc_set_user_law_chunked, LIB), Int32, (Ptr{Cvoid}, Cstring, Int32),
                             h[], data.P.source, data.P.chunk_arg))
        end
    end
    keep = Any[]
    for (u, updt) in enumerate(updates)
        coords = Int32.(collect(updt.coords) .- 1)       # 0-based at the ABI
        if updt isa CUDAMALAUpdate
            kern, step, pos = KERNEL_MALA, Float64[updt.tau], UInt8[]
        else
            kern, step, pos = kernel_abi(updt.rw)
        end
        prior, pp = prior_abi(updt.prior)
        adapt = adapt_abi(updt.adpt)
        GC.@preserve coords step pos pp begin
            upd = Update(kern, length(coords), pointer(coords), pointer(step), isempty(pos) ? C_NULL : pointer(pos),
                         prior, length(pp), isempty(pp) ? C_NULL : pointer(pp), adapt)
            check(h[], ccall((:extmcmc_set_update, LIB), Int32, (Ptr{Cvoid}, Int32, Ref{Update}), h[], u - 1, upd))
        end
        if updt.adpt isa eMCMC.HaarioTypeAdaptation
            fref = Ref{Any}(updt.adpt.fλ); push!(keep, fref)
            cb = @cfunction(lambda_trampoline, Cdouble, (Cdouble, Int64, Int64, Ptr{Cvoid}))
            check(h[], ccall((:extmcmc_set_lambda_fn, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Cvoid}, Ptr{Cvoid}),
                             h[], u - 1, cb, pointer_from_objref(fref)))
        end
    end
    obs = Float64.(reduce(vcat, data.obs))               # row-major [N][d]
    y = data.P isa LogisticLaw ? Float64.(data.y) :
        data.P isa HierNormalLaw ? Float64.(data.groups .- 1) : Float64[]
    GC.@preserve obs y check(h[], ccall((:extmcmc_upload_obs, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int32, Ptr{Float64}), h[], obs, length(data.obs), d,
        isempty(y) ? C_NULL : pointer(y)))
    θ0 = repeat(reshape(θinit, 1, p), C, 1)              # [C, p] column-major == chain fastest
    GC.@preserve θ0 check(h[], ccall((:extmcmc_set_state, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}), h[], θ0))
    sub = CUDAGlobalSub{T}(copy(θinit), [[zeros(T, p) for _ in 1:NU] for _ in 1:M],
                           [[zeros(T, p) for _ in 1:NU] for _ in 1:M], data)
    ws = CUDAGlobalWorkspace{T}(h[], sub, b.report_chain, C, θ0, zeros(T, C, p, NU, M), zeros(T, C, p, NU, M),
                                zeros(C, NU, M), zeros(C, NU, M), zeros(UInt8, C, NU, M), b.block_len, 0, keep)
    finalizer(w -> ccall((:extmcmc_destroy, LIB), Int32, (Ptr{Cvoid},), w.handle), ws)
    ws
end

# create_workspaces (src/workspaces.jl:362-371) calls this once per update, in schedule order
function eMCMC.create_workspace(::CUDAMCMCBackend, updt, gws::CUDAGlobalWorkspace{T}, M) where T
    gws.n_local += 1
    coords = collect(Int, updt.coords)
    mk() = CUDALocalSub{T}(gws.sub_ws.state[coords], [-Inf], [zeros(Float64, 1) for _ in 1:M])   # workspaces.jl:425-426
    CUDALocalWorkspace{T}(gws, gws.n_local, coords, mk(), mk(), fill(false, M),
                          string(eMCMC.remove_curly(typeof(updt))))
end

# ---- accessors of src/workspaces.jl:91-136 (global) and :294-385 (local) ---------------------------
eMCMC.num_mcmc_steps(ws::CUDAGlobalWorkspace) = length(ws.sub_ws.state_history)
eMCMC.num_updt(ws::CUDAGlobalWorkspace) = length(first(ws.sub_ws.state_history))
eMCMC.state(ws::CUDAGlobalWorkspace) = ws.sub_ws.state
eMCMC.state(ws::CUDAGlobalWorkspace, step) = ws.sub_ws.state_history[step.mcmciter][step.pidx]
eMCMC.state°(ws::CUDAGlobalWorkspace, step) = ws.sub_ws.state_proposal_history[step.mcmciter][step.pidx]
eMCMC.state(ws::CUDAGlobalWorkspace, updt::eMCMC.MCMCUpdate) = ws.sub_ws.state[collect(updt.coords)]
eMCMC.accepted(ws::CUDALocalWorkspace, i::Int) = ws.acceptance_history[i]
eMCMC.set_accepted!(ws::CUDALocalWorkspace, i::Int, v) = (ws.acceptance_history[i] = v)
eMCMC.ll(ws::CUDALocalWorkspace) = ws.sub_ws.ll
eMCMC.ll°(ws::CUDALocalWorkspace) = ws.sub_ws°.ll
eMCMC.ll(ws::CUDALocalWorkspace, i::Int) = ws.sub_ws.ll_history[i]
eMCMC.ll°(ws::CUDALocalWorkspace, i::Int) = ws.sub_ws°.ll_history[i]   # (the reference ignores i, workspaces.jl:337)
eMCMC.state(ws::CUDALocalWorkspace) = ws.sub_ws.state
eMCMC.state°(ws::CUDALocalWorkspace) = ws.sub_ws°.state
eMCMC.llr(ws::CUDALocalWorkspace, i::Int) = sum(eMCMC.ll°(ws, i) .- eMCMC.ll(ws, i))
eMCMC.name_of_update(ws::CUDALocalWorkspace) = ws.updt_name

# every chain, chain-fastest arrays (no counterpart in the reference, which has one chain)
all_states(ws::CUDAGlobalWorkspace) = ws.all_state
all_state_history(ws::CUDAGlobalWorkspace) = ws.all_state_history
all_acceptance_history(ws::CUDAGlobalWorkspace) = ws.all_acceptance_history

# estim_mean / estim_cov (src/workspaces.jl:121-136): GenericChainStats of the report chain;
# chain_stats returns all chains: mean [C, p], cov [C, p, p] (entry (a, b) at a + b p)
function chain_stats(ws::CUDAGlobalWorkspace)
    C, p = size(ws.all_state); NU = eMCMC.num_updt(ws)
    m = zeros(C, p); cv = zeros(C, p * p); ra = zeros(C, NU); na = zeros(Int64, C, NU); np = zeros(Int64, C, NU)
    GC.@preserve m cv ra na np check(ws.handle, ccall((:extmcmc_get_stats, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Int64}), ws.handle, m, cv, ra, na, np))
    (mean = m, cov = reshape(cv, C, p, p), rolling_ar = ra, n_accept = na, n_prop = np)
end
eMCMC.estim_mean(ws::CUDAGlobalWorkspace) = chain_stats(ws).mean[ws.report_chain, :]
eMCMC.estim_cov(ws::CUDAGlobalWorkspace) = chain_stats(ws).cov[ws.report_chain, :, :]

"Current per-chain step-size state of update u (1-based): eps [C, p_u], Sigma_B [C, p_u^2] or tau [C, 1]"
function step_sizes(ws::CUDAGlobalWorkspace, u::Int, rows::Int)
    out = zeros(ws.n_chains, rows)
    GC.@preserve out check(ws.handle, ccall((:extmcmc_get_eps, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}), ws.handle, u - 1, out))
    out
end

# ---- __run! (src/run.jl:64-83): walk the schedule on the host, ship blocks; callbacks define the
#      sync points.  The copy-back of block k overlaps the execution of block k+1 (the ring holds
#      2 x block_len rows).
function eMCMC.__run!(gws::CUDAGlobalWorkspace, local_wss, updates, schedule, callbacks)
    block = Step[]; seq = Ref(0); pending = Ref{Any}(nothing)
    finish_fetch!() = begin
        pending[] === nothing && return
        store_rows!(gws, local_wss, pending[]); pending[] = nothing
    end
    flush!() = begin
        isempty(block) && return
        check(gws.handle, ccall((:extmcmc_run_block, LIB), Int32, (Ptr{Cvoid}, Ptr{Step}, Int32),
                                gws.handle, block, length(block)))
        finish_fetch!()                                   # rows of the previous block
        check(gws.handle, ccall((:extmcmc_history_fetch_begin, LIB), Int32, (Ptr{Cvoid}, Int64, Int64),
                                gws.handle, seq[], seq[] + length(block)))
        pending[] = copy(block); seq[] += length(block); empty!(block)
    end
    drain!() = begin                                      # host-visible point: everything mirrored on the host
        finish_fetch!()
        check(gws.handle, ccall((:extmcmc_sync, LIB), Int32, (Ptr{Cvoid},), gws.handle))
    end
    for step in schedule
        pre = [cb for cb in callbacks if eMCMC.check_if_execute(cb, step, eMCMC.__PRESTEP)]
        isempty(pre) || (flush!(); drain!(); foreach(cb -> eMCMC.execute!(cb, gws, local_wss, step, eMCMC.__PRESTEP), pre))
        push!(block, Step(step.mcmciter, something(step.prev_mcmciter, 0), step.pidx - 1,
                          step.prev_pidx === nothing ? -1 : step.prev_pidx - 1))
        post = [cb for cb in callbacks if eMCMC.check_if_execute(cb, step, eMCMC.__POSTSTEP)]
        if !isempty(post)
            flush!(); drain!(); foreach(cb -> eMCMC.execute!(cb, gws, local_wss, step, eMCMC.__POSTSTEP), post)
        elseif length(block) >= gws.block_len
            flush!()
        end
    end
    flush!(); drain!()
    refresh_state!(gws)
end

function refresh_state!(gws::CUDAGlobalWorkspace)
    GC.@preserve gws check(gws.handle, ccall((:extmcmc_get_state, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}),
                                             gws.handle, gws.all_state, C_NULL))
    gws.sub_ws.state .= gws.all_state[gws.report_chain, :]
end

# rows of a finished block: pinned staging area -> all-chain arrays -> the reference-shaped mirrors
function store_rows!(gws, local_wss, block)
    n = length(block); C, p = size(gws.all_state)
    th = zeros(C, p, n); thp = zeros(C, p, n); l = zeros(C, n); lp = zeros(C, n); a = zeros(UInt8, C, n)
    GC.@preserve th thp l lp a check(gws.handle, ccall((:extmcmc_history_fetch_end, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{UInt8}), gws.handle, th, thp, l, lp, a))
    r = gws.report_chain
    for (k, s) in enumerate(block)
        i, j = s.mcmciter, s.pidx + 1
        gws.all_state_history[:, :, j, i] .= th[:, :, k]; gws.all_state_proposal_history[:, :, j, i] .= thp[:, :, k]
        gws.all_ll_history[:, j, i] .= l[:, k]; gws.all_llprop_history[:, j, i] .= lp[:, k]
        gws.all_acceptance_history[:, j, i] .= a[:, k]
        gws.sub_ws.state_history[i][j] .= th[r, :, k]
        gws.sub_ws.state_proposal_history[i][j] .= thp[r, :, k]
        gws.sub_ws.state .= th[r, :, k]
        lw = local_wss[j]
        lw.sub_ws.ll_history[i][1] = l[r, k]; lw.sub_ws°.ll_history[i][1] = lp[r, k]
        lw.sub_ws.ll[1] = l[r, k]; lw.sub_ws°.ll[1] = lp[r, k]
        lw.sub_ws.state .= th[r, lw.coords, k]; lw.sub_ws°.state .= thp[r, lw.coords, k]
        lw.acceptance_history[i] = a[r, k] != 0
    end
end

# ---- SavingCallback with several chains: one file per chain, each in the reference's row format
#      (src/callbacks.jl:246-256); with one chain the reference's own method applies unchanged.
chain_file(name, c) = (stem = splitext(name); string(stem[1], "_chain", c, stem[2]))
function eMCMC.execute!(sc::eMCMC.SavingCallback, ws::CUDAGlobalWorkspace, local_wss, step, flag::Any)
    ws.n_chains == 1 && return invoke(eMCMC.execute!, Tuple{eMCMC.SavingCallback,eMCMC.GlobalWorkspace,Any,Any,Any},
                                      sc, ws, local_wss, step, flag)
    iter_start = eMCMC.find_starting_idx(sc, step)
    for c in 1:ws.n_chains
        open(chain_file(sc.filename, c - 1), "a") do f
            for i in iter_start:(step.mcmciter - 1), j in 1:eMCMC.num_updt(ws)
                θ = join(["$θₖ, " for θₖ in ws.all_state_history[c, :, j, i]])
                θ° = join(["$θₖ, " for θₖ in ws.all_state_proposal_history[c, :, j, i]])
                write(f, string("$i, $j, ", "!, ", θ, "!, ", θ°, "!, ", "$(ws.all_ll_history[c, j, i]), ", "!, ", "0.0, ",
                                "!,", "$(ws.all_acceptance_history[c, j, i] != 0), ", "\n"))
            end
        end
    end
end

end # module
