# rollout_bayesian_optimization.jl -- drop-in entry file for the reference's drivers and notebooks
# (experiments/*.jl do `include("../rollout_bayesian_optimization.jl")`, nonmyopic_bayesopt.jl:98).
#
# What it does (SURVEY.md section 8b):
#   1. includes the user's OWN checkout of the reference for everything off the hot path
#      (ENV["ROLLOUT_BO_REFERENCE_DIR"]; same order as the reference's entry file l.15-30) -- no reference source is
#      copied into this repository;
#   2. defines the two names the shipped nonmyopic driver needs but HEAD never defines (RBFsurrogate, HORIZON);
#   3. RE-DEFINES the hot-path methods with identical signatures as marshalling + `ccall` into librbo.so:
#        simulate_trajectory_mc(T, tp; ...)            rollout.jl:279-340
#        simulate_trajectory_mc(T, tp, observable; ...) rollout.jl:342-404 (same body at HEAD, Q17)
#        multistart_base_solve!(::Surrogate, xfinal; ...) rbf_optim.jl:103-134 (what both live drivers time)
#      Julia's last-definition-wins makes this a drop-in: the drivers run unchanged;
#   4. defines what utils.jl:235-265 calls but HEAD never defines -- simulate_adjoint_trajectory(surrogate, tp; ...) -- and re-defines
#      stochastic_solve so that the surrogate, normals and starts stay RESIDENT on the device across the ascent iterations;
#      stochastic_solve_batch runs the whole ascent from a batch of restarts on the device in one call.
#
# Resident inputs: the handle remembers a fingerprint of the surrogate / normals / starts it holds and re-uploads only what changed
# (a BO iteration changes the surrogate; an ascent iteration changes only x0). rbo_condition! appends an observation on the device.
#
# rand(dim) of solve_dual_y (rollout.jl:133, SURVEY.md hard part 2): reproduced EXACTLY by a two-phase call -- values and best
# indices first, then rand(d) is drawn on the host only for the case-3 samples, j = t, t-1, .., 1, in sample order (the reference's
# own consumption of the global RNG), then the device-resident x-path is replayed bitwise with the gradient (RBO_FLAG_REPLAY_TAPE).
#
# NOT RUN in the build environment (Julia is not installed there); the Python mirror
# (rollout-bayesian-optimization_b200/api.py) drives the same C entry points in the tests.
#
# Environment:
#   ROLLOUT_BO_REFERENCE_DIR  directory of the reference checkout (default: parent of this file's directory)
#   LIBRBO                    path of librbo.so (default: ../csrc/librbo.so next to this file)
#   RBO_DEVICE                CUDA device index (default 0)

const _RBO_REF = get(ENV, "ROLLOUT_BO_REFERENCE_DIR", normpath(joinpath(@__DIR__, "..", "..", "..")))
const librbo = get(ENV, "LIBRBO", normpath(joinpath(@__DIR__, "..", "csrc", "librbo.so")))

using Plots, Sobol, Distributions, LinearAlgebra, Optim, ForwardDiff, Distributed, Statistics, SharedArrays, Roots,
      FastGaussQuadrature, IterTools, Random

for f in ("constants.jl", "testfns.jl", "lazy_struct.jl", "low_discrepancy.jl", "optim.jl", "radial_basis_functions.jl",
          "decision_rules.jl", "radial_basis_surrogates.jl", "cost_functions.jl", "rbf_optim.jl", "observables.jl",
          "trajectory.jl", "rollout.jl", "optimizers.jl", "utils.jl")
    include(joinpath(_RBO_REF, f))
end

# ---- fix-ups for experiments/nonmyopic_bayesopt.jl (SURVEY.md 0.4) -----------------------------------------------
if !@isdefined(RBFsurrogate)
    const RBFsurrogate = Surrogate                     # l.101 `random_solver(s::RBFsurrogate, ...)`
end
if @isdefined(cli_args) && !@isdefined(HORIZON)
    HORIZON = cli_args["horizon"]                      # l.198, 236, 237
end

# ---- C ABI (include/rbo.h) ----------------------------------------------------------------------------------------
struct RboSolverOpts
    maxit::Int32; maxtry::Int32
    gtol::Float64; xtol::Float64; pred_tol::Float64; eta::Float64; delta0_box::Float64; delta0_ell::Float64; stol::Float64
end
mutable struct RboSummary
    mean::Float64; std::Float64; n_traj::Int32; n_failed::Int32
    kernel_ms::Float64; flops::Float64; flops_executed::Float64; n_evals::Int64; gpu_launches::Int32; tail_ms::Float64
    RboSummary() = new(0, 0, 0, 0, 0, 0, 0, 0, 0, 0)
end

const _RBO_KERNEL_ID = IdDict{Any, Cint}(Matern12 => 0, Matern32 => 1, Matern52 => 2, SquaredExponential => 3, Periodic => 4)
const _RBO_RULE_ID = Dict("EI" => Cint(0), "POI" => Cint(1), "LCB" => Cint(2))
const _RBO_STATUS = Dict(1 => "PosDefException: update_cholesky! (rbs.jl:412)", 2 => "DomainError: sqrt (rbs.jl:528)",
                         3 => "PosDefException: joint covariance (rbs.jl:537)",
                         4 => "ArgumentError: reducing over an empty collection (rbf_optim.jl:97)",
                         5 => "SingularException (rollout.jl:188)")

mutable struct RboHandle
    ptr::Ptr{Cvoid}
    function RboHandle(device::Integer = parse(Int, get(ENV, "RBO_DEVICE", "0")))
        ref = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:rbo_create, librbo), Cint, (Ref{Ptr{Cvoid}}, Cint), ref, device)
        rc == 0 || error("rbo_create failed ($rc): " * unsafe_string(ccall((:rbo_last_error, librbo), Cstring, (Ptr{Cvoid},), C_NULL)))
        h = new(ref[])
        finalizer(x -> ccall((:rbo_destroy, librbo), Cint, (Ptr{Cvoid},), x.ptr), h)
        return h
    end
end
_rbo_check(h::RboHandle, rc) = rc == 0 || error("librbo error $rc: " * unsafe_string(ccall((:rbo_last_error, librbo), Cstring, (Ptr{Cvoid},), h.ptr)))

const _RBO_HANDLE = Ref{Union{Nothing, RboHandle}}(nothing)
_rbo_handle() = (_RBO_HANDLE[] === nothing && (_RBO_HANDLE[] = RboHandle()); _RBO_HANDLE[])

"""EI's sigma_tol is captured in a closure (decision_rules.jl:84) and cannot be read back from the struct; the
reference never changes its default."""
_rbo_sigma_tol(g) = 1e-8

# fs.X (d x (cap+h+1)), fs.L.data ((cap+h+1)^2, column-major lower), fs.y, fs.cs[1], fs.sigma_n2, fs.psi, fs.g  (rbs.jl:320-381)
function _rbo_set_surrogate!(h::RboHandle, X::Matrix{Float64}, Ldata::Matrix{Float64}, y::Vector{Float64}, c::Vector{Float64},
                             N::Int, ψ, g, σn2::Float64)
    θk = Vector{Float64}(ψ.θ)
    _rbo_check(h, ccall((:rbo_set_surrogate, librbo), Cint,
        (Ptr{Cvoid}, Cint, Cint, Ptr{Float64}, Cint, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Float64}, Float64, Cint, Ptr{Float64}, Cint, Cint, Float64),
        h.ptr, size(X, 1), N, X, size(X, 1), Ldata, size(Ldata, 1), y, c, σn2, _RBO_KERNEL_ID[ψ.constructor], θk, length(θk),
        _RBO_RULE_ID[g.name], _rbo_sigma_tol(g)))
end

# ---- resident inputs ----------------------------------------------------------------------------------------------------
const _RBO_RESIDENT = Dict{Symbol, UInt}()   # fingerprints of what the handle currently holds
_rbo_fp(xs...) = hash(xs)

"""Uploads the base part of the fantasy surrogate unless the handle already holds it (same data, kernel, rule)."""
function _rbo_sync_surrogate!(h::RboHandle, fs)
    N = get_known_observations(fs)
    fp = _rbo_fp(N, size(fs.X, 1), view(fs.X, :, 1:N), view(fs.y, 1:N), Vector{Float64}(fs.ψ.θ), fs.ψ.constructor, fs.g.name, fs.σn2)
    get(_RBO_RESIDENT, :surrogate, UInt(0)) == fp && return
    _rbo_set_surrogate!(h, fs.X, fs.L.data, fs.y, fs.cs[1], N, fs.ψ, fs.g, fs.σn2)
    _RBO_RESIDENT[:surrogate] = fp
    delete!(_RBO_RESIDENT, :normals); delete!(_RBO_RESIDENT, :starts)     # conservative: a new input dimension invalidates them
end
function _rbo_sync_normals!(h::RboHandle, rn::Array{Float64, 3})
    fp = _rbo_fp(size(rn), rn[1], rn[end], sum(rn))   # content-based: a deepcopy of the TrajectoryParameters keeps the normals resident
    get(_RBO_RESIDENT, :normals, UInt(0)) == fp && return
    M = size(rn, 1)
    _rbo_check(h, ccall((:rbo_set_normals, librbo), Cint, (Ptr{Cvoid}, Ptr{Float64}, Cint, Cint, Cint, Cint), h.ptr, rn, M, size(rn, 3), 0, M))
    _RBO_RESIDENT[:normals] = fp
end
function _rbo_sync_starts!(h::RboHandle, starts::Matrix{Float64})
    fp = _rbo_fp(size(starts), sum(starts), starts[1], starts[end])
    get(_RBO_RESIDENT, :starts, UInt(0)) == fp && return
    _rbo_check(h, ccall((:rbo_set_starts, librbo), Cint, (Ptr{Cvoid}, Ptr{Float64}, Cint), h.ptr, starts, size(starts, 2)))
    _RBO_RESIDENT[:starts] = fp
end

"""condition!(s::Surrogate, x, y) (rbs.jl:214-222) mirrored on the device-resident surrogate: call it right after the host-side
`condition!` of a BO iteration and the next simulate call uploads nothing (the fingerprint is refreshed by the caller's next sync)."""
function rbo_condition!(x::Vector{Float64}, y::Float64)
    h = _rbo_handle()
    _rbo_check(h, ccall((:rbo_condition, librbo), Cint, (Ptr{Cvoid}, Ptr{Float64}, Float64), h.ptr, x, y))
    delete!(_RBO_RESIDENT, :surrogate)   # the next sync compares against the host copy again (cheap: a hash of X, y)
    return nothing
end

function _rbo_rollout!(h, tp, θ, fmini, mode::Int, flags::Int, dual, resolutions, gx, gθ, best_index, status, summary)
    _rbo_check(h, ccall((:rbo_rollout, librbo), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Cint, Cint, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ref{RboSummary}),
        h.ptr, tp.x0, θ, length(θ), tp.spatial_lbs, tp.spatial_ubs, tp.horizon, fmini, mode, flags,
        dual === nothing ? C_NULL : dual, C_NULL, resolutions, gx === nothing ? C_NULL : gx, gθ === nothing ? C_NULL : gθ,
        best_index === nothing ? C_NULL : best_index, C_NULL, status, summary))
end

function _rbo_first_error(status)
    bad = findfirst(!=(0), status)
    isnothing(bad) || error("sample $bad: " * get(_RBO_STATUS, Int(status[bad]), "error"))   # serial semantics: first failing sample
end

function _rbo_simulate(T::Trajectory, tp::TrajectoryParameters, inner_solve_xstarts::Matrix{Float64}, resolutions::Vector{Float64},
                       spatial_gradients_container, hyperparameter_gradients_container; flags::Int = 0)
    h = _rbo_handle()
    fs = get_fantasy_surrogate(T)
    set_start!(T, get_starting_point(tp))                                   # rollout.jl:287
    _rbo_sync_surrogate!(h, fs)
    _rbo_sync_normals!(h, tp.rnstream_sequence)                             # M x (d+1) x (h+1), column-major (trajectory.jl:47)
    _rbo_sync_starts!(h, inner_solve_xstarts)
    M, d, hor = tp.mc_iters, length(tp.x0), tp.horizon
    want_grad = !isnothing(spatial_gradients_container) && !isnothing(hyperparameter_gradients_container)  # rollout.jl:319
    fmini = minimum(get_observations(get_base_surrogate(T)))               # rollout.jl:109,234 (zero-padded vector, Q2)
    status = zeros(Int32, M)
    summary = RboSummary()
    θ = Vector{Float64}(tp.θ)
    if want_grad && hor > 0
        # phase 1: values and best indices (no gradient work)
        best_index = zeros(Int32, M)
        _rbo_rollout!(h, tp, θ, fmini, 0, flags, nothing, resolutions, nothing, nothing, best_index, status, summary)
        _rbo_first_error(status)
        # the reference's consumption of the global RNG (rollout.jl:259-262 -> :133): case-3 samples only, j = t:-1:1, sample order
        dual = zeros(d, hor, M)
        for m in 1:M
            t = Int(best_index[m])
            if resolutions[m] > 0.0 && t >= 1
                for j in t:-1:1
                    dual[:, j, m] = rand(d)
                end
            end
        end
        # phase 2: bitwise replay of the device-resident x-path with the adjoint (RBO_FLAG_REPLAY_TAPE = 8)
        _rbo_rollout!(h, tp, θ, fmini, 1, flags | 8, dual, resolutions, spatial_gradients_container, hyperparameter_gradients_container,
                      nothing, status, summary)
    else
        _rbo_rollout!(h, tp, θ, fmini, want_grad ? 1 : 0, flags, nothing, resolutions,
                      want_grad ? spatial_gradients_container : nothing, want_grad ? hyperparameter_gradients_container : nothing,
                      nothing, status, summary)
    end
    _rbo_first_error(status)
    μxθ = Distributions.mean(resolutions)                                  # rollout.jl:328-337
    σ_μxθ = Distributions.std(resolutions, mean = μxθ)
    if !want_grad
        return ExpectedTrajectoryOutput(μxθ = μxθ, σ_μxθ = σ_μxθ)
    end
    ∇μx = vec(Distributions.mean(spatial_gradients_container, dims = 2))
    σ_∇μx = vec(Distributions.std(spatial_gradients_container, dims = 2, mean = ∇μx))
    ∇μθ = vec(Distributions.mean(hyperparameter_gradients_container, dims = 2))
    σ_∇μθ = vec(Distributions.std(hyperparameter_gradients_container, dims = 2, mean = ∇μθ))
    return ExpectedTrajectoryOutput(μxθ = μxθ, σ_μxθ = σ_μxθ, ∇μx = ∇μx, σ_∇μx = σ_∇μx, ∇μθ = ∇μθ, σ_∇μθ = σ_∇μθ)
end

# ---- re-definitions (identical signatures; last definition wins) --------------------------------------------------
function simulate_trajectory_mc(T::Trajectory, tp::TrajectoryParameters;
        inner_solve_xstarts::Matrix{T1}, resolutions::Vector{T1},
        spatial_gradients_container::Union{Nothing, Matrix{T1}} = nothing,
        hyperparameter_gradients_container::Union{Nothing, Matrix{T1}} = nothing) where T1 <: Real
    return _rbo_simulate(T, tp, inner_solve_xstarts, resolutions, spatial_gradients_container, hyperparameter_gradients_container)
end

function simulate_trajectory_mc(T::Trajectory, tp::TrajectoryParameters, observable::AbstractObservable;
        inner_solve_xstarts::Matrix{T1}, resolutions::Vector{T1},
        spatial_gradients_container::Union{Nothing, Matrix{T1}} = nothing,
        hyperparameter_gradients_container::Union{Nothing, Matrix{T1}} = nothing) where T1 <: Real
    # rollout.jl:342-404 ignores `observable` as well: it builds a fresh StochasticObservable per sample (l.359-364)
    return _rbo_simulate(T, tp, inner_solve_xstarts, resolutions, spatial_gradients_container, hyperparameter_gradients_container)
end

# simulate_trajectory_ghq (rollout.jl:409-467): one trajectory per entry of `indices`, GaussHermiteObservable draws
function simulate_trajectory_ghq(T::Trajectory, tp::TrajectoryParameters;
        inner_solve_xstarts::Matrix{T1}, resolutions::Vector{T1}, nodes::Vector{T1}, weights::Vector{T1}, indices,
        spatial_gradients_container::Union{Nothing, Matrix{T1}} = nothing,
        hyperparameter_gradients_container::Union{Nothing, Matrix{T1}} = nothing) where T1 <: Real
    h = _rbo_handle()
    empty!(_RBO_RESIDENT)                                                   # this call replaces the resident inputs directly
    fs = get_fantasy_surrogate(T)
    set_start!(T, get_starting_point(tp))                                   # rollout.jl:422
    N = get_known_observations(fs)
    _rbo_set_surrogate!(h, fs.X, fs.L.data, fs.y, fs.cs[1], N, fs.ψ, fs.g, fs.σn2)
    depth, M, d, hor = length(first(indices)), length(indices), length(tp.x0), tp.horizon
    depth >= hor + 1 || error("AssertionError: Maximum invocations have been used")          # observables.jl:55
    nd = Matrix{Float64}(undef, depth, M); wt = similar(nd)
    for (m, idx) in enumerate(vec(indices))                                 # rollout.jl:431-432
        nd[:, m] = nodes[idx]; wt[:, m] = weights[idx]
    end
    _rbo_check(h, ccall((:rbo_set_quadrature, librbo), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Cint, Cint), h.ptr, nd, wt, depth, M))
    _rbo_check(h, ccall((:rbo_set_starts, librbo), Cint, (Ptr{Cvoid}, Ptr{Float64}, Cint), h.ptr, inner_solve_xstarts, size(inner_solve_xstarts, 2)))
    want_grad = !isnothing(spatial_gradients_container) && !isnothing(hyperparameter_gradients_container)
    dual = want_grad ? rand(d, max(hor, 1), M) : zeros(0)
    fmini = minimum(get_observations(get_base_surrogate(T)))
    vals = zeros(M); gx = zeros(d, M); gθ = zeros(length(tp.θ), M)
    status = zeros(Int32, M); summary = RboSummary(); θ = Vector{Float64}(tp.θ)
    _rbo_check(h, ccall((:rbo_rollout, librbo), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Cint, Cint, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ref{RboSummary}),
        h.ptr, tp.x0, θ, length(θ), tp.spatial_lbs, tp.spatial_ubs, hor, fmini, want_grad ? 1 : 0, 2 #= RBO_FLAG_GAUSS_HERMITE =#,
        want_grad ? dual : C_NULL, C_NULL, vals, want_grad ? gx : C_NULL, want_grad ? gθ : C_NULL, C_NULL, C_NULL, status, summary))
    bad = findfirst(!=(0), status)
    isnothing(bad) || error("sample $bad: " * get(_RBO_STATUS, Int(status[bad]), "error"))
    resolutions[1:M] = vals                                                 # rollout.jl:444
    μxθ = Distributions.mean(resolutions)                                  # rollout.jl:455-456: the whole vector
    σ_μxθ = Distributions.std(resolutions, mean = μxθ)
    want_grad || return ExpectedTrajectoryOutput(μxθ = μxθ, σ_μxθ = σ_μxθ)
    spatial_gradients_container[:, 1:M] = gx
    hyperparameter_gradients_container[:, 1:M] = gθ
    ∇μx = vec(Distributions.mean(spatial_gradients_container, dims = 2))
    σ_∇μx = vec(Distributions.std(spatial_gradients_container, dims = 2, mean = ∇μx))
    ∇μθ = vec(Distributions.mean(hyperparameter_gradients_container, dims = 2))
    σ_∇μθ = vec(Distributions.std(hyperparameter_gradients_container, dims = 2, mean = ∇μθ))
    return ExpectedTrajectoryOutput(μxθ = μxθ, σ_μxθ = σ_μxθ, ∇μx = ∇μx, σ_∇μx = σ_∇μx, ∇μθ = ∇μθ, σ_∇μθ = σ_∇μθ)
end

# Not in the reference: the estimator at every column of x0s (d x B) in ONE launch -- what a serial loop over
# simulate_trajectory_mc with set_starting_point!(tp, x0) computes (same normals for every starting point). Returns a vector of
# ExpectedTrajectoryOutput. Used by drivers that restart the stochastic ascent from a batch of x0 (utils.jl:235-265).
function simulate_trajectory_mc_batch(T::Trajectory, tp::TrajectoryParameters, x0s::Matrix{Float64}; inner_solve_xstarts::Matrix{Float64})
    h = _rbo_handle()
    empty!(_RBO_RESIDENT)
    fs = get_fantasy_surrogate(T)
    N = get_known_observations(fs)
    _rbo_set_surrogate!(h, fs.X, fs.L.data, fs.y, fs.cs[1], N, fs.ψ, fs.g, fs.σn2)
    rn = tp.rnstream_sequence
    M, d, hor, B = tp.mc_iters, length(tp.x0), tp.horizon, size(x0s, 2)
    _rbo_check(h, ccall((:rbo_set_normals, librbo), Cint, (Ptr{Cvoid}, Ptr{Float64}, Cint, Cint, Cint, Cint), h.ptr, rn, M, size(rn, 3), 0, M))
    _rbo_check(h, ccall((:rbo_set_starts, librbo), Cint, (Ptr{Cvoid}, Ptr{Float64}, Cint), h.ptr, inner_solve_xstarts, size(inner_solve_xstarts, 2)))
    θ = Vector{Float64}(tp.θ)
    vals = zeros(M, B); gx = zeros(d, M, B); gθ = zeros(length(θ), M, B); status = zeros(Int32, M, B)
    dual = rand(d, max(hor, 1), M)
    summary = RboSummary()
    _rbo_check(h, ccall((:rbo_rollout_batch, librbo), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Cint, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Cint, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ref{RboSummary}),
        h.ptr, x0s, B, θ, length(θ), tp.spatial_lbs, tp.spatial_ubs, hor, minimum(get_observations(get_base_surrogate(T))), 1, dual,
        vals, gx, gθ, status, summary))
    bad = findfirst(!=(0), status)
    isnothing(bad) || error("trajectory $(Tuple(bad)): " * get(_RBO_STATUS, Int(status[bad]), "error"))
    return map(1:B) do b
        μ = Distributions.mean(vals[:, b]); ∇μx = vec(Distributions.mean(gx[:, :, b], dims = 2)); ∇μθ = vec(Distributions.mean(gθ[:, :, b], dims = 2))
        ExpectedTrajectoryOutput(μxθ = μ, σ_μxθ = Distributions.std(vals[:, b], mean = μ), ∇μx = ∇μx,
                                 σ_∇μx = vec(Distributions.std(gx[:, :, b], dims = 2, mean = ∇μx)), ∇μθ = ∇μθ,
                                 σ_∇μθ = vec(Distributions.std(gθ[:, :, b], dims = 2, mean = ∇μθ)))
    end
end

function multistart_base_solve!(surrogate::Surrogate, xfinal::Vector{T};
        spatial_lbs::Vector{T}, spatial_ubs::Vector{T}, guesses::Matrix{T}, θfixed::Vector{T}) where T <: Real
    if get_name(get_decision_rule(surrogate)) == "Random"                 # rbf_optim.jl:111-114 stays on the host RNG
        xfinal[:] = spatial_lbs .+ (spatial_ubs .- spatial_lbs) .* rand(length(spatial_lbs))
        return nothing
    end
    h = _rbo_handle()
    empty!(_RBO_RESIDENT)
    N = get_observed(surrogate)
    _rbo_set_surrogate!(h, surrogate.X, surrogate.L.data, surrogate.y, surrogate.c[1:N], N, surrogate.ψ, surrogate.g, surrogate.σn2)
    _rbo_check(h, ccall((:rbo_set_starts, librbo), Cint, (Ptr{Cvoid}, Ptr{Float64}, Cint), h.ptr, guesses, size(guesses, 2)))
    α = Ref{Float64}(0.0)
    _rbo_check(h, ccall((:rbo_multistart_base_solve, librbo), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ref{Float64}, Ptr{Cvoid}),
        h.ptr, θfixed, length(θfixed), spatial_lbs, spatial_ubs, xfinal, α, C_NULL))
    return nothing
end

# gen_low_discrepancy_sequence (utils.jl:65-74) and generate_initial_guesses (utils.jl:145-153) keep their host
# definitions from the reference checkout; librbo's device generators (rbo_generate_normals,
# rbo_generate_initial_guesses) are used when the normals never have to visit the host (bench.py).


# ---- the stochastic-gradient-ascent loop (utils.jl:235-265) ---------------------------------------------------------------
# HEAD calls simulate_adjoint_trajectory(surrogate, tpc; ...), which is defined nowhere (SURVEY.md 0.3): it is the Monte-Carlo
# estimator with its adjoint gradient on a trajectory built from the surrogate. The Trajectory / FantasySurrogate are cached per
# surrogate so that the loop allocates them once; with the resident inputs above an ascent iteration uploads only x0.
const _RBO_TRAJ = Ref{Any}(nothing)
function _rbo_trajectory(surrogate::Surrogate, tp::TrajectoryParameters)
    key = (objectid(surrogate), get_observed(surrogate), tp.horizon)
    c = _RBO_TRAJ[]
    if c === nothing || c[1] != key
        fs = FantasySurrogate(surrogate, tp.horizon)
        T = Trajectory(surrogate, fs; start = get_starting_point(tp), hypers = get_hyperparameters(tp), horizon = tp.horizon)
        _RBO_TRAJ[] = (key, T)
        return T
    end
    return c[2]
end

function simulate_adjoint_trajectory(surrogate::Surrogate, tp::TrajectoryParameters;
        inner_solve_xstarts::Matrix{Float64}, resolutions::Vector{Float64},
        spatial_gradients_container::Union{Nothing, Matrix{Float64}} = nothing,
        hyperparameter_gradients_container::Union{Nothing, Matrix{Float64}} = nothing)
    T = _rbo_trajectory(surrogate, tp)
    return _rbo_simulate(T, tp, inner_solve_xstarts, resolutions, spatial_gradients_container, hyperparameter_gradients_container)
end

# stochastic_solve (utils.jl:235-265), same signature and iteration cap (50); only the undefined callee is resolved. Every iteration
# is one simulate_adjoint_trajectory with the same normals (common random numbers) and a new x0.
function stochastic_solve(; optimizer::StochasticGradientAscent, surrogate::Surrogate, tp::TrajectoryParameters, es::ExperimentSetup,
                          start::AbstractVector)
    tpc = deepcopy(tp)
    set_starting_point!(tpc, deepcopy(start))
    for iter in 1:50
        eto = simulate_adjoint_trajectory(surrogate, tpc,
            inner_solve_xstarts = get_starts(es), resolutions = get_container(es, symbol = :f),
            spatial_gradients_container = get_container(es, symbol = :grad_f),
            hyperparameter_gradients_container = get_container(es, symbol = :grad_hypers))
        if eswavs(∇f = gradient(eto), var_∇f = std_gradient(eto) .^ 2, sample_size = tp.mc_iters)   # utils.jl:114-123
            break
        end
        update!(optimizer, x = get_starting_point(tpc), ∇f = gradient(eto))                            # optimizers.jl:16-22, 48-75
    end
    return get_starting_point(tpc)
end

# Not in the reference: stochastic_solve from every column of `starts` (d x B) in ONE library call (rbo_stochastic_solve_batch): each
# restart has its own optimiser state (from `optimizer`'s hyper-parameters; every restart starts fresh) and its own ESWAVS stop, all
# iterations run on the device and the host synchronises once. The dual directions are one rand(d, h, M) buffer shared by every
# restart and iteration (not the per-iteration rand(dim) consumption of stochastic_solve). Returns the d x B final iterates.
# Like the rest of this file it is not run in the build environment (no Julia); the Python mirror api.stochastic_solve_batch drives
# the same entry point in the tests.
struct RboSgaOpts
    optimizer::Int32; max_iterations::Int32; use_eswavs::Int32; project::Int32
    eta::Float64; beta1::Float64; beta2::Float64; eps::Float64
end
function _rbo_sga_opts(o::StochasticGradientAscent)
    o isa Adam || return RboSgaOpts(0, 50, 1, 0, o.η, 0.0, 0.0, 0.0)                       # StandardSGA (optimizers.jl:6-22)
    o.t == 0 || error("stochastic_solve_batch: the Adam optimiser has already stepped; pass an unused one")
    return RboSgaOpts(1, 50, 1, 0, o.η, o.β1, o.β2, hasproperty(o, :ϵ) ? o.ϵ : o.ε)          # optimizers.jl:25-40; utils.jl:244
end
function stochastic_solve_batch(; optimizer::StochasticGradientAscent, surrogate::Surrogate, tp::TrajectoryParameters, es::ExperimentSetup,
                                starts::Matrix{Float64})
    h = _rbo_handle()
    T = _rbo_trajectory(surrogate, tp)
    _rbo_sync_surrogate!(h, get_fantasy_surrogate(T))
    _rbo_sync_normals!(h, tp.rnstream_sequence)
    _rbo_sync_starts!(h, get_starts(es))
    M, d, hor, B = tp.mc_iters, length(tp.x0), tp.horizon, size(starts, 2)
    θ = Vector{Float64}(tp.θ)
    dual = rand(d, max(hor, 1), M)
    opts = Ref(_rbo_sga_opts(optimizer))
    xfinal = zeros(d, B); n_iter = zeros(Int32, B); end_status = zeros(Int32, B); fail = zeros(Int32, 2, B)
    _rbo_check(h, ccall((:rbo_stochastic_solve_batch, librbo), Cint,
        (Ptr{Cvoid}, Ref{RboSgaOpts}, Ptr{Float64}, Cint, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Ptr{Float64},
         Ptr{Float64}, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cvoid}),
        h.ptr, opts, starts, B, θ, length(θ), tp.spatial_lbs, tp.spatial_ubs, hor, minimum(get_observations(surrogate)), dual,
        xfinal, n_iter, end_status, fail, C_NULL, C_NULL, C_NULL, C_NULL, C_NULL, C_NULL))
    for b in 1:B
        end_status[b] == 2 || continue                                                      # RBO_SGA_FAILED: the serial loop would throw
        error("restart $b, sample $(fail[1, b] + 1): " * get(_RBO_STATUS, Int(fail[2, b]), "error"))
    end
    return xfinal
end


# ---- single-process multi-GPU (SURVEY.md section 8e) -----------------------------------------------------------------------
# One handle per device; contiguous shards of the sample indices; the launches are asynchronous (rbo_rollout_device returns after
# the launch), so all GPUs work concurrently; rbo_get_results copies each shard of the containers back and the statistics are taken
# over the filled containers exactly as rollout.jl:328-337. (A multi-process host all-reduces rbo_partial_sums_device instead, as
# bench.py does with NCCL.) The rand(dim) stream is reproduced by the same two-phase scheme as on one GPU.
const _RBO_HANDLES = RboHandle[]
function _rbo_handles(ndev::Int)
    while length(_RBO_HANDLES) < ndev
        push!(_RBO_HANDLES, RboHandle(length(_RBO_HANDLES)))
    end
    return _RBO_HANDLES[1:ndev]
end

function simulate_trajectory_mc_multigpu(T::Trajectory, tp::TrajectoryParameters, ndev::Int;
        inner_solve_xstarts::Matrix{Float64}, resolutions::Vector{Float64},
        spatial_gradients_container::Matrix{Float64}, hyperparameter_gradients_container::Matrix{Float64})
    hs = _rbo_handles(ndev)
    fs = get_fantasy_surrogate(T)
    set_start!(T, get_starting_point(tp))
    N = get_known_observations(fs)
    rn = tp.rnstream_sequence
    M, d, hor = tp.mc_iters, length(tp.x0), tp.horizon
    θ = Vector{Float64}(tp.θ)
    fmini = minimum(get_observations(get_base_surrogate(T)))
    bounds = [div(M * g, ndev) for g in 0:ndev]
    for (g, h) in enumerate(hs)
        _rbo_set_surrogate!(h, fs.X, fs.L.data, fs.y, fs.cs[1], N, fs.ψ, fs.g, fs.σn2)
        _rbo_check(h, ccall((:rbo_set_normals, librbo), Cint, (Ptr{Cvoid}, Ptr{Float64}, Cint, Cint, Cint, Cint), h.ptr, rn, M, size(rn, 3), bounds[g], bounds[g+1] - bounds[g]))
        _rbo_check(h, ccall((:rbo_set_starts, librbo), Cint, (Ptr{Cvoid}, Ptr{Float64}, Cint), h.ptr, inner_solve_xstarts, size(inner_solve_xstarts, 2)))
    end
    launch(h, mode, flags, dual_dev) = _rbo_check(h, ccall((:rbo_rollout_device, librbo), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Cint, Cint, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}),
        h.ptr, tp.x0, θ, length(θ), tp.spatial_lbs, tp.spatial_ubs, hor, fmini, mode, flags, dual_dev, C_NULL, C_NULL))
    fetch!(h, lo, hi, v, gx, gθ, bi, st) = _rbo_check(h, ccall((:rbo_get_results, librbo), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}),
        h.ptr, pointer(v, lo + 1), gx === nothing ? C_NULL : pointer(gx, d * lo + 1), gθ === nothing ? C_NULL : pointer(gθ, length(θ) * lo + 1),
        bi === nothing ? C_NULL : pointer(bi, lo + 1), C_NULL, pointer(st, lo + 1)))
    status = zeros(Int32, M); best_index = zeros(Int32, M)
    # phase 1 on every device (values, best indices), then the reference's RNG consumption on the host, then phase 2 (replay + adjoint)
    foreach(h -> launch(h, 0, 0, C_NULL), hs)
    for (g, h) in enumerate(hs)
        fetch!(h, bounds[g], bounds[g+1], resolutions, nothing, nothing, best_index, status)
    end
    _rbo_first_error(status)
    dual = zeros(d, max(hor, 1), M)
    for m in 1:M
        t = Int(best_index[m])
        if resolutions[m] > 0.0 && t >= 1
            for j in t:-1:1
                dual[:, j, m] = rand(d)
            end
        end
    end
    # rbo_rollout (host pointers) uploads the shard's dual directions; it is synchronous per handle, so phase 2 is issued through the
    # device entry point after an explicit upload would be the asynchronous alternative -- phase 2 is ~5 % of the work (no inner solves)
    for (g, h) in enumerate(hs)
        lo, hi = bounds[g], bounds[g+1]
        summary = RboSummary()
        _rbo_check(h, ccall((:rbo_rollout, librbo), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Cint, Cint, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ref{RboSummary}),
            h.ptr, tp.x0, θ, length(θ), tp.spatial_lbs, tp.spatial_ubs, hor, fmini, 1, 8 #= RBO_FLAG_REPLAY_TAPE =#,
            pointer(dual, d * max(hor, 1) * lo + 1), C_NULL, pointer(resolutions, lo + 1), pointer(spatial_gradients_container, d * lo + 1),
            pointer(hyperparameter_gradients_container, length(θ) * lo + 1), C_NULL, C_NULL, pointer(status, lo + 1), summary))
    end
    _rbo_first_error(status)
    empty!(_RBO_RESIDENT)
    μxθ = Distributions.mean(resolutions); σ_μxθ = Distributions.std(resolutions, mean = μxθ)
    ∇μx = vec(Distributions.mean(spatial_gradients_container, dims = 2))
    ∇μθ = vec(Distributions.mean(hyperparameter_gradients_container, dims = 2))
    return ExpectedTrajectoryOutput(μxθ = μxθ, σ_μxθ = σ_μxθ, ∇μx = ∇μx, σ_∇μx = vec(Distributions.std(spatial_gradients_container, dims = 2, mean = ∇μx)),
                                    ∇μθ = ∇μθ, σ_∇μθ = vec(Distributions.std(hyperparameter_gradients_container, dims = 2, mean = ∇μθ)))
end
