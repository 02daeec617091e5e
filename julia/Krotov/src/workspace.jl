# KrotovWrk -- the workspace of the reference (src/workspace.jl:30-200 of JuliaQuantumControl/Krotov.jl) with the device
# as the owner of the heavy fields.  The field names of the reference are kept (callbacks read them); what used to be
# 2N propagators and 3N storage arrays is ONE libkrotov_cuda handle plus thin views.  NOT EXECUTED IN THIS REPOSITORY.
using QuantumControl: QuantumControl, Trajectory
using QuantumControl.QuantumPropagators.Controls: get_controls, get_control_derivs, discretize_on_midpoints, evaluate
using QuantumControl.QuantumPropagators: QuantumPropagators, Cheby
using QuantumControl.Functionals: make_chi, J_T_sm, J_T_ss, J_T_re
using LinearAlgebra
using SparseArrays
using Dates: now

import .LibKrotovCuda

# ---- Chebyshev settings of one direction (what init_prop / reinit_prop! keep in a ChebyWrk) ------------------------------
# All propagators of a direction see the same pulses, so their control ranges move in lock-step; the spectral envelope
# and the coefficients are per distinct generator.  The reference's range hook (src/optimize.jl:238-244) decides when
# they are re-derived; the result travels to the device through `krotov_set_cheby`.
mutable struct ChebySettings
    generators::Vector{Any}            # distinct generators of this direction (adjoint generators backward)
    controls::Tuple
    tlist::Vector{Float64}
    backward::Bool
    limit::Float64                     # cheby_coeffs_limit
    buffer::Float64                    # specrange_buffer
    specrange_kwargs::Dict{Symbol,Any} # specrange_method, E_min, E_max, ...
    ranges::Vector{Tuple{Float64,Float64}}
    E_min::Vector{Float64}
    Delta::Vector{Float64}
    dt_class_of_step::Vector{Int32}
    dt_of_class::Vector{Float64}
    m::Matrix{Int32}                   # [n_dt_class, n_gen]
    coeffs::Array{Float64,3}           # [m_max, n_dt_class, n_gen]
end

function ChebySettings(generators, controls, tlist, pulses, backward; limit = 1e-12, buffer = 0.01, kwargs...)
    ranges = [(minimum(p), maximum(p)) for p in pulses]   # init_prop: un-widened ranges of the guess pulses
    s = ChebySettings(collect(Any, generators), controls, Vector{Float64}(tlist), backward, limit, buffer,
                      Dict{Symbol,Any}(kwargs), ranges, Float64[], Float64[], Int32[], Float64[],
                      Matrix{Int32}(undef, 0, 0), Array{Float64,3}(undef, 0, 0, 0))
    classify_steps!(s)
    derive!(s)
    s
end

# dt classes in propagation order: coefficients are re-derived only when the step differs from the one they belong to
function classify_steps!(s::ChebySettings)
    t = s.tlist
    N_T = length(t) - 1
    sgn = s.backward ? -1.0 : 1.0
    steps = s.backward ? (N_T:-1:1) : (1:N_T)
    classes = Float64[]
    s.dt_class_of_step = zeros(Int32, N_T)
    for n in steps
        dt = sgn * (t[n+1] - t[n])
        c = findfirst(x -> abs(x - dt) <= 1e-12 * max(1.0, abs(x)), classes)
        if c === nothing
            push!(classes, dt)
            c = length(classes)
        end
        s.dt_class_of_step[n] = c - 1
    end
    s.dt_of_class = classes
end

function derive!(s::ChebySettings)
    n_gen = length(s.generators)
    s.E_min = Vector{Float64}(undef, n_gen)
    s.Delta = Vector{Float64}(undef, n_gen)
    for (g, G) in enumerate(s.generators)
        lo = IdDict(c => r[1] for (c, r) in zip(s.controls, s.ranges))
        hi = IdDict(c => r[2] for (c, r) in zip(s.controls, s.ranges))
        a0, b0 = QuantumPropagators.SpectralRange.specrange(evaluate(G; vals_dict = hi); s.specrange_kwargs...)
        a1, b1 = QuantumPropagators.SpectralRange.specrange(evaluate(G; vals_dict = lo); s.specrange_kwargs...)
        E_lo, E_hi = min(a0, a1), max(b0, b1)
        delta = s.buffer * (E_hi - E_lo)
        s.E_min[g] = E_lo - delta / 2
        s.Delta[g] = (E_hi - E_lo) + delta
    end
    per = [[QuantumPropagators.Cheby.cheby_coeffs(s.Delta[g], dt; limit = s.limit) for dt in s.dt_of_class] for g in 1:n_gen]
    m_max = maximum(length(a) for row in per for a in row)
    s.m = Int32[length(per[g][c]) for c in eachindex(s.dt_of_class), g in 1:n_gen]
    s.coeffs = zeros(Float64, m_max, length(s.dt_of_class), n_gen)
    for g in 1:n_gen, c in eachindex(s.dt_of_class)
        s.coeffs[1:length(per[g][c]), c, g] .= per[g][c]
    end
end

# the range check of `reinit_prop!(...; transform_control_ranges)`: true when the device tables must be refreshed
function reinit!(s::ChebySettings, pulses, transform_control_ranges)
    stale = false
    for (l, p) in enumerate(pulses)
        lo, hi = transform_control_ranges(s.controls[l], minimum(p), maximum(p), true)
        stale |= lo < s.ranges[l][1] || hi > s.ranges[l][2]
    end
    if stale
        s.ranges = [transform_control_ranges(s.controls[l], minimum(p), maximum(p), false) for (l, p) in enumerate(pulses)]
        derive!(s)
    end
    stale
end

push!(s::ChebySettings, handle, direction) =
    LibKrotovCuda.set_cheby(handle, direction, s.dt_class_of_step, s.dt_of_class, s.E_min, s.Delta, s.m, s.coeffs)

# ---- views that stand in for the per-trajectory objects of the reference ------------------------------------------------
struct PropagatorView   # `wrk.fw_propagators[k]`, `wrk.bw_propagators[k]`
    wrk::Any
    k::Int
    backward::Bool
end
function Base.getproperty(v::PropagatorView, name::Symbol)
    name === :state || return getfield(v, name)
    wrk, k = getfield(v, :wrk), getfield(v, :k)
    getfield(v, :backward) ? wrk.bw_storage[k][:, 1] : final_states(wrk)[k]
end

struct StorageView      # `wrk.fw_storage[k]`, `wrk.bw_storage[k]` -> Matrix d x (N_T+1), fetched from HBM on demand
    wrk::Any
    which::Cint
end
Base.length(s::StorageView) = length(s.wrk.trajectories)
function Base.getindex(s::StorageView, k::Integer)
    wrk = s.wrk
    d, N_T = length(wrk.trajectories[k].initial_state), length(wrk.result.tlist) - 1
    out = Matrix{ComplexF64}(undef, d, N_T + 1)
    LibKrotovCuda.get_storage!(wrk.handle, s.which, k - 1, 0, N_T + 1, out)
    out
end

mutable struct KrotovWrk
    trajectories
    adjoint_trajectories
    kwargs
    controls
    pulses0::Vector{Vector{Float64}}   # the two pulse buffers alternate between guess and update
    pulses1::Vector{Vector{Float64}}
    g_a_int::Vector{Float64}
    update_shapes::Vector{Vector{Float64}}
    lambda_vals::Vector{Float64}
    J_T_takes_tau::Bool
    chi_takes_tau::Bool
    result
    control_derivs
    fw_prop_kwargs::Vector{Dict{Symbol,Any}}
    bw_prop_kwargs::Vector{Dict{Symbol,Any}}
    fw_storage       # StorageView (needs `store_fw_states=true`)
    fw_storage2      # never read or written by the reference (src/workspace.jl:129-130): nothing
    bw_storage       # StorageView
    fw_propagators   # Vector{PropagatorView}
    bw_propagators
    use_threads::Bool
    # ---- device side
    handle::LibKrotovCuda.Handle
    chi_kind::Cint                     # KROTOV_CHI_*: which boundary condition the device forms by itself
    fw_cheby::ChebySettings
    bw_cheby::ChebySettings
    states_cache::Union{Nothing,Matrix{ComplexF64}}
    # ---- second order (`sigma`, documented at src/optimize.jl:104-105 of the reference, TODOs at :187, :350, :369)
    sigma            # nothing | a number | a callable sigma(t), optionally with a method `refresh!(sigma; info...)`
    sigma_info       # what `update_sigma!` hands to `refresh!`: Psi^(i)(T) and the chi(T) the iteration started from
end

# The one value a sigma takes over the time grid (sampled like the pulses).  The device path folds a time-independent
# sigma into the boundary condition of the backward sweep (see `krotov_iteration`); anything else is refused.
function sigma_value(sigma, tlist)
    vals = sigma isa Number ? fill(Float64(sigma), length(tlist) - 1) : discretize_on_midpoints(t -> Float64(sigma(t)), tlist)
    all(isfinite, vals) || throw(ArgumentError("sigma(t) is not finite on the time grid"))
    all(==(vals[1]), vals) || throw(ArgumentError(
        "sigma(t) varies over the time grid: the device path folds a time-independent sigma into the boundary " *
        "condition of the backward sweep; re-estimate it per iteration in `refresh!` instead"))
    vals[1]
end

function final_states(wrk::KrotovWrk)
    if wrk.states_cache === nothing
        d, N = length(wrk.trajectories[1].initial_state), length(wrk.trajectories)
        buf = Matrix{ComplexF64}(undef, d, N)
        LibKrotovCuda.get_states!(wrk.handle, buf)
        wrk.states_cache = buf
    end
    [wrk.states_cache[:, k] for k in axes(wrk.states_cache, 2)]
end

# prop_* keywords: problem keywords first, trajectory properties override; later prefixes override earlier ones
function harvest_prop_kwargs(traj, kwargs, prefixes)
    out = Dict{Symbol,Any}()
    for source in (kwargs, Dict(pairs(getfield(traj, :kwargs)))), prefix in prefixes, (key, val) in source
        name = String(key)
        startswith(name, prefix) && (out[Symbol(name[length(prefix)+1:end])] = val)
    end
    out
end

builtin_chi_kind(J_T) = J_T === J_T_sm ? LibKrotovCuda.KROTOV_CHI_SM :
                        J_T === J_T_ss ? LibKrotovCuda.KROTOV_CHI_SS :
                        J_T === J_T_re ? LibKrotovCuda.KROTOV_CHI_RE : LibKrotovCuda.KROTOV_CHI_HOST

function KrotovWrk(problem::QuantumControl.ControlProblem; verbose = false)
    kwargs = Dict(problem.kwargs)   # shallow copy; modified below
    trajectories = collect(problem.trajectories)
    N = length(trajectories)
    controls = get_controls(trajectories)
    isempty(controls) && error("no controls in trajectories: cannot optimize")
    tlist = Vector{Float64}(problem.tlist)
    N_T, L = length(tlist) - 1, length(controls)
    control_derivs = [get_control_derivs(traj.generator, controls) for traj in trajectories]

    # ---- pulse options: `pulse_options` wins over `lambda_a` / `update_shape` (same warnings as the reference)
    if haskey(kwargs, :pulse_options)
        haskey(kwargs, :update_shape) && @warn("`update_shape` is ignored due to given `pulse_options`")
        haskey(kwargs, :lambda_a) && @warn("`lambda_a=$(kwargs[:lambda_a])` is ignored due to given `pulse_options`")
    elseif !haskey(kwargs, :update_shape) && !haskey(kwargs, :lambda_a)
        @warn "Using default pulse_options: (:lambda_a => 1.0, :update_shape => (t -> 1.0))"
    end
    fallback = Dict(:lambda_a => convert(Float64, get(kwargs, :lambda_a, 1.0)), :update_shape => get(kwargs, :update_shape, t -> 1.0))
    pulse_options = get(kwargs, :pulse_options, IdDict(c => fallback for c in controls))
    all(c -> haskey(pulse_options, c), controls) || error("pulse_options must be defined for all controls")
    update_shapes = [discretize_on_midpoints(pulse_options[c][:update_shape], tlist) for c in controls]
    lambda_vals = Float64[pulse_options[c][:lambda_a] for c in controls]

    # ---- result and pulses: fresh, or continued from a previous (possibly foreign) result
    if haskey(kwargs, :continue_from)
        @info "Continuing previous optimization"
        result = convert(KrotovResult, kwargs[:continue_from])
        result.iter_stop = get(kwargs, :iter_stop, 5000)
        result.converged = false
        result.start_local_time = now()
        result.message = "in progress"
        pulses0 = [discretize_on_midpoints(c, tlist) for c in result.optimized_controls]
    else
        result = KrotovResult(problem)
        pulses0 = [discretize_on_midpoints(c, tlist) for c in controls]
    end
    pulses1 = map(copy, pulses0)

    # ---- propagator keywords: only the piecewise Chebyshev propagator runs on the device
    kwargs[:piecewise] = true
    adjoint_trajectories = [adjoint(traj) for traj in trajectories]
    fw_prop_kwargs = [harvest_prop_kwargs(t, kwargs, ("prop_", "fw_prop_")) for t in trajectories]
    bw_prop_kwargs = [harvest_prop_kwargs(t, kwargs, ("prop_", "bw_prop_")) for t in adjoint_trajectories]
    for pk in bw_prop_kwargs
        pk[:backward] = true
    end
    for pk in Iterators.flatten((fw_prop_kwargs, bw_prop_kwargs))
        get(pk, :method, nothing) in (Cheby, :Cheby, :cheby) ||
            throw(ArgumentError("prop_method=$(get(pk, :method, nothing)): libkrotov_cuda serves the `Cheby` propagator only"))
        haskey(pk, :callback) && throw(ArgumentError("per-step propagation callbacks cannot run inside the device sweep"))
    end

    haskey(kwargs, :J_T) || throw(ArgumentError("`optimize` for `method=Krotov` must be passed the functional `J_T`."))
    J_T = kwargs[:J_T]
    user_chi = haskey(kwargs, :chi)
    user_chi || (kwargs[:chi] = make_chi(J_T, trajectories))
    sig = Tuple{typeof(result.states),typeof(trajectories)}
    J_T_takes_tau = hasmethod(J_T, sig, (:tau,))
    chi_takes_tau = hasmethod(kwargs[:chi], sig, (:tau,))
    have_targets = all(t -> hasproperty(t, :target_state) && t.target_state !== nothing, trajectories)
    chi_kind = (user_chi || !have_targets) ? LibKrotovCuda.KROTOV_CHI_HOST : builtin_chi_kind(J_T)

    # ---- the device problem: distinct generators by identity, dense column-major terms
    gens = unique(objectid, [t.generator for t in trajectories])
    gen_of = Int32[findfirst(g -> g === t.generator, gens) - 1 for t in trajectories]
    d = length(trajectories[1].initial_state)
    vals = zeros(ComplexF64, d, d, 1 + L, length(gens))
    present = ones(UInt8, 1 + L, length(gens))
    for (g, G) in enumerate(gens)
        derivs = get_control_derivs(G, controls)
        vals[:, :, 1, g] .= Matrix(evaluate(G; vals_dict = IdDict(c => 0.0 for c in controls)))   # drift
        for l in 1:L
            if derivs[l] === nothing
                present[1+l, g] = 0
            else
                vals[:, :, 1+l, g] .= Matrix(derivs[l])
            end
        end
    end
    sigma = get(kwargs, :sigma, nothing)
    if sigma !== nothing
        all(ishermitian(@view vals[:, :, t, g]) for t in 1:(1+L), g in eachindex(gens)) || throw(ArgumentError(
            "`sigma` (second-order Krotov) needs Hermitian generators and control operators: the device path folds the " *
            "second-order term into the boundary condition chi(T)"))
        get(kwargs, :skip_initial_forward_propagation, false) && throw(ArgumentError(
            "`sigma` needs the forward states of the guess pulses: it cannot be combined with `skip_initial_forward_propagation`"))
        sigma_value(sigma, tlist)
        chi_kind = LibKrotovCuda.KROTOV_CHI_HOST   # chi(T) - sigma/2 Psi(T) is formed on the host and pushed with set_chi
    end
    psi0 = reduce(hcat, [Vector{ComplexF64}(t.initial_state) for t in trajectories])
    targets = have_targets ? reduce(hcat, [Vector{ComplexF64}(t.target_state) for t in trajectories]) : Matrix{ComplexF64}(undef, 0, 0)
    weights = Float64[hasproperty(t, :weight) ? t.weight : 1.0 for t in trajectories]
    S = reduce(hcat, update_shapes)   # Matrix(N_T, L): [L][N_T] on the wire
    store_fw = get(kwargs, :store_fw_states, false)
    handle = GC.@preserve tlist gen_of vals present psi0 targets weights S lambda_vals begin
        LibKrotovCuda.create(LibKrotovCuda.Problem(
            sizeof(LibKrotovCuda.Problem), d, N, L, N_T, length(gens), LibKrotovCuda.KROTOV_GEN_DENSE_COLMAJOR, 0,
            pointer(tlist), pointer(gen_of), C_NULL, C_NULL, Ptr{Float64}(pointer(vals)), pointer(present),
            Ptr{Float64}(pointer(psi0)), have_targets ? Ptr{Float64}(pointer(targets)) : C_NULL, pointer(weights),
            pointer(S), pointer(lambda_vals), chi_kind, 0, store_fw ? 1 : 0, get(kwargs, :device, 0),
            get(kwargs, :force_path, 0), get(kwargs, :replicated_forward, false) ? 1 : 0, LibKrotovCuda.KROTOV_PROP_CHEBY, ntuple(_ -> Int32(0), 5)))
    end

    pk = fw_prop_kwargs[1]
    init_pulses = haskey(kwargs, :continue_from) ? [discretize_on_midpoints(c, tlist) for c in controls] : pulses0
    spec = Dict{Symbol,Any}(k => v for (k, v) in pk if k in (:specrange_method, :E_min, :E_max))
    common = (; limit = get(pk, :cheby_coeffs_limit, 1e-12), buffer = get(pk, :specrange_buffer, 0.01))
    fw_cheby = ChebySettings(gens, controls, tlist, init_pulses, false; common..., spec...)
    bw_cheby = ChebySettings(map(adjoint, gens), controls, tlist, init_pulses, true; common..., spec...)
    push!(fw_cheby, handle, LibKrotovCuda.KROTOV_FORWARD)
    push!(bw_cheby, handle, LibKrotovCuda.KROTOV_BACKWARD)

    wrk = KrotovWrk(
        trajectories, adjoint_trajectories, kwargs, controls, pulses0, pulses1, zeros(L), update_shapes, lambda_vals,
        J_T_takes_tau, chi_takes_tau, result, control_derivs, fw_prop_kwargs, bw_prop_kwargs,
        nothing, nothing, nothing, nothing, nothing, get(kwargs, :use_threads, false),
        handle, chi_kind, fw_cheby, bw_cheby, nothing, sigma, nothing,
    )
    wrk.fw_storage = StorageView(wrk, LibKrotovCuda.KROTOV_FORWARD)
    wrk.bw_storage = StorageView(wrk, LibKrotovCuda.KROTOV_BACKWARD)
    wrk.fw_propagators = [PropagatorView(wrk, k, false) for k in 1:N]
    wrk.bw_propagators = [PropagatorView(wrk, k, true) for k in 1:N]
    wrk
end
