# AriannaCUDA.jl -- thin Julia shim that plugs libarianna_cuda.so (include/arianna_cuda.h) in behind Arianna.jl's
# own `Simulation` / `run!` / `Metropolis` / `StoreCallbacks` / `StoreTrajectories` / `PolicyGradientEstimator`.
#
# STATUS: written against the C ABI and the reference sources, NOT executed -- the build environment has no Julia
# toolchain (SURVEY.md §7 item 9).  The Python mirror (montecarlo_b200/arianna.py) exercises the identical call
# sequence through the identical ABI and is what the parity tests run.
#
# Design (SURVEY.md §8b): `CudaEnsemble <: AriannaSystem` is ONE system that *is* M device-resident chains, so
# `chains = [ensemble]` lets the unmodified reference driver run:  Metropolis.make_step! calls
# `mc_sweep!(ensemble, pool, rng; mc_steps)` once per step, which we overload to only COUNT pending steps; any
# observation (energy, acceptance, trajectory, estimator) first flushes them as one fused K-step kernel launch.
module AriannaCUDA

using Arianna
using Arianna.PolicyGuided
using ComponentArrays
using Libdl
using Random

export CudaEnsemble, callback_acceptance_cuda, flush!, device_positions, nccl_unique_id, comm_init!, plan!, run_host_job!,
       device_update!, set_ladder!, replica_exchange!, exchange_counters, ladder_sums

const MAX_MOVES = 16
const libarianna = Ref{String}(get(ENV, "ARIANNA_CUDA_LIB", "libarianna_cuda.so"))

# mirror of `struct arianna_config` (include/arianna_cuda.h) -- field order and widths must match exactly
struct AriannaConfig
    struct_size::UInt32
    device::Int32
    n_chains::Int64
    chain_offset::Int64
    n_chains_total::Int64
    seed::Int64
    beta::Float64
    potential::Int32
    n_moves::Int32
    sigma::NTuple{MAX_MOVES,Float64}
    weight::NTuple{MAX_MOVES,Float64}
    rng_mode::Int32
    arith_mode::Int32
    stream::Ptr{Cvoid}
    dtype::Int32                  # 0 = Float64, 1 = Float32 (Particle{Float32}, σ = 0.1f0)
    reserved::Int32
end

struct OptimiserSpec             # arianna_optimiser
    kind::Int32
    reserved::Int32
    p1::Float64
    p2::Float64
end

struct GradientRecord            # arianna_gradient_data
    j::Float64
    dj::Float64
    dlogq_forward::Float64
    g::Float64
    n::Float64
end

const POT = Dict(:harmonic => Int32(0), :quartic => Int32(1), :double_well => Int32(2))

function check(h::Ptr{Cvoid}, rc::Int32)
    rc == 0 && return nothing
    msg = unsafe_string(ccall((:arianna_last_error, libarianna[]), Cstring, (Ptr{Cvoid},), h))
    rc == 1 ? throw(ArgumentError(msg)) : error("libarianna_cuda error $rc: $msg")
end

"""
    CudaEnsemble(x0, β, pool; seed=1, potential=:harmonic, arith=:fast, chain_offset=0, n_total=length(x0))

M = length(x0) Metropolis chains of the `particle_1d` system resident in the HBM of the current CUDA device.
Replaces `chains = [System(x, β) for x in x0]` (MC_harmonic_oscillator.jl:13): use `chains = [ensemble]`.
"""
mutable struct CudaEnsemble{T<:AbstractFloat} <: AriannaSystem
    handle::Ptr{Cvoid}
    M::Int
    β::T
    pool::Any
    pending::Int            # Metropolis steps counted by mc_sweep! but not yet launched
    cache_t::Int            # steps_done at which (energy, acceptance) were last reduced
    energy::Float64
    acceptance::Vector{Float64}
    # look-ahead over callback-only stores (plan!): MC steps already executed beyond the driver's time, the records
    # of the stores inside that stretch keyed by "MC steps done", and the planner closure installed by plan!
    ahead::Int
    series::Dict{Int,Tuple{Float64,Vector{Float64}}}
    lookahead::Any
end

function CudaEnsemble(x0::Vector{Float64}, β::Float64, pool; seed::Int=1, potential::Symbol=:harmonic,
                      arith::Symbol=:fast, rng::Symbol=:philox, chain_offset::Int=0, n_total::Int=length(x0),
                      device::Int=-1)
    nm = length(pool)
    nm <= MAX_MOVES || throw(ArgumentError("at most $MAX_MOVES moves per pool"))
    pad(v) = ntuple(k -> k <= nm ? Float64(v[k]) : 0.0, MAX_MOVES)
    cfg = AriannaConfig(UInt32(sizeof(AriannaConfig)), Int32(device), length(x0), chain_offset, n_total, seed, β,
                        POT[potential], Int32(nm), pad([m.parameters.σ for m in pool]), pad([m.weight for m in pool]),
                        Int32(rng == :xoshiro ? 1 : 0), Int32(arith == :exact ? 0 : 1), C_NULL, Int32(0), Int32(0))
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(C_NULL, ccall((:arianna_create, libarianna[]), Int32, (Ref{AriannaConfig}, Ref{Ptr{Cvoid}}), cfg, h))
    ens = CudaEnsemble{Float64}(h[], length(x0), β, pool, 0, -1, NaN, fill(NaN, nm), 0,
                                Dict{Int,Tuple{Float64,Vector{Float64}}}(), nothing)
    check(ens.handle, ccall((:arianna_set_state, libarianna[]), Int32, (Ptr{Cvoid}, Ptr{Float64}), ens.handle, x0))
    if rng == :xoshiro
        # the reference's own generators, rngs = [Xoshiro(seed + c - 1) for c in 1:M] (metropolis.jl:262-263), run on the
        # device: upload their states (xoshiro256++ s0..s3); the ziggurat tables default to the engine's own
        states = Matrix{UInt64}(undef, 4, length(x0))
        for c in 1:length(x0)
            r = Xoshiro(seed + chain_offset + c - 1)
            states[1, c], states[2, c], states[3, c], states[4, c] = r.s0, r.s1, r.s2, r.s3
        end
        check(ens.handle, ccall((:arianna_set_rng_state, libarianna[]), Int32, (Ptr{Cvoid}, Ptr{UInt64}), ens.handle, states))
    end
    finalizer(e -> ccall((:arianna_destroy, libarianna[]), Int32, (Ptr{Cvoid},), e.handle), ens)
    return ens
end

"""
    nccl_unique_id() -> Vector{UInt8}          (rank 0; broadcast it with MPI.jl / Distributed / a file)
    comm_init!(ens, id, rank, nranks)          (every rank, ens built with chain_offset / n_total of its shard)

Multi-GPU: one Julia process per GPU; the callback and estimator sums are all-reduced inside libarianna_cuda.so.
"""
function nccl_unique_id()
    id = Vector{UInt8}(undef, 128)
    check(C_NULL, ccall((:arianna_nccl_unique_id, libarianna[]), Int32, (Ptr{UInt8},), id))
    return id
end
comm_init!(ens, id::Vector{UInt8}, rank::Int, nranks::Int) =
    check(ens.handle, ccall((:arianna_comm_init, libarianna[]), Int32, (Ptr{Cvoid}, Ptr{UInt8}, Int32, Int32),
                            ens.handle, id, rank, nranks))

# Metropolis(chains; pool) deep-copies the pool per chain and the estimator deep-copies the chains
# (metropolis.jl:289, estimator.jl:86): a raw handle must never be duplicated.
Base.deepcopy_internal(e::CudaEnsemble, ::IdDict) = e

# --- the hot path --------------------------------------------------------------------------------------------
# mc_sweep!(system, pool, rng; mc_steps) (metropolis.jl:203-212), exported and overloadable (src/Arianna.jl:36)
function Arianna.mc_sweep!(ens::CudaEnsemble, pool, rng; mc_steps=1)
    if ens.ahead > 0                               # steps already run by a series launch (look-ahead)
        mc_steps <= ens.ahead || error("look-ahead plan violated: more Metropolis steps than planned")
        ens.ahead -= mc_steps
    else
        ens.pending += mc_steps
    end
    return nothing
end

"""
    plan!(simulation)

Call once before `run!(simulation)`.  The schedule is known up front (`simulation.schedulers`), so when
`StoreCallbacks` fires the ensemble can execute every following callback-only store interval, up to the next event
that observes or changes the chains in any other way, as ONE `arianna_sweep_series` call (chains stay in registers
across the intervals; one record per store is reduced on the device; one all-reduce per stretch).  Mirrors
`montecarlo_b200/arianna.py:_make_lookahead`.  Without `plan!` every store is one fused launch (still correct).
"""
function plan!(simulation::Simulation)
    ens = simulation.chains[1]
    algs = simulation.algorithms
    met = findall(a -> a isa Metropolis, algs)
    cbs = findall(a -> a isa StoreCallbacks && all(cb -> nameof(cb) in (:callback_energy, :callback_acceptance_cuda), a.callbacks), algs)
    (length(met) == 1 && !isempty(cbs) && minimum(cbs) > met[1]) || return nothing
    m = met[1]
    # never looks at the chains during the t-loop: Metropolis itself, the progress printer, and every algorithm whose
    # make_step! is the no-op default of algorithms.jl:25 (e.g. StoreLastFrames only acts in finalise)
    default_step = which(Arianna.make_step!, Tuple{Simulation,Arianna.AriannaAlgorithm})
    passive(a) = a isa Metropolis || a isa Arianna.PrintTimeSteps ||
                 which(Arianna.make_step!, Tuple{typeof(simulation),typeof(a)}) === default_step
    times(pred) = sort(unique(vcat([simulation.schedulers[k] for k in eachindex(algs)
                                    if !(k in cbs) && !passive(algs[k]) && pred(k)]..., Int[])))
    # a barrier listed AFTER Metropolis sees the state after the Metropolis step of its time (the stretch may include a
    # store AT that time); one listed BEFORE Metropolis sees the state before it: the stretch must stop short of it
    barriers_post, barriers_pre = times(k -> k > m), times(k -> k < m)
    stores = sort(unique(vcat([simulation.schedulers[k] for k in cbs]...)))
    msched = sort(simulation.schedulers[m])
    step = algs[m].sweepstep
    ens.lookahead = function ()
        t = simulation.t
        ib = searchsortedfirst(barriers_post, t)
        tb = ib <= length(barriers_post) ? barriers_post[ib] : simulation.steps + 1
        ip = searchsortedlast(barriers_pre, t) + 1
        tp = ip <= length(barriers_pre) ? barriers_pre[ip] : simulation.steps + 2
        out, prev = Int64[], t
        for ts in stores[searchsortedlast(stores, t)+1:end]
            (ts > tb || ts >= tp || length(out) >= 4096) && break
            push!(out, step * (searchsortedlast(msched, ts) - searchsortedlast(msched, prev)))
            prev = ts
        end
        return out
    end
    return nothing
end

"""
    run_host_job!(ens, x_in, Ks; x_out=nothing, n_slices=16) -> records::Matrix{Float64} ((2 + nmoves) × length(Ks))

A whole callbacks-only job with host buffers in one call (arianna_run_host_job): chains in, `length(Ks)` store
intervals of `Ks[i]` Metropolis steps, `(Σe, Σacc/tot per move, count)` per store out, final chains out; the library pipelines
slices of chains so that the PCIe copies overlap the sweeps.  With a communicator the records are all-reduced.
"""
function run_host_job!(ens::CudaEnsemble, x_in::Union{Nothing,Vector{Float64}}, Ks::Vector{Int64};
                       x_out::Union{Nothing,Vector{Float64}}=nothing, n_slices::Int=16)
    flush!(ens)
    n = length(Ks)
    rec = Matrix{Float64}(undef, 2 + length(ens.pool), n)
    check(ens.handle, ccall((:arianna_run_host_job, libarianna[]), Int32,
                            (Ptr{Cvoid}, Ptr{Float64}, Int32, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Int32), ens.handle,
                            x_in === nothing ? C_NULL : pointer(x_in), n, Ks, C_NULL,
                            x_out === nothing ? C_NULL : pointer(x_out), n_slices))
    check(ens.handle, ccall((:arianna_series_global, libarianna[]), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}),
                            ens.handle, n, rec))
    ens.cache_t = -1
    return rec
end

"One arianna_sweep_series call for [pending, K_1, K_2, ...]; every record lands in ens.series."
function run_series!(ens::CudaEnsemble, Ks::Vector{Int64})
    push_params!(ens)
    n = length(Ks)
    nm = length(ens.pool)
    rec = Matrix{Float64}(undef, 2 + nm, n)            # per store: Σe, Σ_c acc_ck/tot_ck for every move k, chain count
    check(ens.handle, ccall((:arianna_sweep_series, libarianna[]), Int32, (Ptr{Cvoid}, Int32, Ptr{Int64}, Ptr{Float64}),
                            ens.handle, n, Ks, C_NULL))
    check(ens.handle, ccall((:arianna_series_global, libarianna[]), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}),
                            ens.handle, n, rec))                      # all-reduced when a communicator is attached
    t = Ref{Int64}(0)
    check(ens.handle, ccall((:arianna_steps_done, libarianna[]), Int32, (Ptr{Cvoid}, Ref{Int64}), ens.handle, t))
    done = t[] - sum(Ks)
    empty!(ens.series)
    for i in 1:n
        done += Ks[i]
        ens.series[done] = (rec[1, i] / rec[2 + nm, i], rec[2:1 + nm, i] ./ rec[2 + nm, i])
    end
    ens.pending, ens.ahead, ens.cache_t = 0, sum(Ks[2:end]), -1
    return nothing
end

function push_params!(ens::CudaEnsemble)
    for (k, move) in enumerate(ens.pool)          # σ may have been mutated in place by learning_step! (learning.jl:33)
        θ = Ref(Float64(move.parameters.σ))
        lognorm = Ref(log(2π * move.parameters.σ^2) / 2)   # particle_1d.jl:53, Julia's own `log` for replay parity
        check(ens.handle, ccall((:arianna_set_params, libarianna[]), Int32,
                                (Ptr{Cvoid}, Int32, Ref{Float64}, Int32, Ref{Float64}), ens.handle, k - 1, θ, 1, lognorm))
    end
end

"Launch the pending Metropolis steps as ONE fused kernel (K = steps since the last observation)."
function flush!(ens::CudaEnsemble; reduce::Bool=false)
    ens.ahead == 0 || error("the device ensemble ran ahead of the schedule and something outside the plan observed it")
    push_params!(ens)
    if ens.pending > 0
        check(ens.handle, ccall((:arianna_sweep, libarianna[]), Int32, (Ptr{Cvoid}, Int64, UInt32),
                                ens.handle, ens.pending, reduce ? 1 : 0))
        ens.pending = 0
        ens.cache_t = -1
    end
    return nothing
end

function reduce_callbacks!(ens::CudaEnsemble)
    t = Ref{Int64}(0)
    if ens.pending == 0 && !isempty(ens.series)           # a store inside a stretch that already ran
        check(ens.handle, ccall((:arianna_steps_done, libarianna[]), Int32, (Ptr{Cvoid}, Ref{Int64}), ens.handle, t))
        hit = get(ens.series, t[] - ens.ahead, nothing)
        if hit !== nothing
            ens.energy, ens.cache_t = hit[1], ens.ahead == 0 ? t[] : -1
            ens.acceptance .= hit[2]
            return nothing
        end
        ens.ahead == 0 || error("look-ahead plan violated: callbacks requested at an unplanned time")
    end
    if ens.pending > 0 && ens.lookahead !== nothing
        Ks = ens.lookahead()
        if !isempty(Ks)
            run_series!(ens, vcat(Int64[ens.pending], Ks))
            return reduce_callbacks!(ens)
        end
    end
    flush!(ens; reduce=true)
    check(ens.handle, ccall((:arianna_steps_done, libarianna[]), Int32, (Ptr{Cvoid}, Ref{Int64}), ens.handle, t))
    if ens.cache_t != t[]
        e = Ref{Float64}(0.0)
        # *_global == the local call on one GPU; with a communicator (comm_init!) it all-reduces over NVLink first
        check(ens.handle, ccall((:arianna_callbacks_global, libarianna[]), Int32, (Ptr{Cvoid}, Ref{Float64}, Ptr{Float64}),
                                ens.handle, e, ens.acceptance))
        ens.energy, ens.cache_t = e[], t[]
    end
    return nothing
end

# `callback_energy(simulation) = mean(system.e for system in simulation.chains)` (particle_1d.jl:68-70) keeps working
# verbatim because `ensemble.e` IS the device-reduced mean energy of its M chains.
function Base.getproperty(ens::CudaEnsemble, s::Symbol)
    if s === :e
        reduce_callbacks!(ens)
        return getfield(ens, :energy)
    elseif s === :x
        return device_positions(ens)
    end
    return getfield(ens, s)
end

"callback_acceptance for device chains: per-move MEAN OVER CHAINS of accepted/total (metropolis.jl:319-321)."
function callback_acceptance_cuda(simulation)
    ens = simulation.chains[1]
    reduce_callbacks!(ens)
    return copy(getfield(ens, :acceptance))
end

function device_positions(ens::CudaEnsemble)
    flush!(ens)
    x = Vector{Float64}(undef, getfield(ens, :M))
    check(ens.handle, ccall((:arianna_get_state, libarianna[]), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}),
                            ens.handle, x, C_NULL))
    return x
end

# store_trajectory(io, system, t, fmt) (particle_1d.jl:63-66): one binary frame (t, x[M]) instead of M text files
function Arianna.store_trajectory(io, ens::CudaEnsemble, t::Int, ::Arianna.DAT)
    write(io, Int64(t))
    write(io, device_positions(ens))
    return nothing
end

# --- replica exchange (parallel tempering) across per-chain β ladders -----------------------------------------
# Every L = length(betas) consecutive chains (global index) form one ladder, chain g at β = betas[g % L + 1]; the shard
# (chain_offset, M) must hold whole ladders.  A `ReplicaExchange <: AriannaAlgorithm` whose make_step! calls
# replica_exchange! sits next to Metropolis in algorithm_list.
"""
    set_ladder!(ens, betas)      per-chain β from a ladder of L = length(betas) rungs (arianna_set_ladder)
    replica_exchange!(ens)       one exchange round, even / odd rung pairs alternating (arianna_replica_exchange)
    exchange_counters(ens)       (accepted[L-1], attempted[L-1], rounds) of the local shard
    ladder_sums(ens)             per-rung callback sums, L × (2 + n_moves): (Σe, Σ acc/tot per move, count)
"""
function set_ladder!(ens::CudaEnsemble, betas::Vector{Float64})
    check(ens.handle, ccall((:arianna_set_ladder, libarianna[]), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}),
                            ens.handle, length(betas), betas))
    return nothing
end

function replica_exchange!(ens::CudaEnsemble)
    flush!(ens)
    check(ens.handle, ccall((:arianna_replica_exchange, libarianna[]), Int32, (Ptr{Cvoid},), ens.handle))
    ens.cache_t = -1                              # the swap changed the energies behind the cached record
    empty!(ens.series)
    return nothing
end

function exchange_counters(ens::CudaEnsemble, L::Int)
    acc = Vector{Int64}(undef, L - 1)
    rounds = Ref{Int64}(0)
    check(ens.handle, ccall((:arianna_exchange_counters, libarianna[]), Int32, (Ptr{Cvoid}, Ptr{Int64}, Ref{Int64}),
                            ens.handle, acc, rounds))
    R = rounds[]
    attempted = [(getfield(ens, :M) ÷ L) * (iseven(k - 1) ? (R + 1) ÷ 2 : R ÷ 2) for k in 1:L-1]
    return acc, attempted, R
end

function ladder_sums(ens::CudaEnsemble, L::Int)
    flush!(ens)
    w = 2 + length(getfield(ens, :pool))
    out = Matrix{Float64}(undef, w, L)            # column r = the record of rung r (C row-major [L][w])
    check(ens.handle, ccall((:arianna_ladder_sums, libarianna[]), Int32, (Ptr{Cvoid}, Ptr{Float64}), ens.handle, out))
    return permutedims(out)
end

# --- PGMC ----------------------------------------------------------------------------------------------------
# make_step!(sim, ::PolicyGradientEstimator) (estimator.jl:111-134) for a simulation whose chains are device-resident:
# one fused device pass per learnable move; the summed record comes back as GradientData with n = M·q_batch.
function Arianna.make_step!(simulation::Simulation{<:CudaEnsemble}, algorithm::PolicyGradientEstimator)
    ens = simulation.chains[1]
    flush!(ens)
    ids = Int32.(algorithm.learn_ids .- 1)
    check(ens.handle, ccall((:arianna_pgmc_reset, libarianna[]), Int32, (Ptr{Cvoid},), ens.handle))
    check(ens.handle, ccall((:arianna_pgmc_estimate, libarianna[]), Int32, (Ptr{Cvoid}, Int32, Ptr{Int32}, Int32),
                            ens.handle, algorithm.q_batch_size, ids, length(ids)))
    recs = Vector{GradientRecord}(undef, length(ids))
    check(ens.handle, ccall((:arianna_pgmc_read_global, libarianna[]), Int32, (Ptr{Cvoid}, Ptr{GradientRecord}, Int32),
                            ens.handle, recs, length(ids)))
    for (k, r) in enumerate(recs)
        gd = Arianna.PolicyGuided.GradientData(r.j, ComponentArray(σ=r.dj), ComponentArray(σ=r.dlogq_forward),
                                               fill(r.g, 1, 1), Int(r.n))
        algorithm.gradients_data[k] = algorithm.gradients_data[k] + gd             # estimator.jl:130
        algorithm.objectives[k] = algorithm.gradients_data[k].j / algorithm.gradients_data[k].n
    end
    return nothing
end

# PolicyGradientUpdate on the device (arianna_pgmc_update_device): the averaging, learning_step! of every learnable move
# and the reset of the accumulators run in one kernel; σ stays in a device-resident block that the sweeps read.  Opt-in:
# call `device_update!(simulation, update_algorithm)` from a `make_step!` overload, or use it directly; it needs the
# estimator sums to be ACCUMULATED on the device, i.e. an estimator step that does not reset them (accumulate = true).
optimiser_spec(o::Arianna.PolicyGuided.VPG) = OptimiserSpec(Int32(1), Int32(0), o.η, 0.0)
optimiser_spec(o::Arianna.PolicyGuided.BLPG) = OptimiserSpec(Int32(2), Int32(0), o.η, 0.0)
optimiser_spec(o::Arianna.PolicyGuided.BLAPG) = OptimiserSpec(Int32(3), Int32(0), o.δ, o.ϵid)
optimiser_spec(o::Arianna.PolicyGuided.NPG) = OptimiserSpec(Int32(4), Int32(0), o.η, o.ϵid)
optimiser_spec(o::Arianna.PolicyGuided.ANPG) = OptimiserSpec(Int32(5), Int32(0), o.δ, o.ϵid)
optimiser_spec(o::Arianna.PolicyGuided.BLANPG) = OptimiserSpec(Int32(6), Int32(0), o.δ, o.ϵid)
optimiser_spec(::Any) = OptimiserSpec(Int32(0), Int32(0), 0.0, 0.0)           # Static

function device_update!(simulation::Simulation, algorithm::PolicyGradientUpdate)
    ens = simulation.chains[1]
    ids = Int32.(algorithm.learn_ids .- 1)
    specs = [optimiser_spec(algorithm.optimisers[k]) for k in algorithm.learn_ids]
    check(ens.handle, ccall((:arianna_pgmc_update_device, libarianna[]), Int32,
                            (Ptr{Cvoid}, Ptr{Int32}, Ptr{OptimiserSpec}, Int32), ens.handle, ids, specs, length(ids)))
    # refresh the host Moves (one small synchronising read; StoreParameters prints move.parameters)
    check(ens.handle, ccall((:arianna_params_sync, libarianna[]), Int32, (Ptr{Cvoid},), ens.handle))
    θ = Ref{Float64}(0.0)
    for k in algorithm.learn_ids
        check(ens.handle, ccall((:arianna_get_params, libarianna[]), Int32, (Ptr{Cvoid}, Int32, Ref{Float64}, Int32),
                                ens.handle, k - 1, θ, 1))
        ens.pool[k].parameters.σ = θ[]
    end
    return nothing
end

end # module
