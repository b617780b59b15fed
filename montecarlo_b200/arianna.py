"""Host-side mirror of Arianna.jl's API for the multi-chain Metropolis hot path, driving libarianna_cuda.so.

Julia is not available in the build environment, so the host code that the north star places in Julia (a thin
`ccall` shim, see INTEGRATION.md and julia/AriannaCUDA.jl) is mirrored here in Python with the SAME names,
argument meaning, event order and error behaviour, so that the parity tests read like the reference's tests:

    chains = ParticleEnsemble(x0, β)                      # [System(4rand(rng) - 2, β) for _ in 1:M]
    pool = (Move(Displacement(0.0), StandardGaussian(), ComponentArray(σ=0.1), 1.0),)
    algorithm_list = (
        dict(algorithm=Metropolis, pool=pool, seed=seed, parallel=False),
        dict(algorithm=StoreCallbacks, callbacks=(callback_energy, callback_acceptance), scheduler=sampletimes),
        dict(algorithm=StoreTrajectories, scheduler=sampletimes),
    )
    simulation = Simulation(chains, algorithm_list, steps, path=path)
    run(simulation)                                       # run!(simulation)

Names that differ only because of Python syntax: `run!` -> `run`, `make_step!` -> `make_step`, NamedTuples ->
dicts.  Citations are path:line under the reference tree.

The chains live ONLY in HBM (one CudaEnsemble per process/GPU); `Metropolis.make_step` is lazy -- it only counts
pending steps -- and any observation (callbacks, trajectories, the PGMC estimator, reading `x`) first flushes
the pending steps as ONE fused K-step kernel launch.  That is how K = gap between store points reaches the kernel
without changing the driver loop (simulation.jl:184-191).
"""
from __future__ import annotations

import math
import os
import time
from typing import Callable, Optional, Sequence

import numpy as np

from .engine import CudaEnsemble

__all__ = [
    "AriannaSystem", "Particle", "System", "ParticleEnsemble", "Action", "Policy", "Displacement",
    "StandardGaussian", "ComponentArray", "Move", "Metropolis", "Simulation", "run", "build_schedule",
    "StoreCallbacks", "StoreTrajectories", "StoreLastFrames", "StoreParameters", "PrintTimeSteps",
    "callback_energy", "callback_acceptance", "mc_sweep", "DAT", "TXT", "shard_bounds",
    "ReplicaExchange", "callback_ladder_energy", "callback_ladder_acceptance", "callback_exchange_acceptance",
]


# ---------------------------------------------------------------------------------------------------------
# distributed plumbing: one process per GPU, chains sharded contiguously, NCCL only for the tiny sum vectors
# ---------------------------------------------------------------------------------------------------------
def _dist():
    try:
        import torch.distributed as dist
    except Exception:  # torch is optional for single-GPU use
        return None
    return dist if dist.is_available() and dist.is_initialized() else None


def shard_bounds(n_total: int, rank: int, world: int):
    """Contiguous block partition of the global chain ids (SURVEY.md §8e): (offset, count) of `rank`."""
    base, rem = divmod(int(n_total), int(world))
    count = base + (1 if rank < rem else 0)
    offset = rank * base + min(rank, rem)
    return offset, count


def allreduce_sums(local: np.ndarray, device_tensor=None) -> np.ndarray:
    """Sum a small f64 vector over all ranks.  With NCCL a device-side copy of the engine's buffer is reduced (no
    host round trip before the collective); with gloo (CPU tests) the host copy is reduced."""
    dist = _dist()
    if dist is None or dist.get_world_size() == 1:
        return local
    import torch
    if dist.get_backend() == "nccl" and device_tensor is not None:
        t = device_tensor.clone()  # keep the engine's local sums intact (they may be accumulated further)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t.cpu().numpy()
    t = torch.from_numpy(np.array(local, dtype=np.float64))
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t.numpy()


def means_from_sums(sums: np.ndarray, n_moves: int):
    """[Σe, Σ acc/tot per move, count] -> (callback_energy, callback_acceptance)."""
    cnt = sums[1 + n_moves]
    return sums[0] / cnt, sums[1:1 + n_moves] / cnt


# ---------------------------------------------------------------------------------------------------------
# System / actions / policies (example/particle_1d/particle_1d.jl)
# ---------------------------------------------------------------------------------------------------------
class AriannaSystem:
    """abstract type AriannaSystem (src/Arianna.jl:17)."""


class Particle(AriannaSystem):
    """mutable struct Particle{T}(x, β, e) (particle_1d.jl:9-16) -- host-side value object, only used to describe
    initial conditions for small ensembles; the running chains live in HBM."""

    def __init__(self, x: float, beta: float, potential: str = "harmonic"):
        self.x = float(x)
        self.β = self.beta = float(beta)
        self.potential = potential


def System(x, beta, potential: str = "harmonic"):
    """System(x, β) = Particle(x, β) (particle_1d.jl:18)."""
    return Particle(x, beta, potential)


class Action:
    """abstract type Action (metropolis.jl:15)."""


class Policy:
    """abstract type Policy (metropolis.jl:22)."""


class Displacement(Action):
    """mutable struct Displacement{T}(δ) (particle_1d.jl:26-28).  δ is per-chain scratch: register-only on device."""

    def __init__(self, delta: float = 0.0):
        self.δ = self.delta = float(delta)


class StandardGaussian(Policy):
    """struct StandardGaussian <: Policy (particle_1d.jl:48): δ ~ Normal(0, σ)."""


class ComponentArray:
    """ComponentArray(σ=...) [EXT ComponentArrays]: a named 1-vector θ = (σ), shared by every chain
    (metropolis.jl:253-260) and mutated in place by learning_step! (learning.jl:33)."""

    def __init__(self, σ: Optional[float] = None, sigma: Optional[float] = None):
        v = σ if σ is not None else sigma
        if v is None:
            raise TypeError("ComponentArray(σ=...) needs a value")
        self.data = np.array([float(v)], dtype=np.float64)

    @property
    def σ(self) -> float:
        return float(self.data[0])

    @σ.setter
    def σ(self, v: float):
        self.data[0] = float(v)

    sigma = σ

    def __eq__(self, other):
        return isinstance(other, ComponentArray) and np.array_equal(self.data, other.data)

    def __repr__(self):
        return f"ComponentArray(σ={self.σ!r})"


class Move:
    """mutable struct Move(action, policy, parameters, weight, total_calls, accepted_calls) (metropolis.jl:140-162).
    With the chains on the device the host Move holds the counters SUMMED over chains (refreshed on flush)."""

    def __init__(self, action: Action, policy: Policy, parameters: ComponentArray, weight: float):
        if not isinstance(action, Displacement) or not isinstance(policy, StandardGaussian):
            raise TypeError("the CUDA engine implements Move(Displacement, StandardGaussian, ComponentArray(σ), weight)")
        self.action, self.policy, self.parameters = action, policy, parameters
        self.weight = float(weight)
        self.total_calls = 0
        self.accepted_calls = 0


class ParticleEnsemble(AriannaSystem):
    """`chains::Vector{Particle}` as ONE object: M chains resident in HBM (the Python twin of the Julia shim's
    CudaEnsemble).  Construct from host positions (sharded automatically when torch.distributed is initialised)
    or synthetically (x0 = 4u − 2 from the engine's counter-based stream, MC_harmonic_oscillator.jl:13)."""

    def __init__(self, x0=None, beta=1.0, *, n_chains: Optional[int] = None, potential: str = "harmonic",
                 arith: str = "fast", rng: str = "philox", device: int = -1, init_seed: Optional[int] = None,
                 dtype: str = "f64"):
        if x0 is None and n_chains is None:
            raise ValueError("give x0 (host positions) or n_chains (synthetic initial condition)")
        if x0 is not None and not isinstance(x0, np.ndarray) and len(x0) and isinstance(x0[0], Particle):
            betas = [p.β for p in x0]
            beta = betas[0] if len(set(betas)) == 1 else np.array(betas)
            potential = x0[0].potential
            x0 = np.array([p.x for p in x0], dtype=np.float64)
        self.x0 = None if x0 is None else np.ascontiguousarray(x0, dtype=np.float64)
        self.n_total = int(n_chains if self.x0 is None else self.x0.size)
        # β may be one value or one value per chain (every Particle carries its own β, particle_1d.jl:11): a β sweep
        # such as BASELINE config 5 runs as ONE ensemble / one launch
        self.betas = None
        if np.ndim(beta) > 0:
            self.betas = np.ascontiguousarray(beta, dtype=np.float64)
            if self.betas.shape != (self.n_total,):
                raise ValueError("per-chain beta must have one entry per chain")
            beta = float(self.betas[0])
        self.β = self.beta = float(beta)
        self.potential, self.arith, self.rng, self.device = potential, arith, rng, device
        # element type of the chains: Particle{Float64} or Particle{Float32} (particle_1d.jl:9-16)
        self.dtype = {"f64": "f64", "f32": "f32", "float64": "f64", "float32": "f32"}[str(np.dtype(dtype)) if not isinstance(dtype, str) else dtype]
        self.init_seed = init_seed
        dist = _dist()
        self.rank = dist.get_rank() if dist else 0
        self.world = dist.get_world_size() if dist else 1
        self.offset, self.n_local = shard_bounds(self.n_total, self.rank, self.world)
        self.engine: Optional[CudaEnsemble] = None
        self.pool: Optional[Sequence[Move]] = None
        self.pending = 0
        self._cb_cache = None  # (steps_done, energy, acceptance)
        # look-ahead (set by run()): the engine may execute a whole stretch of callback-only store intervals in one
        # arianna_sweep_series call; `_ahead` = MC steps already executed beyond the driver's current time, and
        # `_series_cache` maps "MC steps done" -> (energy, acceptance) for the stores inside that stretch
        self._lookahead = None
        self._ahead = 0
        self._series_cache = {}
        self.max_lookahead = 4096

    def __len__(self):
        return self.n_total

    # bound by Metropolis (the engine needs the pool and the seed)
    def _bind(self, pool: Sequence[Move], seed: int):
        if self.engine is not None:
            raise RuntimeError("this ensemble is already bound to a Metropolis algorithm")
        self.pool = pool
        self.engine = CudaEnsemble(self.n_local, self.β, [m.parameters.σ for m in pool], [m.weight for m in pool],
                                   seed=seed, chain_offset=self.offset, n_chains_total=self.n_total,
                                   potential=self.potential, rng=self.rng, arith=self.arith, device=self.device,
                                   **({"dtype": "f32"} if self.dtype == "f32" else {}))
        if self.x0 is not None:
            self.engine.set_state(self.x0[self.offset:self.offset + self.n_local])
        else:
            self.engine.init_synthetic(seed if self.init_seed is None else self.init_seed)
        if self.betas is not None:
            self.engine.set_betas(self.betas[self.offset:self.offset + self.n_local])
        if self.rng == "xoshiro" and hasattr(self.engine, "set_rng_state"):
            # rngs = [Xoshiro(seed + c - 1) for c in 1:M] (metropolis.jl:262-263): Julia 1.7-1.10's own seeding, hashed on
            # the host in chunks and uploaded (julia_rng.py; [EXT], pinned by the Julia manual's known answers)
            from .julia_rng import xoshiro_states
            st = np.empty((self.n_local, 4), dtype=np.uint64)
            for a in range(0, self.n_local, 1 << 20):
                b = min(self.n_local, a + (1 << 20))
                st[a:b] = xoshiro_states(np.arange(seed + self.offset + a, seed + self.offset + b, dtype=np.int64))
            self.engine.set_rng_state(st)

    def _push_params(self):
        if getattr(self, "_params_on_device", False):
            return                       # the on-device optimiser owns σ: the host copies are refreshed by pull_params
        for k, m in enumerate(self.pool):
            if self.engine.get_params(k) != m.parameters.σ:
                self.engine.set_params(k, m.parameters.σ)

    def pull_params(self):
        """Refresh the host Moves' σ from the device (only needed after PolicyGradientUpdate(on_device=True))."""
        if getattr(self, "_params_on_device", False):
            for k, m in enumerate(self.pool):
                m.parameters.σ = self.engine.get_params(k)      # (the first call synchronises and pulls the whole block)

    def flush(self, reduce: bool = False):
        """Run the pending Metropolis steps as one fused launch."""
        if self.engine is None:
            raise RuntimeError("no Metropolis algorithm is attached to these chains")
        if self._ahead > 0:
            raise RuntimeError("the device ensemble ran ahead of the schedule (look-ahead over callback-only stores) "
                               "and something not in the plan observed or changed the chains")
        if self.pending > 0:
            self._push_params()
            self.engine.sweep(self.pending, reduce=reduce)
            self.pending = 0
            self._cb_cache = None

    def _advance(self, n: int):
        """n more Metropolis steps requested by the driver: queue them, or consume steps already run ahead."""
        if self._ahead > 0:
            if n > self._ahead:
                raise RuntimeError("look-ahead plan violated: more Metropolis steps than planned")
            self._ahead -= n
        else:
            self.pending += n

    def _series_supported(self):
        return (self._lookahead is not None and self.rng == "philox" and self.dtype == "f64"
                and hasattr(self.engine, "sweep_series"))

    def _run_series(self, Ks):
        """One arianna_sweep_series call for [pending, K_1, K_2, ...]; every record lands in the cache."""
        self._push_params()
        dist = _dist()
        nm = len(self.pool)
        if dist is not None and dist.get_world_size() > 1 and dist.get_backend() == "nccl":
            import torch
            self.engine.sweep_series(Ks, read=False)
            with torch.cuda.stream(self.engine.torch_stream()):
                rec = allreduce_sums(None, self.engine.series_tensor()).reshape(len(Ks), 2 + nm)   # ONE all-reduce
        else:
            rec = allreduce_sums(self.engine.sweep_series(Ks).reshape(-1)).reshape(len(Ks), 2 + nm)
        done = self.engine.steps_done - int(sum(Ks))
        self._series_cache = {}
        for K, r in zip(Ks, rec):
            done += int(K)
            e, a = means_from_sums(r, nm)
            self._series_cache[done] = (float(e), a)
        self.pending = 0
        self._ahead = int(sum(Ks[1:]))
        self._cb_cache = None

    def _callbacks(self):
        if self._ahead > 0 or (self.pending == 0 and self._series_cache):
            hit = self._series_cache.get(self.engine.steps_done - self._ahead) if self.pending == 0 else None
            if hit is not None:
                return hit
            if self._ahead > 0:
                raise RuntimeError("look-ahead plan violated: callbacks requested at an unplanned time")
        if self.pending > 0 and self._series_supported():
            ahead = self._lookahead()
            if ahead:
                self._run_series([self.pending] + ahead)
                return self._series_cache[self.engine.steps_done - self._ahead]
        self.flush(reduce=True)
        sd = self.engine.steps_done
        if self._cb_cache is None or self._cb_cache[0] != sd:
            dist = _dist()
            if dist is not None and dist.get_world_size() > 1 and dist.get_backend() == "nccl":
                import torch
                with torch.cuda.stream(self.engine.torch_stream()):
                    sums = allreduce_sums(None, self.engine.callback_sums_tensor())
            else:
                sums = allreduce_sums(self.engine.callback_sums())
            e, a = means_from_sums(sums, len(self.pool))
            self._cb_cache = (sd, float(e), a)
        return self._cb_cache[1], self._cb_cache[2]

    @property
    def x(self) -> np.ndarray:
        """Local shard of positions (system.x), in the chains' element type."""
        self.flush()
        return self.engine.get_state_f32() if self.dtype == "f32" else self.engine.get_state()

    @property
    def e(self) -> np.ndarray:
        self.flush()
        return self.engine.get_state(with_energy=True)[1]

    def sync_move_counters(self):
        self.flush()
        acc, tot = self.engine.counters()
        for k, m in enumerate(self.pool):
            m.accepted_calls, m.total_calls = int(acc[k]), int(tot[k])


# ---------------------------------------------------------------------------------------------------------
# build_schedule (src/simulation.jl:95-117)
# ---------------------------------------------------------------------------------------------------------
def _unique(seq):
    seen, out = set(), []
    for v in seq:
        if v not in seen:
            seen.add(v)
            out.append(v)
    return out


def build_schedule(steps: int, burn: int, spec):
    """Three methods, dispatched on the type of `spec` like the reference dispatches on Int / AbstractFloat /
    Vector{Int}."""
    if isinstance(spec, bool):
        raise TypeError("build_schedule: Δt must be an Int, a Float64 base or a block")
    if isinstance(spec, (int, np.integer)):
        if spec <= 0:
            raise ValueError("build_schedule: step must be positive")  # Julia: ArgumentError("step cannot be zero")
        return _unique(list(range(burn, steps + 1, int(spec))) + [steps])          # :95-97
    if isinstance(spec, (float, np.floating)):
        nmax = math.floor(math.log(steps - burn, spec))                             # :104-106
        mid = []
        for n in range(0, nmax + 1):
            v = spec ** n
            if v != math.floor(v):
                raise ValueError(f"InexactError: Int({v})")
            mid.append(burn + int(v))
        return _unique([burn] + mid + [steps])
    block = [int(b) for b in spec]                                                  # :113-117
    nblock = (steps - burn) // block[-1]
    out = []
    for m in range(1, nblock + 1):
        out.extend(b + burn + (m - 1) * block[-1] for b in block)
    return [t for t in _unique(out + [steps]) if t <= steps]


# ---------------------------------------------------------------------------------------------------------
# Algorithms (src/algorithms.jl, src/metropolis.jl)
# ---------------------------------------------------------------------------------------------------------
class AriannaAlgorithm:
    """abstract type AriannaAlgorithm with no-op lifecycle defaults (algorithms.jl:6-37)."""

    def initialise(self, simulation):
        return None

    def make_step(self, simulation):
        return None

    def finalise(self, simulation):
        return None

    def write_algorithm(self, io, scheduler):
        io.write(f"\t{type(self).__name__}\n")
        io.write(f"\t\tCalls: {sum(1 for x in scheduler if 0 < x <= scheduler[-1])}\n")


def mc_sweep(system: ParticleEnsemble, pool, rng=None, *, mc_steps: int = 1):
    """mc_sweep!(system, pool, rng; mc_steps) (metropolis.jl:203-212) for device-resident chains: lazy."""
    system._advance(int(mc_steps))


class Metropolis(AriannaAlgorithm):
    """Metropolis(chains; pool, sweepstep=1, seed=1, R=Xoshiro, parallel=false, extras...) (metropolis.jl:232-291).
    `parallel` and `R` are accepted for drop-in compatibility; the device engine is always parallel over chains
    and uses its counter-based stream keyed by seed + c − 1 (or rng="xoshiro" on the ensemble)."""

    def __init__(self, chains: ParticleEnsemble, *, pool=None, sweepstep: int = 1, seed: int = 1, R=None,
                 parallel: bool = False, **extras):
        if pool is None:
            raise TypeError("Metropolis: pool is required")
        if not isinstance(chains, ParticleEnsemble):
            raise TypeError("Metropolis: chains must be a ParticleEnsemble")
        self.pool = tuple(pool)
        self.pools = [self.pool]  # all chains alias one pool object (metropolis.jl:253-260)
        self.sweepstep, self.seed, self.parallel = int(sweepstep), int(seed), bool(parallel)
        chains._bind(self.pool, self.seed)

    def make_step(self, simulation):                       # metropolis.jl:302-309
        mc_sweep(simulation.chains, self.pool, None, mc_steps=self.sweepstep)

    def write_algorithm(self, io, scheduler):              # metropolis.jl:346-363
        io.write("\tMetropolis\n")
        io.write(f"\t\tCalls: {sum(1 for x in scheduler if 0 < x <= scheduler[-1])}\n")
        io.write(f"\t\tMC steps per simulation step: {self.sweepstep}\n")
        io.write(f"\t\tSeed: {self.seed}\n")
        io.write("\t\tParallel: true\n\t\tDevice: CUDA sm_100a (libarianna_cuda)\n\t\tMoves:\n")
        for k, move in enumerate(self.pool, 1):
            io.write(f"\t\t\tMove {k}:\n\t\t\t\tAction: {type(move.action).__name__}\n")
            io.write(f"\t\t\t\tPolicy: {type(move.policy).__name__}\n")
            io.write(f"\t\t\t\tParameters: [{move.parameters.σ!r}]\n\t\t\t\tWeight: {move.weight!r}\n")


def callback_energy(simulation) -> float:
    """mean(system.e for system in simulation.chains) (particle_1d.jl:68-70), fused device reduction."""
    return simulation.chains._callbacks()[0]


def callback_acceptance(simulation):
    """Per-move mean over chains of accepted_calls / total_calls (metropolis.jl:319-321); NaN at t = 0."""
    return [float(v) for v in simulation.chains._callbacks()[1]]


class ReplicaExchange(AriannaAlgorithm):
    """ReplicaExchange(chains; dependencies=(Metropolis,), ladder): parallel tempering across per-chain β ladders.
    Every L = len(ladder) consecutive chains (by global index) form one ladder, chain g at β = ladder[g % L].  Each call
    runs ONE exchange round on the device: round R proposes to swap the positions of rungs (r, r + 1) with
    r ≡ R (mod 2) in every ladder and accepts with min(1, exp((β_r − β_{r+1})(e_r − e_{r+1}))).  β and the Move
    counters stay with the rung (the temperature), only the configurations travel.  Every rank's shard must hold whole
    ladders."""

    def __init__(self, chains, *, dependencies=None, ladder=None, **extras):
        if not dependencies or len(dependencies) != 1 or not isinstance(dependencies[0], Metropolis):
            raise TypeError("ReplicaExchange: dependencies=(Metropolis,) is required")
        if ladder is None:
            raise TypeError("ReplicaExchange: ladder (the β of each rung) is required")
        self.ladder = np.ascontiguousarray(ladder, dtype=np.float64)
        L = self.ladder.size
        if self.ladder.ndim != 1 or not 2 <= L <= 256:
            raise ValueError("ReplicaExchange: the ladder must have 2 to 256 rungs")
        if chains.offset % L or chains.n_local % L:
            raise ValueError(f"ReplicaExchange: the shard of rank {chains.rank}, chains [{chains.offset}, "
                             f"{chains.offset + chains.n_local}), does not hold whole ladders of {L} chains")
        chains.engine.set_ladder(self.ladder)
        chains.betas = np.tile(self.ladder, chains.n_total // L)
        chains.β = chains.beta = float(self.ladder[0])

    def make_step(self, simulation):
        ch = simulation.chains
        ch.flush()
        ch.engine.replica_exchange()
        ch._cb_cache = None            # the swap changed the energies behind every cached record
        ch._series_cache = {}

    def write_algorithm(self, io, scheduler):
        calls = sum(1 for x in scheduler if 0 < x <= scheduler[-1])
        io.write(f"\tReplicaExchange\n\t\tCalls: {calls}\n")
        io.write(f"\t\tLadder: {self.ladder.size} rungs\n\t\tβ: {_jl(list(self.ladder))}\n")
        io.write(f"\t\tRounds: {calls} (one per call, even and odd rung pairs alternating)\n")


def _allreduce_host(v: np.ndarray) -> np.ndarray:
    """allreduce_sums of a host vector; under NCCL the collective needs a device copy of it."""
    dist = _dist()
    dev = None
    if dist is not None and dist.get_world_size() > 1 and dist.get_backend() == "nccl":
        import torch
        dev = torch.from_numpy(np.ascontiguousarray(v)).cuda()
    return allreduce_sums(v, dev)


def _ladder_sums(simulation) -> np.ndarray:
    ch = simulation.chains
    ch.flush()
    s = ch.engine.ladder_sums()
    return _allreduce_host(s.reshape(-1)).reshape(s.shape)


def callback_ladder_energy(simulation):
    """Mean energy of every rung of the β ladder (ReplicaExchange): [L] values, ensemble-wide."""
    s = _ladder_sums(simulation)
    return [float(v) for v in s[:, 0] / s[:, -1]]


def callback_ladder_acceptance(simulation):
    """callback_acceptance restricted to each rung: per rung, the per-move mean of accepted_calls / total_calls."""
    s = _ladder_sums(simulation)
    with np.errstate(all="ignore"):
        return [[float(v) for v in row[1:-1] / row[-1]] for row in s]


def callback_exchange_acceptance(simulation):
    """Accepted / attempted swaps of every rung pair (r, r + 1) since the ladder was set; NaN before the first attempt."""
    acc, att, _ = simulation.chains.engine.exchange_counters()
    tot = _allreduce_host(np.concatenate([acc, att]).astype(np.float64))
    with np.errstate(all="ignore"):
        return [float(v) for v in tot[:acc.size] / tot[acc.size:]]


def _jl(v) -> str:
    """Render like Julia's string interpolation of Float64 / Vector{Float64} ("$(x)")."""
    if isinstance(v, (list, tuple, np.ndarray)):
        return "[" + ", ".join(_jl(x) for x in v) + "]"
    if isinstance(v, (float, np.floating)):
        if math.isnan(v):
            return "NaN"
        if math.isinf(v):
            return "Inf" if v > 0 else "-Inf"
        v = float(v)
        r = repr(v)
        if "e" not in r and v != 0.0 and abs(v) >= 1e6:
            # Python keeps fixed notation up to 1e16, Julia (Ryu shortest, Base.show) switches at 1e6: "1.0e6"
            digits = r.replace("-", "").replace(".", "").lstrip("0")
            digits = digits.rstrip("0") or "0"
            ex = len(r.replace("-", "").split(".")[0]) - 1
            m = digits[0] + "." + (digits[1:] or "0")
            return ("-" if v < 0 else "") + f"{m}e{ex}"
        if "e" in r:                                   # Python "1e-05" / "1.5e+16" -> Julia "1.0e-5" / "1.5e16"
            m, ex = r.split("e")
            if "." not in m:
                m += ".0"
            return f"{m}e{int(ex)}"
        return r
    return str(v)


class StoreCallbacks(AriannaAlgorithm):
    """StoreCallbacks(chains; path, callbacks, store_first=true, store_last=false) (algorithms.jl:62-109):
    `<name>.dat` per callback (name = function name minus "callback_"), one line "$t $(callback(sim))" per call.
    Only rank 0 writes."""

    def __init__(self, chains, *, path=None, callbacks=None, store_first: bool = True, store_last: bool = False,
                 **extras):
        self.callbacks = tuple(callbacks or ())
        self.paths = [os.path.join(path, cb.__name__.replace("callback_", "") + ".dat") for cb in self.callbacks]
        self.files = []
        self.store_first, self.store_last = store_first, store_last
        self.records = {cb.__name__: [] for cb in self.callbacks}
        self._write = getattr(chains, "rank", 0) == 0
        if self._write:
            os.makedirs(path, exist_ok=True)

    def initialise(self, simulation):
        self.files = [open(p, "w") for p in self.paths] if self._write else []
        if self.store_first:
            self.make_step(simulation)

    def make_step(self, simulation):
        for i, cb in enumerate(self.callbacks):
            v = cb(simulation)
            self.records[cb.__name__].append((simulation.t, v))
            if self._write:
                self.files[i].write(f"{simulation.t} {_jl(v)}\n")
                self.files[i].flush()

    def finalise(self, simulation):
        if self.store_last:
            self.make_step(simulation)
        for f in self.files:
            f.close()


class DAT:
    extension = ".dat"


class TXT:
    extension = ".txt"


class StoreTrajectories(AriannaAlgorithm):
    """StoreTrajectories(chains; path, fmt=DAT(), store_first=true, store_last=false) (algorithms.jl:154-210).

    The reference writes one text file per chain ("$t $(x)" per line, particle_1d.jl:63-66), which cannot scale
    to 2^26 chains.  Here every rank appends (t, x[n_local]) frames to ONE binary file
    `trajectories/rank<r>.bin` (int64 t, then n_local float64).  A frame leaves the GPU through
    arianna_get_state_async -- a device-side snapshot drained into one of two page-locked host buffers on the copy
    stream -- and is written to disk at the NEXT store (or in finalise), i.e. while the following sweep already runs.
    For ensembles of at most `text_limit` chains the reference's per-chain text layout
    `trajectories/<c>/trajectory.dat` is ALSO produced so reference post-processing scripts keep working."""

    def __init__(self, chains, *, path=None, fmt=None, store_first: bool = True, store_last: bool = False,
                 text_limit: int = 4096, **extras):
        self.fmt = fmt or DAT()
        self.store_first, self.store_last = store_first, store_last
        self.dir = os.path.join(path, "trajectories")
        os.makedirs(self.dir, exist_ok=True)
        self.text = len(chains) <= text_limit
        self.bin_path = os.path.join(self.dir, f"rank{chains.rank}.bin")
        self.offset, self.n_local = chains.offset, chains.n_local
        self.text_paths = []
        if self.text:
            for c in range(self.offset + 1, self.offset + self.n_local + 1):  # 1-based chain ids like the reference
                d = os.path.join(self.dir, str(c))
                os.makedirs(d, exist_ok=True)
                self.text_paths.append(os.path.join(d, "trajectory" + self.fmt.extension))
        self.frames = 0
        self._bufs, self._pending, self._cur = None, None, 0

    def initialise(self, simulation):
        self.bin = open(self.bin_path, "wb")
        self.text_files = [open(p, "w") for p in self.text_paths]
        if self.store_first:
            self.make_step(simulation)

    def _write(self, t, x):
        self.bin.write(np.int64(t).tobytes())
        self.bin.write(x.tobytes())
        self.frames += 1
        for f, v in zip(self.text_files, x):
            f.write(f"{t} {_jl(float(v))}\n")                   # store_trajectory, particle_1d.jl:63-66
            f.flush()

    def _drain(self, engine):
        if self._pending is not None:
            t, i = self._pending
            engine.copy_wait()                                   # that frame only, not the sweep queued after it
            self._write(t, self._bufs[i].numpy())
            self._pending = None

    def make_step(self, simulation):
        ch = simulation.chains
        eng = ch.engine
        if not hasattr(eng, "get_state_async"):                  # test doubles: plain synchronous read
            self._write(simulation.t, ch.x)
            return
        ch.flush()                                               # launches the pending sweep (asynchronous) ...
        self._drain(eng)                                         # ... and writes the previous frame while it runs
        if self._bufs is None:
            import torch
            self._bufs = [torch.empty(self.n_local, dtype=torch.float64).pin_memory() for _ in range(2)]
        eng.get_state_async(self._bufs[self._cur].data_ptr())
        self._pending = (simulation.t, self._cur)
        self._cur ^= 1

    def finalise(self, simulation):
        if self.store_last:
            self.make_step(simulation)
        if self._pending is not None:
            self._drain(simulation.chains.engine)
        self.bin.close()
        for f in self.text_files:
            f.close()
        self._bufs = None

    @staticmethod
    def read_binary(path: str, n_local: int):
        """-> (t[frames], x[frames][n_local])"""
        rec = np.dtype([("t", "<i8"), ("x", "<f8", (n_local,))])
        a = np.fromfile(path, dtype=rec)
        return a["t"], a["x"]


class StoreLastFrames(AriannaAlgorithm):
    """StoreLastFrames (algorithms.jl:221-251): final state; binary `lastframe_rank<r>.bin` (+ per-chain text for
    small ensembles)."""

    def __init__(self, chains, *, path=None, fmt=None, text_limit: int = 4096, **extras):
        self.fmt = fmt or DAT()
        self.dir = os.path.join(path, "trajectories")
        os.makedirs(self.dir, exist_ok=True)
        self.text = len(chains) <= text_limit

    def finalise(self, simulation):
        ch = simulation.chains
        x = ch.x
        with open(os.path.join(self.dir, f"lastframe_rank{ch.rank}.bin"), "wb") as f:
            f.write(np.int64(simulation.t).tobytes())
            f.write(x.tobytes())
        if self.text:
            for i, v in enumerate(x):
                d = os.path.join(self.dir, str(ch.offset + i + 1))
                os.makedirs(d, exist_ok=True)
                with open(os.path.join(d, "lastframe" + self.fmt.extension), "w") as f:
                    f.write(f"{simulation.t} {_jl(float(v))}\n")


class StoreParameters(AriannaAlgorithm):
    """StoreParameters(chains; dependencies=(Metropolis,), ids, store_first=true) (metropolis.jl:380-450):
    `parameters/<k>/parameters.dat`, lines "$t $(collect(parameters))"."""

    def __init__(self, chains, *, dependencies=None, path=None, ids=None, store_first: bool = True,
                 store_last: bool = False, **extras):
        assert dependencies is not None and len(dependencies) == 1
        assert isinstance(dependencies[0], Metropolis)
        pool = dependencies[0].pool
        self.ids = list(range(1, len(pool) + 1)) if ids is None else list(ids)  # 1-based like the reference
        self.parameters_list = [pool[k - 1].parameters for k in self.ids]
        self.store_first, self.store_last = store_first, store_last
        self._write = getattr(chains, "rank", 0) == 0
        self.paths = []
        for k in self.ids:
            d = os.path.join(path, "parameters", str(k))
            if self._write:
                os.makedirs(d, exist_ok=True)
            self.paths.append(os.path.join(d, "parameters.dat"))
        self.files = []

    def initialise(self, simulation):
        self.files = [open(p, "w") for p in self.paths] if self._write else []
        if self.store_first:
            self.make_step(simulation)

    def make_step(self, simulation):
        simulation.chains.pull_params()                          # no-op unless the optimiser runs on the device
        for f, p in zip(self.files, self.parameters_list):
            f.write(f"{simulation.t} {_jl(list(p.data))}\n")
            f.flush()

    def finalise(self, simulation):
        if self.store_last:
            self.make_step(simulation)
        for f in self.files:
            f.close()


class PrintTimeSteps(AriannaAlgorithm):
    """Progress line (algorithms.jl:310-323); cosmetic."""

    def __init__(self, chains, **extras):
        self.rank = getattr(chains, "rank", 0)

    def make_step(self, simulation):
        if self.rank == 0 and simulation.verbose:
            print(f"\rProgress: {100.0 * simulation.t / simulation.steps:.0f}% t = {simulation.t}", end="")


# ---------------------------------------------------------------------------------------------------------
# Simulation / run!  (src/simulation.jl)
# ---------------------------------------------------------------------------------------------------------
class Simulation:
    """Simulation(chains, algorithm_list, steps; path="data", verbose=false) (simulation.jl:16-88)."""

    def __init__(self, chains, algorithm_list, steps: int, *, path: str = "data", verbose: bool = False):
        if not isinstance(chains, ParticleEnsemble):
            chains = ParticleEnsemble(chains)
        self.chains, self.steps, self.t = chains, int(steps), 0
        self.path, self.verbose = path, verbose
        algorithms, schedulers, names = [], [], []
        for constructor in algorithm_list:                                   # :72-84
            names.append(constructor["algorithm"])
            scheduler = constructor.get("scheduler", range(1, self.steps + 1))
            kwargs = {k: v for k, v in constructor.items() if k not in ("algorithm", "scheduler", "dependencies")}
            if "dependencies" in constructor:
                # dependencies are resolved by constructor identity among the algorithms already built (:78-80)
                parents = [a for a, n in zip(algorithms, names) if n in constructor["dependencies"]]
                kwargs["dependencies"] = parents
            kwargs.update(path=path, steps=self.steps, verbose=verbose)
            algorithms.append(constructor["algorithm"](chains, **kwargs))
            schedulers.append(list(scheduler))
        assert len(schedulers) == len(algorithms)                            # :45
        for s in schedulers:
            assert all(0 <= x <= self.steps for x in s), "scheduler entries must lie in 0..steps"      # :46
            assert all(a <= b for a, b in zip(s, s[1:])), "schedulers must be sorted"                  # :47
        self.algorithms, self.schedulers = tuple(algorithms), tuple(schedulers)
        # counters[k] = findfirst(x -> x > 0, scheduler) (:49); None mirrors Julia's `nothing`
        self.counters = [next((i for i, x in enumerate(s) if x > 0), None) for s in self.schedulers]
        if chains.rank == 0:
            os.makedirs(path, exist_ok=True)

    def write_summary(self):
        if self.chains.rank != 0:
            return
        with open(os.path.join(self.path, "summary.log"), "w") as f:          # :124-143
            f.write("SIMULATION SUMMARY\n\nSimulation:\n")
            f.write(f"\tSteps: {self.steps}\n\tNumber of chains: {len(self.chains)}\n")
            f.write(f"\tNumber of algorithms: {len(self.algorithms)}\n\tVerbose: {str(self.verbose).lower()}\n")
            f.write(f"\tStarted on {time.strftime('%Y-%m-%dT%H:%M:%S')}\n\nSystem:\n\tParticleEnsemble (CUDA)\n\n")
            f.write("Algorithms:\n")
            for a, s in zip(self.algorithms, self.schedulers):
                a.write_algorithm(f, s)
            f.write("\n")


def _make_lookahead(sim: "Simulation"):
    """Look-ahead over callback-only stores.  The schedule is known up front (sim.schedulers), so when StoreCallbacks
    fires at time t the ensemble can run every following store interval up to the next event that observes or
    changes the chains in any other way (trajectory frames, the PGMC estimator/update, parameter stores, ...) as ONE
    arianna_sweep_series call.  Returns a function () -> [K_1, K_2, ...] (MC steps between the coming callback-only
    store times, as of sim.t), or None when the algorithm list does not allow it."""
    import bisect
    algs = sim.algorithms
    met = [k for k, a in enumerate(algs) if isinstance(a, Metropolis)]
    cbs = [k for k, a in enumerate(algs) if isinstance(a, StoreCallbacks)
           and all(cb in (callback_energy, callback_acceptance) for cb in a.callbacks)]
    if len(met) != 1 or not cbs or min(cbs) < met[0]:
        return None                      # callbacks listed before Metropolis see the state BEFORE the step at t
    m = met[0]
    passive = (Metropolis, PrintTimeSteps)

    def is_passive(a):     # never looks at the chains during the t-loop (e.g. StoreLastFrames only acts in finalise)
        return isinstance(a, passive) or type(a).make_step is AriannaAlgorithm.make_step

    # Barriers = times at which some other algorithm looks at (or changes) the chains.  One listed AFTER Metropolis sees
    # the state after the Metropolis step of its time tb (the stretch may include a store AT tb); one listed BEFORE
    # Metropolis sees the state before that step (simulation.jl:184-191 runs the list in order), so the stretch must
    # stop short of tb.
    def times(pred):
        return sorted({t for k, a in enumerate(algs) if k not in cbs and not is_passive(a) and pred(k)
                       for t in sim.schedulers[k]})
    barriers_post, barriers_pre = times(lambda k: k > m), times(lambda k: k < m)
    stores = sorted({t for k in cbs for t in sim.schedulers[k]})
    msched = sorted(sim.schedulers[m])
    step = algs[m].sweepstep
    chains = sim.chains

    def lookahead():
        t = sim.t
        ib = bisect.bisect_left(barriers_post, t)
        tb = barriers_post[ib] if ib < len(barriers_post) else sim.steps + 1    # first one at or after now
        ip = bisect.bisect_right(barriers_pre, t)                                # (those at t have already fired)
        tp = barriers_pre[ip] if ip < len(barriers_pre) else sim.steps + 2      # first one after now
        i0 = bisect.bisect_right(stores, t)
        out, prev = [], t
        for ts in stores[i0:i0 + chains.max_lookahead]:
            if ts > tb or ts >= tp:
                break
            out.append(step * (bisect.bisect_right(msched, ts) - bisect.bisect_right(msched, prev)))
            prev = ts
        # an algorithm with store_last fires once more in finalise(), at t = steps: the stretch must not pass the end
        return out

    return lookahead


def run(simulation: Simulation):
    """run!(simulation) (simulation.jl:175-204): initialise all, t-loop in list order, finalise in `finally`."""
    sim = simulation
    sim.chains._lookahead = _make_lookahead(sim) if getattr(sim, "lookahead", True) else None
    try:
        for a in sim.algorithms:
            a.initialise(sim)
        sim.write_summary()
        t0 = time.perf_counter()
        scheds, counters, algs = sim.schedulers, sim.counters, sim.algorithms
        for t in range(1, sim.steps + 1):
            sim.t = t
            for k in range(len(algs)):
                # Julia indexes scheduler[counter] and would throw past the end; build_schedule always appends
                # `steps`, so a counter past the end means "never again"
                ck = counters[k]
                if ck is not None and ck < len(scheds[k]) and t == scheds[k][ck]:
                    algs[k].make_step(sim)
                    counters[k] = ck + 1
        sim.chains.flush()
        sim.chains.engine.synchronize()
        sim.chains.pull_params()
        sim.sim_time = time.perf_counter() - t0
        if sim.chains.rank == 0:
            with open(os.path.join(sim.path, "summary.log"), "a") as f:
                f.write(f"Report:\n\tSimulation time: {sim.sim_time} s\n")
    finally:
        for a in sim.algorithms:
            a.finalise(sim)
        _finalise_summary(sim)
    return None


def _finalise_summary(sim: "Simulation"):
    """finalise_summary (simulation.jl:153-165): size of everything under `path` and the completion stamp."""
    if sim.chains.rank != 0 or not os.path.exists(os.path.join(sim.path, "summary.log")):
        return
    total = 0
    for root, _, files in os.walk(sim.path):
        for name in files:
            total += os.path.getsize(os.path.join(root, name))
    with open(os.path.join(sim.path, "summary.log"), "a") as f:
        f.write(f"\tSimulation size: {_jl(total / 1024 ** 2)} MB\n")
        f.write(f"\tStatus: Completed on {time.strftime('%Y-%m-%dT%H:%M:%S')}\n")
