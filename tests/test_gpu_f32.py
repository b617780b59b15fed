"""Float32 ensembles (SURVEY.md §8 f3): Particle{Float32}, Displacement{Float32}, ComponentArray(σ = 0.1f0) -- the
Float32 instantiation of the reference's generic code (particle_1d.jl:9-16, metropolis.jl:176), with Julia's promotion
rules deciding the precision of every operation (oracle/arianna_oracle.c:mc_step_exact_f32).

Bars: replay -> decisions and Float32 positions bit-identical to the oracle; native stream -> 3σ agreement with the
analytic harmonic averages (the north star's two proofs), chunk / shard invariance bit for bit, loose agreement with the
oracle's libm restatement of the stream."""
import math

import numpy as np
import pytest

import montecarlo_b200 as mb
from oracle import oracle as O

pytestmark = pytest.mark.gpu
POTS = {"harmonic": O.POT_HARMONIC, "quartic": O.POT_QUARTIC, "double_well": O.POT_DOUBLE_WELL}


@pytest.mark.parametrize("pot", ["harmonic", "quartic", "double_well"])
def test_f32_replay_bit_exact(pot):
    M, K, beta, sigma = 10007, 67, 2.0, 0.1
    x0 = O.init_synthetic(11, 0, M)
    gen = O.Ensemble(x0, beta, [sigma])
    gen.seed_xoshiro(42)
    _, z, ua = gen.draws_xoshiro(K)                                  # Float64 draws; randn(rng, Float32) rounds z inside
    ref = O.Ensemble32(x0, beta, sigma, potential=POTS[pot])
    dref = ref.sweep_replay(z, ua, want_decisions=True)
    with mb.CudaEnsemble(M, beta, [sigma], potential=pot, arith="exact", dtype="f32") as eng:
        eng.set_state(x0)                                            # Float64 view: rounded to Float32
        assert np.array_equal(eng.get_state_f32(), x0.astype(np.float32))
        dec = eng.sweep_replay(None, z, ua, want_decisions=True)
        x, e = eng.get_state_f32(with_energy=True)
        assert np.array_equal(dec, dref)
        assert x.dtype == np.float32 and np.array_equal(x, ref.x) and np.array_equal(e, ref.e)
        assert np.array_equal(eng.chain_counters()[0][0].astype(np.int64), ref.acc)
        xd, ed = eng.get_state(with_energy=True)                     # the Float64 view widens exactly
        assert np.array_equal(xd, ref.x.astype(np.float64)) and np.array_equal(ed, ref.e.astype(np.float64))
        me, ma = eng.callbacks()
        assert abs(me / np.mean(ref.e.astype(np.float64)) - 1) < 1e-12   # Σe is accumulated in Float64 on the device ...
        assert abs(me / ref.callback_energy() - 1) < 1e-4                # ... the reference's Float32 mean loses digits
        assert abs(ma[0] / ref.callback_acceptance() - 1) < 1e-12


def test_f32_replay_per_chain_beta_and_set_state_f32():
    M, K = 4099, 40
    x0 = O.init_synthetic(5, 0, M).astype(np.float32)
    betas = np.linspace(0.5, 4.0, M).astype(np.float32)
    gen = O.Ensemble(x0, 2.0, [0.3])
    gen.seed_xoshiro(7)
    _, z, ua = gen.draws_xoshiro(K)
    ref = O.Ensemble32(x0, 2.0, 0.3)
    dref = ref.sweep_replay(z, ua, want_decisions=True, betas=betas)
    with mb.CudaEnsemble(M, 2.0, [0.3], arith="exact", dtype="f32") as eng:
        eng.set_state_f32(x0)
        eng.set_betas(betas.astype(np.float64))
        d1 = eng.sweep_replay(None, z[:13], ua[:13], want_decisions=True)
        d2 = eng.sweep_replay(None, z[13:], ua[13:], want_decisions=True)
        assert np.array_equal(np.concatenate([d1, d2]), dref) and np.array_equal(eng.get_state_f32(), ref.x)


@pytest.mark.parametrize("arith", ["fast", "exact"])
def test_f32_native_distribution_and_invariance(arith):
    """distribution_test.jl:31-37 for Float32 chains: ⟨x⟩ = 0, std x = 1/√(2β), ⟨E⟩ = 1/(2β) within 3σ (+ the Float32
    resolution of x), acceptance = (2/π)·atan(2s/σ); launch chunking and sharding change nothing, bit for bit."""
    M, beta, sigma, seed = 1 << 20, 2.0, 0.3, 42
    s = 1 / math.sqrt(2 * beta)
    with mb.CudaEnsemble(M, beta, [sigma], seed=seed, arith=arith, dtype="f32") as eng:
        eng.init_synthetic()
        assert np.array_equal(eng.get_state_f32(), O.init_synthetic(seed, 0, M).astype(np.float32))
        eng.sweep(1000)
        a0 = eng.chain_counters()[0][0].astype(np.int64).sum()
        eng.sweep(201, reduce=True)
        me, ma = eng.callbacks()
        x = eng.get_state_f32().astype(np.float64)
        a1 = eng.chain_counters()[0][0].astype(np.int64).sum()
        assert abs(x.mean()) < 3 * s / math.sqrt(M) and abs(x.std() - s) < 3 * s / math.sqrt(2 * M)
        assert abs(me - 1 / (2 * beta)) < 3 * math.sqrt(1 / (2 * beta ** 2) / M) + 1e-6
        assert abs(me - np.mean(x * x)) < 1e-6
        assert abs((a1 - a0) / (201 * M) - 2 / math.pi * math.atan(2 * s / sigma)) < 3 * 0.5 / math.sqrt(201 * M) * 6
        assert abs(ma[0] - a1 / (1201 * M)) < 1e-12

    def run(chunks, off=0, n=5000):
        with mb.CudaEnsemble(n, beta, [sigma], seed=3, chain_offset=off, arith=arith, dtype="f32") as e2:
            e2.init_synthetic()
            for k in chunks:
                e2.sweep(k, reduce=(k % 2 == 0))
            return e2.get_state_f32(), e2.chain_counters()[0][0]

    xr, ar = run([20])
    for chunks in ([7, 12, 1], [1] * 20, [3, 17]):
        xx, aa = run(chunks)
        assert np.array_equal(xx, xr) and np.array_equal(aa, ar), chunks
    xa, aa = run([20], 0, 1234)
    xb, ab = run([20], 1234, 5000 - 1234)
    assert np.array_equal(np.concatenate([xa, xb]), xr) and np.array_equal(np.concatenate([aa, ab]), ar)


def test_f32_native_follows_the_oracle_restatement():
    """The native Float32 stream (one Philox block per pair: MUFU Box-Muller + two 32-bit accept uniforms) against the
    oracle's libm restatement of the same words: normals agree to ~1e-6, so nearly every decision and every position
    agrees -- a loose anchor; the parity bar of native mode is statistical.  Every potential, both arithmetics."""
    M, K, seed, off = 20000, 50, 42, 777
    x0 = O.init_synthetic(seed, off, M)
    z, ua = O.draws_philox_f32(seed, off, M, 0, K)
    for pot in POTS:
        ref = O.Ensemble32(x0, 2.0, 0.1, potential=POTS[pot])
        ref.sweep_replay(z, ua)
        assert 0.05 < ref.acc.sum() / (K * M) < 0.95
        for arith in ("exact", "fast"):
            with mb.CudaEnsemble(M, 2.0, [0.1], seed=seed, chain_offset=off, potential=pot, arith=arith,
                                 dtype="f32") as eng:
                eng.init_synthetic()
                eng.sweep(K)
                x = eng.get_state_f32()
                acc = eng.chain_counters()[0][0].astype(np.int64)
            assert np.mean(acc == ref.acc) > 0.999, (pot, arith)
            same = acc == ref.acc
            assert np.max(np.abs(x[same].astype(np.float64) - ref.x[same])) < 1e-4, (pot, arith)


def test_f32_unsupported_paths_fail_loudly():
    with mb.CudaEnsemble(1000, 2.0, [0.1], dtype="f32") as eng:
        for call in (lambda: eng.sweep_series([10]), lambda: eng.run_host_job([10]), lambda: eng.pgmc_estimate(2, [0])):
            with pytest.raises(mb.AriannaError) as ei:
                call()
            assert ei.value.code == 4                                   # ARIANNA_ERR_UNSUPPORTED
    with pytest.raises(mb.AriannaError):
        mb.CudaEnsemble(1000, 2.0, [0.1, 0.2], [0.5, 0.5], dtype="f32")
    with pytest.raises(mb.AriannaError):
        mb.CudaEnsemble(1000, 2.0, [0.1], rng="xoshiro", dtype="f32")
    with mb.CudaEnsemble(1000, 2.0, [0.1]) as eng:
        with pytest.raises(mb.AriannaError):
            eng.get_state_f32()


def test_f32_through_the_driver_mirror(tmp_path):
    """Particle{Float32} chains through Simulation / run!: StoreCallbacks every 10 steps (one fused launch per store;
    the series fusion is a Float64 path) and a trajectory frame in Float32."""
    M, steps, burn = 1 << 16, 600, 300
    chains = mb.ParticleEnsemble(n_chains=M, beta=2.0, dtype="f32")
    pool = (mb.Move(mb.Displacement(0.0), mb.StandardGaussian(), mb.ComponentArray(σ=0.3), 1.0),)
    st = mb.build_schedule(steps, burn, 10)
    sim = mb.Simulation(chains, (dict(algorithm=mb.Metropolis, pool=pool, seed=42),
                                 dict(algorithm=mb.StoreCallbacks, callbacks=(mb.callback_energy, mb.callback_acceptance),
                                      scheduler=st)), steps, path=str(tmp_path))
    mb.run(sim)
    en = np.loadtxt(tmp_path / "energy.dat")[1:, 1]
    assert abs(en.mean() - 0.25) < 3 * math.sqrt(1 / 8 / M)
    assert chains.x.dtype == np.float32 and chains.engine.launch_count <= len(st) + 3
