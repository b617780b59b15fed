"""GPU tests of replica exchange (parallel tempering) across per-chain β ladders: parity with the CPU oracle, shard
invariance and argument errors, the physics it exists for (harmonic ladder averages and swap rates, double-well
barrier crossing) and the host mirror's ReplicaExchange / ladder callbacks."""
import math
import os

import numpy as np
import pytest

import montecarlo_b200 as mb
from montecarlo_b200 import _lib as L_
from oracle import oracle as O

import exchange_oracle as XO

pytestmark = pytest.mark.gpu

POTS = {"harmonic": O.POT_HARMONIC, "quartic": O.POT_QUARTIC, "double_well": O.POT_DOUBLE_WELL}
SCHEDULE = [7, 10, 3, 8, 5, 12, 1, 6, 9, 4] * 2          # K between the 20 exchange rounds: odd and even, both parities


def _ladder(rng, L):
    return rng.uniform(0.25, 8.0, L)


@pytest.mark.parametrize("M,L,pot,sigma,weight", [
    (1 << 16, 8, "harmonic", [0.3], [1.0]),
    (5 << 13, 5, "double_well", [0.3, 0.05], [0.5, 0.5]),
    (6 << 12, 6, "quartic", [0.3], [1.0]),
    (1 << 14, 2, "double_well", [0.4], [1.0]),                          # one rung pair
    (120 << 8, 256, "harmonic", [0.3, 0.1, 0.05], [0.5, 0.25, 0.25]),   # kMaxLadder rungs: 255 swap counters
])
def test_parity_with_the_oracle(M, L, pot, sigma, weight):
    """EXACT: the device replays the native stream's draws (draws_philox) and runs its own exchange rounds; the oracle
    does the same on the CPU.  Positions bit-identical, Move and swap counters identical, ladder records to 1e-12.
    FAST: native sweeps against the same oracle, counters identical and |Δx| < 1e-12 (the native-Philox bar)."""
    rng = np.random.default_rng(M + L)
    seed, ladder = 17, _ladder(rng, L)
    betas = np.tile(ladder, M // L)
    x0 = O.init_synthetic(seed, 0, M)
    ref = O.Ensemble(x0, 1.0, sigma, weight, potential=POTS[pot])
    multi = len(sigma) > 1
    xacc = np.zeros(L - 1, np.int64)
    draws, done = [], 0
    for R, K in enumerate(SCHEDULE):
        uc, z, ua = O.draws_philox(seed, 0, M, done, K, with_cat=multi)
        draws.append((uc, z, ua))
        ref.sweep_replay(uc, z, ua, betas=betas)
        xacc += XO.exchange(ref, L, seed, R, 0, betas=betas)
        done += K
    assert 0 < xacc.sum() < (M // L) * (L - 1) * len(SCHEDULE) // 2
    assert 0.05 < ref.acc.sum() / ref.tot.sum() < 0.95                # a wrong potential or β would show
    if pot == "double_well":
        assert 0 < np.count_nonzero(ref.x < 0) < M
    ref_sums = XO.ladder_sums(ref, L)
    for arith in ("exact", "fast"):
        with mb.CudaEnsemble(M, 1.0, sigma, weight, seed=seed, potential=pot, arith=arith) as eng:
            eng.init_synthetic()
            eng.set_ladder(ladder)
            for (uc, z, ua), K in zip(draws, SCHEDULE):
                if arith == "exact":
                    eng.sweep_replay(uc if multi else None, z, ua)
                else:
                    eng.sweep(K)
                eng.replica_exchange()
            x = eng.get_state()
            acc, tot = eng.chain_counters()
            a, att, rounds = eng.exchange_counters()
            sums = eng.ladder_sums()
        if arith == "exact":
            assert np.array_equal(x, ref.x), float(np.max(np.abs(x - ref.x)))
        else:
            assert np.max(np.abs(x - ref.x)) < 1e-12
        assert np.array_equal(acc.astype(np.int64), ref.acc) and np.array_equal(tot.astype(np.int64), ref.tot)
        assert np.array_equal(a, xacc) and rounds == len(SCHEDULE)
        assert np.array_equal(att, [(M // L) * len(SCHEDULE) // 2] * (L - 1))
        np.testing.assert_allclose(sums, ref_sums, rtol=1e-12, equal_nan=True)


def test_shards_chunks_and_errors():
    M, L, seed = 3 * 1024 * 7, 7, 5
    ladder = np.geomspace(0.5, 6.0, L)

    def run(off, n, chunks):
        with mb.CudaEnsemble(n, 1.0, [0.4], seed=seed, chain_offset=off, n_chains_total=M) as eng:
            eng.init_synthetic()
            eng.set_ladder(ladder)
            for K in chunks:
                eng.sweep(K)
                eng.replica_exchange()
            return eng.get_state(), eng.exchange_counters()[0], eng.ladder_sums()

    x, a, s = run(0, M, [10] * 12)
    xa, aa, sa = run(0, 7 * 1000, [10] * 12)
    xb, ab, sb = run(7 * 1000, M - 7 * 1000, [10] * 12)
    assert np.array_equal(np.concatenate([xa, xb]), x)
    assert np.array_equal(aa + ab, a) and a.sum() > 0
    np.testing.assert_allclose(sa + sb, s, rtol=1e-12)
    with mb.CudaEnsemble(M, 1.0, [0.4], seed=seed) as eng:  # Metropolis chunking between rounds does not matter
        eng.init_synthetic()
        eng.set_ladder(ladder)
        for _ in range(12):
            eng.sweep(3)
            eng.sweep(7)
            eng.replica_exchange()
        assert np.array_equal(eng.get_state(), x)
        # another ladder shape resets the rounds and counters; the same shape keeps them
        eng.set_ladder(ladder * 2)
        assert eng.exchange_counters()[2] == 12
        eng.set_ladder(np.geomspace(0.5, 6.0, 3))
        a3, att3, r3 = eng.exchange_counters()
        assert r3 == 0 and not a3.any() and not att3.any()
        n0 = eng.launch_count
        eng.replica_exchange()
        eng.ladder_sums()
        assert eng.launch_count == n0 + 3                   # one exchange kernel, reduce + fold
    errors = []
    with mb.CudaEnsemble(M, 1.0, [0.4]) as eng:
        for fn in (eng.replica_exchange, eng.exchange_counters, eng.ladder_sums):   # before set_ladder
            with pytest.raises(mb.AriannaError) as e:
                fn()
            errors.append(e.value.code)
        for bad in (np.ones(1), np.ones(257), np.ones(5)):   # L < 2, L > 256, 5 does not divide M
            with pytest.raises(mb.AriannaError) as e:
                eng.set_ladder(bad)
            errors.append(e.value.code)
    with mb.CudaEnsemble(7 * 64, 1.0, [0.4], chain_offset=3, n_chains_total=7 * 65) as eng:   # misaligned offset
        with pytest.raises(mb.AriannaError) as e:
            eng.set_ladder(ladder)
        errors.append(e.value.code)
    assert errors == [L_.ERR_INVALID] * len(errors)
    for kw in (dict(dtype="f32"), dict(rng="xoshiro")):
        with mb.CudaEnsemble(7 * 64, 1.0, [0.4], **kw) as eng:
            codes = []
            for fn in (lambda: eng.set_ladder(ladder), eng.replica_exchange, eng.exchange_counters, eng.ladder_sums):
                with pytest.raises(mb.AriannaError) as e:
                    fn()
                codes.append(e.value.code)
            assert codes == [L_.ERR_UNSUPPORTED] * 4, kw


def _chi2_swap_rate(b0, b1, n=4_000_000, seed=0):
    """E[min(1, exp((b0 − b1)(E0 − E1)))] for E_i = x_i², x_i ~ N(0, 1/(2 b_i)) independent, with its MC error."""
    g = np.random.default_rng(seed)
    e0 = g.chisquare(1, n) / (2 * b0)
    e1 = g.chisquare(1, n) / (2 * b1)
    a = np.minimum(1.0, np.exp((b0 - b1) * (e0 - e1)))
    return a.mean(), a.std() / math.sqrt(n)


def test_harmonic_ladder_physics():
    M, L = 1 << 22, 16
    ladder = np.geomspace(0.5, 4.0, L)
    n_lad = M // L
    with mb.CudaEnsemble(M, 1.0, [0.5], seed=3) as eng:
        eng.init_synthetic()
        eng.set_ladder(ladder)
        for _ in range(300):
            eng.sweep(10)
            eng.replica_exchange()
        a0, _, R0 = eng.exchange_counters()
        assert R0 % 2 == 0
        eng.sweep(10)
        eng.replica_exchange()                             # one even round: pairs 0, 2, 4, ...
        eng.sweep(10)
        eng.replica_exchange()                             # one odd round: pairs 1, 3, 5, ...
        a1, _, _ = eng.exchange_counters()
        eng.sweep(10)
        x = eng.get_state().reshape(n_lad, L)
    for r in range(L):
        s2 = 1 / (2 * ladder[r])
        xr = x[:, r]
        assert abs(xr.mean()) < 3 * xr.std() / math.sqrt(n_lad), r
        er = xr * xr
        assert abs(er.mean() - s2) < 3 * er.std() / math.sqrt(n_lad), r
    rate = (a1 - a0) / n_lad
    for k in range(L - 1):
        p, mc_err = _chi2_swap_rate(ladder[k], ladder[k + 1], seed=k)
        sigma = math.sqrt(p * (1 - p) / n_lad + mc_err ** 2)
        assert abs(rate[k] - p) < 4 * sigma, (k, rate[k], p, sigma)


def test_double_well_barrier_crossing():
    """What parallel tempering is for: at β = 16 a chain started in the right well of (x² − 1)² stays there (the barrier
    costs e^-16 per crossing; at β = 12, 6 % of the chains had crossed after these 20000 steps on a B200); with a
    ladder up to β = 0.25 and one exchange round every 10 steps the coldest rung samples both wells equally."""
    M, L, steps, every = 1 << 20, 16, 20000, 10
    ladder = np.geomspace(0.25, 16.0, L)[::-1].copy()       # rung 0 is the coldest
    fractions = {}
    for exchange in (False, True):
        with mb.CudaEnsemble(M, 1.0, [0.3], seed=11, potential="double_well") as eng:
            eng.set_state(np.ones(M))
            eng.set_ladder(ladder)
            for _ in range(steps // every):
                eng.sweep(every)
                if exchange:
                    eng.replica_exchange()
            x = eng.get_state().reshape(M // L, L)
        fractions[exchange] = float((x[:, 0] < 0).mean())
    print(f"cold-rung fraction at x < 0: without exchange {fractions[False]:.5f}, with exchange {fractions[True]:.5f}")
    assert fractions[False] < 0.01
    assert abs(fractions[True] - 0.5) < 0.03


def _mirror_run(path, M, L, steps, seed, lookahead):
    chains = mb.ParticleEnsemble(n_chains=M, beta=1.0, potential="double_well")
    pool = (mb.Move(mb.Displacement(0.0), mb.StandardGaussian(), mb.ComponentArray(σ=0.3), 1.0),)
    sim = mb.Simulation(chains, (
        dict(algorithm=mb.Metropolis, pool=pool, seed=seed),
        dict(algorithm=mb.ReplicaExchange, dependencies=(mb.Metropolis,), ladder=list(np.geomspace(0.5, 8.0, L)),
             scheduler=list(range(50, steps + 1, 50))),
        dict(algorithm=mb.StoreCallbacks, callbacks=(mb.callback_energy, mb.callback_acceptance),
             scheduler=list(range(0, steps + 1, 10))),
        dict(algorithm=mb.StoreCallbacks, callbacks=(mb.callback_ladder_energy, mb.callback_ladder_acceptance,
                                                     mb.callback_exchange_acceptance),
             scheduler=list(range(0, steps + 1, 100))),
    ), steps, path=str(path))
    sim.lookahead = lookahead
    mb.run(sim)
    return chains


def test_through_the_mirror(tmp_path):
    M, L, steps, seed = 1 << 16, 8, 1000, 7
    ladder = list(np.geomspace(0.5, 8.0, L))
    chains = _mirror_run(tmp_path, M, L, steps, seed, True)
    plain = _mirror_run(tmp_path / "plain", M, L, steps, seed, False)
    assert np.array_equal(plain.x, chains.x)
    # every 50-step stretch between exchange rounds runs its 5 callback-only stores as ONE series call
    assert chains.engine.launch_count <= plain.engine.launch_count - 3 * (steps // 50), \
        (chains.engine.launch_count, plain.engine.launch_count)
    # the same schedule as direct engine calls
    rows = {k: [] for k in ("energy", "acceptance", "ladder_energy", "ladder_acceptance", "exchange_acceptance")}
    with mb.CudaEnsemble(M, 1.0, [0.3], seed=seed, potential="double_well") as eng:
        eng.init_synthetic()
        eng.set_ladder(ladder)
        pending = 0
        for t in range(0, steps + 1):
            pending += 1 if t else 0
            if t % 10 == 0:
                eng.sweep(pending)
                pending = 0
                if t and t % 50 == 0:
                    eng.replica_exchange()
                e, a = eng.callbacks()
                rows["energy"].append(f"{t} {mb.arianna._jl(float(e))}")
                rows["acceptance"].append(f"{t} {mb.arianna._jl([float(v) for v in a])}")
                if t % 100 == 0:
                    s = eng.ladder_sums()
                    xa, xt, _ = eng.exchange_counters()
                    rows["ladder_energy"].append(f"{t} {mb.arianna._jl([float(v) for v in s[:, 0] / s[:, -1]])}")
                    rows["ladder_acceptance"].append(
                        f"{t} {mb.arianna._jl([[float(v) for v in r[1:-1] / r[-1]] for r in s])}")
                    with np.errstate(all="ignore"):
                        rows["exchange_acceptance"].append(f"{t} {mb.arianna._jl([float(v) for v in xa / xt])}")
        assert np.array_equal(eng.get_state(), chains.x)
    for name, want in rows.items():
        got = open(tmp_path / f"{name}.dat").read().split("\n")[:-1]
        assert len(got) == len(want), name
        for g, w in zip(got, want):
            tg, vg = g.split(" ", 1)
            tw, vw = w.split(" ", 1)
            assert tg == tw, name
            if name in ("energy", "acceptance"):      # series records vs per-store reductions: summation order only
                fg = np.array(eval(vg.replace("NaN", "float('nan')")), dtype=float)
                fw = np.array(eval(vw.replace("NaN", "float('nan')")), dtype=float)
                np.testing.assert_allclose(fg, fw, rtol=1e-12, equal_nan=True, err_msg=f"{name} {tg}")
            else:
                assert vg == vw, (name, tg)
    assert rows["exchange_acceptance"][0] == f"0 {mb.arianna._jl([float('nan')] * (L - 1))}"


_NCCL_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch, torch.distributed as dist
rank = int(os.environ["RANK"]); torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
import montecarlo_b200 as mb
M, steps = 16 * 4096, 400
chains = mb.ParticleEnsemble(n_chains=M, beta=1.0, potential="double_well")
pool = (mb.Move(mb.Displacement(0.0), mb.StandardGaussian(), mb.ComponentArray(σ=0.3), 1.0),)
sim = mb.Simulation(chains, (dict(algorithm=mb.Metropolis, pool=pool, seed=7),
                             dict(algorithm=mb.ReplicaExchange, dependencies=(mb.Metropolis,),
                                  ladder=list(np.geomspace(0.25, 12.0, 16)), scheduler=list(range(10, steps + 1, 10))),
                             dict(algorithm=mb.StoreCallbacks, callbacks=(mb.callback_ladder_energy,
                                  mb.callback_exchange_acceptance), scheduler=list(range(0, steps + 1, 50)))),
                    steps, path={path!r})
mb.run(sim)
np.save(os.path.join({path!r}, f"x_rank{{rank}}.npy"), chains.x)
dist.barrier(); dist.destroy_process_group()
"""


def test_two_gpu_exchange_matches_one_gpu(tmp_path):
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    outs = {}
    for n in (1, 2):
        d = tmp_path / f"n{n}"
        d.mkdir()
        script = d / "worker.py"
        script.write_text(_NCCL_WORKER.format(root=root, path=str(d)))
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                            "--master-addr", "127.0.0.1", "--master-port", str(29700 + n), str(script)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        outs[n] = (np.concatenate([np.load(d / f"x_rank{k}.npy") for k in range(n)]),
                   open(d / "ladder_energy.dat").read(), open(d / "exchange_acceptance.dat").read())
    assert np.array_equal(outs[2][0], outs[1][0])
    assert outs[2][2] == outs[1][2]                           # integer counters: exact
    e1 = [np.array(eval(r.split(" ", 1)[1])) for r in outs[1][1].split("\n")[:-1]]
    e2 = [np.array(eval(r.split(" ", 1)[1])) for r in outs[2][1].split("\n")[:-1]]
    np.testing.assert_allclose(e2, e1, rtol=1e-12)
