"""CPU tests of replica exchange (parallel tempering): the C reference (exchange_oracle.c) against its numpy
restatement, the exact even/odd pairing, and the host mirror (ReplicaExchange, the ladder callbacks, look-ahead
barriers, sharding) over an oracle-backed test double."""
import os
import subprocess
import sys

import numpy as np
import pytest

import montecarlo_b200 as mb
from montecarlo_b200 import arianna as A
from oracle import oracle as O

import exchange_oracle as XO
from fake_engine import OracleEngine

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _states(rng, M, pot):
    x = rng.uniform(-2.0, 2.0, M)
    x[rng.choice(M, 3, replace=False)] = [np.inf, -np.inf, np.nan]      # NaN / inf energies must reject, not crash
    return x


@pytest.mark.parametrize("L", [2, 5, 8])
@pytest.mark.parametrize("pot", [O.POT_HARMONIC, O.POT_QUARTIC, O.POT_DOUBLE_WELL])
def test_c_oracle_equals_numpy_restatement(L, pot):
    rng = np.random.default_rng(L * 10 + pot)
    M, seed, off = 40 * L, 123, 7 * L
    betas = np.tile(rng.uniform(0.25, 8.0, L), M // L)
    x0 = _states(rng, M, pot)
    ens = O.Ensemble(x0, 1.0, [0.1], potential=pot)
    xn = x0.copy()
    acc_c, acc_n = np.zeros(L - 1, np.int64), np.zeros(L - 1, np.int64)
    for R in range(50):
        acc_c += XO.exchange(ens, L, seed, R, off, betas=betas)
        acc_n += XO.exchange_round_np(xn, betas, L, seed, off, R, pot)
        assert np.array_equal(ens.x, xn, equal_nan=True), R
    assert np.array_equal(acc_c, acc_n) and acc_c.sum() > 0
    assert np.array_equal(ens.e, ens._potential(ens.x), equal_nan=True)          # e travels with x
    # a chain whose energy is NaN never swaps: NaN stays where it started
    assert np.isnan(ens.x[np.isnan(x0)]).all()


def test_tag4_draw_is_the_documented_philox_block():
    """u of the pair with lower chain g in round R: word A of Philox4x32-10 with key (4, 'ARIA') and counter
    (sid_lo, R_lo, sid_hi, R_hi << 8), sid = seed + g: with u below every acceptance the pair swaps iff α > u."""
    seed, R, g = 2 ** 33 + 5, 3, 1     # sid above 2^32: both halves of the counter are exercised
    sid = seed + g
    o = O.philox4x32_10([sid & 0xFFFFFFFF, R, sid >> 32, 0], [4, 0x41524941])
    u = float((int(o[0]) | int(o[1]) << 32) >> 11) * 2.0 ** -53
    assert XO.exchange_uniform(sid, R) == u            # the reference's own Philox agrees with the oracle's
    L = 4
    # rungs 1 and 2 (round 3 is odd) at Δ = (β1 − β2)(e1 − e2) = log(α): α just above / below u
    for a, swap in ((u * (1 + 1e-12), True), (u * (1 - 1e-12), False)):
        x = np.array([0.0, 1.0, 0.0, 0.0])                  # e1 − e2 = 1
        betas = np.array([0.0, np.log(a), 0.0, 0.0])         # Δ = (β1 − β2)·1 = log(α)
        ens = O.Ensemble(x, 1.0, [0.1])
        acc = XO.exchange(ens, L, seed, R, 0, betas=betas)
        assert acc[1] == int(swap) and (ens.x[1] == 0.0) == swap
        xn = x.copy()
        assert XO.exchange_round_np(xn, betas, L, seed, 0, R, 0)[1] == int(swap)


@pytest.mark.parametrize("L", [2, 5, 8])
def test_equal_betas_swap_every_active_pair(L):
    """Δ = 0 ⇒ α = 1 > u: every pair of the round swaps, so positions are permuted exactly by the even/odd pairing."""
    M = 6 * L
    x = np.arange(M, dtype=np.float64)
    ens = O.Ensemble(x, 2.0, [0.1])
    ref = x.copy()
    for R in range(7):
        acc = XO.exchange(ens, L, 9, R, 0)
        for b in range(0, M, L):
            for r in range(R & 1, L - 1, 2):
                ref[b + r], ref[b + r + 1] = ref[b + r + 1], ref[b + r]
        assert np.array_equal(ens.x, ref)
        assert np.array_equal(acc, [(M // L) if (k - R) % 2 == 0 else 0 for k in range(L - 1)])


# ---- the host mirror over an oracle-backed engine --------------------------------------------------------------
class ExchangeEngine(OracleEngine):
    """OracleEngine + the replica-exchange entry points, backed by the oracle."""

    def set_ladder(self, betas):
        self.ladder = np.ascontiguousarray(betas, dtype=np.float64)
        L = self.ladder.size
        if not 2 <= L <= 256 or self.chain_offset % L or self.n_chains % L:
            raise ValueError("the shard must hold whole ladders")
        self.set_betas(np.tile(self.ladder, self.n_chains // L))
        self.rounds, self.xacc = 0, np.zeros(L - 1, np.int64)

    def replica_exchange(self):
        self.xacc += XO.exchange(self.ens, self.ladder.size, self.seed, self.rounds, self.chain_offset,
                                 betas=self.betas)
        self.rounds += 1
        self.launch_count += 1

    def exchange_counters(self):
        L, R = self.ladder.size, self.rounds
        att = np.array([(R + 1) // 2 if k % 2 == 0 else R // 2 for k in range(L - 1)]) * (self.n_chains // L)
        return self.xacc.copy(), att, R

    def ladder_sums(self):
        self.launch_count += 2
        return XO.ladder_sums(self.ens, self.ladder.size)


@pytest.fixture
def exchange_engine(monkeypatch):
    monkeypatch.setattr(A, "CudaEnsemble", ExchangeEngine)


LADDER = [0.5, 1.0, 2.0, 4.0]


def _pt_sim(path, M=32, steps=120, ex_every=20, lookahead=True, order="after"):
    chains = mb.ParticleEnsemble(O.init_synthetic(5, 0, M), 1.0, potential="double_well")
    pool = (mb.Move(mb.Displacement(0.0), mb.StandardGaussian(), mb.ComponentArray(σ=0.4), 1.0),)
    ex = dict(algorithm=mb.ReplicaExchange, dependencies=(mb.Metropolis,), ladder=LADDER,
              scheduler=list(range(ex_every, steps + 1, ex_every)))
    cb = dict(algorithm=mb.StoreCallbacks, callbacks=(mb.callback_energy, mb.callback_acceptance),
              scheduler=list(range(0, steps + 1, 5)))
    ladder_cb = dict(algorithm=mb.StoreCallbacks, callbacks=(mb.callback_ladder_energy, mb.callback_ladder_acceptance,
                                                             mb.callback_exchange_acceptance),
                     scheduler=list(range(0, steps + 1, 30)))
    algs = [dict(algorithm=mb.Metropolis, pool=pool, seed=5), ex, cb, ladder_cb]
    if order == "before":                       # stores at exchange times see the state BEFORE the swap
        algs = [algs[0], cb, ex, ladder_cb]
    sim = mb.Simulation(chains, tuple(algs), steps, path=str(path))
    sim.lookahead = lookahead
    return chains, sim


def _reference(M=32, steps=120, ex_every=20, order="after"):
    """Step-by-step oracle: Metropolis step, then exchange / stores in list order."""
    ref = O.Ensemble(O.init_synthetic(5, 0, M), 1.0, [0.4], potential=O.POT_DOUBLE_WELL)
    betas = np.tile(LADDER, M // 4)
    rounds, xacc = 0, np.zeros(3, np.int64)
    energy, ladder = {}, {}
    energy[0] = ref.callback_energy()
    ladder[0] = (XO.ladder_sums(ref, 4), xacc.copy(), 0)
    for t in range(1, steps + 1):
        _, z, ua = O.draws_philox(5, 0, M, t - 1, 1, with_cat=False)
        ref.sweep_replay(None, z, ua, betas=betas)
        if order == "before" and t % 5 == 0:
            energy[t] = ref.callback_energy()
        if t % ex_every == 0:
            xacc += XO.exchange(ref, 4, 5, rounds, 0, betas=betas)
            rounds += 1
        if order == "after" and t % 5 == 0:
            energy[t] = ref.callback_energy()
        if t % 30 == 0:
            ladder[t] = (XO.ladder_sums(ref, 4), xacc.copy(), rounds)
    return ref, energy, ladder


@pytest.mark.parametrize("order", ["after", "before"])
def test_mirror_files_match_the_oracle(tmp_path, exchange_engine, order):
    chains, sim = _pt_sim(tmp_path, order=order)
    mb.run(sim)
    ref, energy, ladder = _reference(order=order)
    assert np.array_equal(chains.engine.get_state(), ref.x)
    rows = open(tmp_path / "energy.dat").read().split("\n")[:-1]
    assert [int(r.split()[0]) for r in rows] == sorted(energy)
    for r in rows:
        t, v = r.split()
        assert abs(float(v) / energy[int(t)] - 1) < 1e-13, t
    le = open(tmp_path / "ladder_energy.dat").read().split("\n")[:-1]
    xa = open(tmp_path / "exchange_acceptance.dat").read().split("\n")[:-1]
    la = open(tmp_path / "ladder_acceptance.dat").read().split("\n")[:-1]
    assert len(le) == len(xa) == len(la) == len(ladder)
    for (t, (s, acc, R)), l1, l2, l3 in zip(sorted(ladder.items()), le, xa, la):
        assert l1 == f"{t} {A._jl([float(v) for v in s[:, 0] / s[:, -1]])}"
        with np.errstate(all="ignore"):
            att = np.array([(R + 1) // 2, R // 2, (R + 1) // 2]) * (32 // 4)
            assert l2 == f"{t} {A._jl([float(v) for v in acc / att])}"
            assert l3 == f"{t} {A._jl([[float(v) for v in row[1:-1] / row[-1]] for row in s])}"
    assert xa[0] == "0 [NaN, NaN, NaN]"                     # no attempt before the first round
    assert "\tReplicaExchange\n\t\tCalls: 6\n\t\tLadder: 4 rungs\n\t\tβ: [0.5, 1.0, 2.0, 4.0]\n" in \
        open(tmp_path / "summary.log").read()


@pytest.mark.parametrize("order", ["after", "before"])
def test_lookahead_stops_at_exchange_times(tmp_path, exchange_engine, order):
    """Exchange rounds and stores of the new callbacks are barriers of the look-ahead: the callback-only stores between
    them are fused into series calls, and every file equals the one of a run without look-ahead."""
    ca, sa = _pt_sim(tmp_path / "look", order=order)
    A_plan = A._make_lookahead(sa)
    mb.run(sa)
    cb, sb = _pt_sim(tmp_path / "plain", lookahead=False, order=order)
    mb.run(sb)
    for name in ("energy.dat", "acceptance.dat", "ladder_energy.dat", "ladder_acceptance.dat",
                 "exchange_acceptance.dat"):
        assert open(tmp_path / "look" / name).read() == open(tmp_path / "plain" / name).read(), name
    assert np.array_equal(ca.engine.get_state(), cb.engine.get_state())
    assert ca.engine.series_calls >= 6 and ca.engine.launch_count < cb.engine.launch_count
    # no stretch crosses an exchange time (every 20) or a store of the ladder callbacks (every 30)
    for t, plan in ((5, [5, 5, 5]), (20, []), (25, [5]), (30, []), (31, [4, 5]), (101, [4, 5, 5, 5])):
        sa.t = t
        assert A_plan() == plan, t


def test_misaligned_shard_raises(tmp_path, exchange_engine):
    chains = mb.ParticleEnsemble(np.zeros(30), 1.0)
    pool = (mb.Move(mb.Displacement(0.0), mb.StandardGaussian(), mb.ComponentArray(σ=0.1), 1.0),)
    with pytest.raises(ValueError):
        mb.Simulation(chains, (dict(algorithm=mb.Metropolis, pool=pool),
                               dict(algorithm=mb.ReplicaExchange, dependencies=(mb.Metropolis,), ladder=LADDER)),
                      10, path=str(tmp_path))


_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
import numpy as np, torch.distributed as dist
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=int(sys.argv[2]))
import montecarlo_b200 as mb
from montecarlo_b200 import arianna as A
from test_exchange_host import ExchangeEngine, _pt_sim
import pathlib
A.CudaEnsemble = ExchangeEngine
chains, sim = _pt_sim(pathlib.Path({path!r}), M={M})
mb.run(sim)
np.save(os.path.join({path!r}, f"x_rank{{chains.rank}}.npy"), chains.x)
dist.barrier(); dist.destroy_process_group()
"""


def _gloo_run(path, world, M=32):
    port = 29500 + (os.getpid() + 7 * world) % 2000
    path.mkdir()
    script = path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT, port=port, path=str(path), M=M))
    procs = [subprocess.Popen([sys.executable, str(script), str(r), str(world)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT) for r in range(world)]
    outs = [p.communicate(timeout=240)[0].decode() for p in procs]
    return [p.returncode for p in procs], outs


def test_two_rank_gloo_equals_one_rank(tmp_path):
    rc1, o1 = _gloo_run(tmp_path / "n1", 1)
    rc2, o2 = _gloo_run(tmp_path / "n2", 2)
    assert rc1 == [0] and rc2 == [0, 0], "\n".join(o1 + o2)
    x1 = np.load(tmp_path / "n1" / "x_rank0.npy")
    x2 = np.concatenate([np.load(tmp_path / "n2" / f"x_rank{r}.npy") for r in range(2)])
    assert np.array_equal(x1, x2)
    for name in ("energy.dat", "ladder_energy.dat", "exchange_acceptance.dat",
                 "ladder_acceptance.dat"):
        a = [r.split(" ", 1) for r in open(tmp_path / "n1" / name).read().split("\n")[:-1]]
        b = [r.split(" ", 1) for r in open(tmp_path / "n2" / name).read().split("\n")[:-1]]
        assert [t for t, _ in a] == [t for t, _ in b], name
        va = np.array([eval(v.replace("NaN", "float('nan')")) for _, v in a], dtype=float)
        vb = np.array([eval(v.replace("NaN", "float('nan')")) for _, v in b], dtype=float)
        np.testing.assert_allclose(va, vb, rtol=1e-13, equal_nan=True, err_msg=name)   # sums split across ranks
    # a rank whose shard does not hold whole ladders refuses to start (M = 36: shards of 18 chains, L = 4)
    rc, outs = _gloo_run(tmp_path / "bad", 2, M=36)
    assert rc != [0, 0] and all("ValueError" in o for o in outs)
