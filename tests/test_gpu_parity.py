"""GPU parity tests: the CUDA engine, called through the C ABI (ctypes), against the CPU oracle on the same seeded
inputs, against the committed golden fixtures, and -- at BASELINE.json's full sizes -- through size-independent
properties (chunking / sharding invariance, determinism, analytic ensemble averages).

Bars (north star): replay mode -> accept/reject decisions bit-identical, positions bit-identical (stricter than
the required 1e-12 relative); native-Philox mode -> identical decisions and |Δx| ≤ 1e-12 against the oracle fed
the same counter-based draws, plus 3σ agreement with the analytic harmonic averages.
"""
import math
import os

import numpy as np
import pytest

import montecarlo_b200 as mb
from montecarlo_b200 import policy_guided as PG
from oracle import oracle as O

pytestmark = pytest.mark.gpu

POTS = {"harmonic": O.POT_HARMONIC, "quartic": O.POT_QUARTIC, "double_well": O.POT_DOUBLE_WELL}


def _xoshiro_draws(x0, beta, sigma, weight, K, seed=42):
    gen = O.Ensemble(x0, beta, sigma, weight)
    gen.seed_xoshiro(seed)
    return gen.draws_xoshiro(K)


def _case(base_id, *values, pot="harmonic", betas=False, fast=False):
    """One parameter set of a test that was first written for the harmonic potential, a scalar β and EXACT arithmetic:
    its id is the id of that base case plus -<potential>, -betas and -fast where the set differs from it, so the ids of
    the original cases do not change."""
    tags = ([pot] if pot != "harmonic" else []) + (["betas"] if betas else []) + (["fast"] if fast else [])
    return pytest.param(*values, id="-".join([base_id] + tags))


def _beta_ladder(M, seed):
    """Per-chain β over 0.25 .. 8, with chain 1 at β = 0 (every move is accepted, in both arithmetics) and chain M/2 at
    β = 50 (almost every uphill move is rejected)."""
    b = np.random.default_rng(seed).uniform(0.25, 8.0, M)
    b[1], b[M // 2] = 0.0, 50.0
    return b


def _assert_sensitive(ref, pot, betas=None):
    """The oracle's run can tell a wrong potential, β or σ apart: 5 % .. 95 % of the moves are accepted (the β = 0 and
    β = 50 chains aside), the β = 0 chain accepted every move, and double-well chains end on both sides of the barrier."""
    keep = np.ones(ref.M, dtype=bool)
    if betas is not None:
        keep = (betas != 0.0) & (betas != 50.0)
        assert np.array_equal(ref.acc[:, betas == 0.0], ref.tot[:, betas == 0.0])
    frac = ref.acc[:, keep].sum() / ref.tot[:, keep].sum()
    assert 0.05 < frac < 0.95, frac
    if pot == "double_well":
        assert 0 < np.count_nonzero(ref.x < 0) < ref.M
    return frac


def _flip_report(bad, x0, K, seed, off, sigma, weight, pot, arith, betas, beta=2.0):
    """(chain, step, α − u) of the first decision that differs between the device and the oracle, for the first chains
    in `bad`: each is re-run alone (one step per launch, the same scalar β and per-chain β as the ensemble) from its
    state x0[c] at step 0, against the oracle with α."""
    rows = []
    for c in bad[:3]:
        b = float(betas[c]) if betas is not None else beta
        uc, z, ua = O.draws_philox(seed, off + c, 1, 0, K)
        ref = O.Ensemble(x0[c:c + 1], b, sigma, weight, potential=POTS[pot])
        dec, _, alpha = ref.sweep_replay(uc, z, ua, want_decisions=True, want_alpha=True)
        with mb.CudaEnsemble(1, beta, sigma, weight, seed=seed, chain_offset=off + c, potential=pot, arith=arith) as eng:
            eng.set_state(x0[c:c + 1])
            if betas is not None:
                eng.set_betas(betas[c:c + 1])
            n = 0
            for t in range(K):
                eng.sweep(1)
                a = int(eng.chain_counters()[0].sum())
                if a - n != dec[t, 0]:
                    rows.append((int(c), t, float(alpha[t, 0] - ua[t, 0])))
                    break
                n = a
    return rows


def _assert_native_parity(x, acc, tot, ref, report):
    """The native-Philox bar: per-chain accept and total counters identical to the oracle fed the same draws, then
    max |Δx| < 1e-12.  `report(bad_chains)` names the first flipped decisions when the counters differ."""
    bad = np.flatnonzero((acc.astype(np.int64) != ref.acc).any(axis=0) | (tot.astype(np.int64) != ref.tot).any(axis=0))
    assert bad.size == 0, (bad.size, report(bad))
    assert np.max(np.abs(x - ref.x)) < 1e-12, float(np.max(np.abs(x - ref.x)))


# ---------------------------------------------------------------------------------------------------------
# replay mode: bit-exact
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pot", ["harmonic", "quartic", "double_well"])
@pytest.mark.parametrize("sigma,weight", [([0.1], [1.0]), ([0.2] * 7, [0.4] + [0.1] * 6), ([1.5, 0.01], [0.3, 0.7])])
@pytest.mark.parametrize("M", [10007, 10006, 512])        # odd M: per-thread loads; even M: bulk-copy (TMA) tiles
def test_replay_bit_exact(pot, sigma, weight, M):
    K, beta = 67, 2.0                                 # ragged M (not a multiple of the block), K not a multiple of 4 or 8
    x0 = O.init_synthetic(11, 0, M)
    uc, z, ua = _xoshiro_draws(x0, beta, sigma, weight, K)
    ref = O.Ensemble(x0, beta, sigma, weight, potential=POTS[pot])
    dec_ref, _, alpha = ref.sweep_replay(uc, z, ua, want_decisions=True, want_alpha=True)
    with mb.CudaEnsemble(M, beta, sigma, weight, potential=pot, arith="exact") as eng:
        eng.set_state(x0)
        dec = eng.sweep_replay(uc if len(sigma) > 1 else None, z, ua, want_decisions=True)
        x, e = eng.get_state(with_energy=True)
        acc, tot = eng.chain_counters()
        bad = np.argwhere(dec != dec_ref)
        # a flip is only legitimate if |α − u| is within an ulp of exp(); report it instead of assuming impossibility
        assert bad.size == 0, [(int(s), int(c), float(alpha[s, c] - ua[s, c])) for s, c in bad[:5]]
        assert np.array_equal(x, ref.x), float(np.max(np.abs(x - ref.x)))
        assert np.array_equal(e, ref.e)
        assert np.array_equal(acc.astype(np.int64), ref.acc) and np.array_equal(tot.astype(np.int64), ref.tot)
        assert eng.steps_done == K
        a_sum, t_sum = eng.counters()
        assert np.array_equal(a_sum, ref.acc.sum(axis=1)) and np.array_equal(t_sum, ref.tot.sum(axis=1))


@pytest.mark.parametrize("name", ["replay_single.npz", "replay_multi.npz", "replay_doublewell.npz"])
def test_replay_golden_fixtures(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name))
    pot = {v: k for k, v in POTS.items()}[int(g["pot"])]
    M = g["x0"].size
    with mb.CudaEnsemble(M, float(g["beta"]), g["sigma"], g["weight"], potential=pot, arith="exact") as eng:
        eng.set_state(g["x0"])
        dec = eng.sweep_replay(g["u_cat"], g["z"], g["u_acc"], want_decisions=True)
        x, e = eng.get_state(with_energy=True)
        acc, tot = eng.chain_counters()
        assert np.array_equal(np.packbits(dec), g["decisions"])
        assert np.array_equal(x, g["x"]) and np.array_equal(e, g["e"])
        assert np.array_equal(acc, g["acc"]) and np.array_equal(tot, g["tot"])
        me, ma = eng.callbacks()
        assert abs(me / float(g["energy"]) - 1) < 1e-13
        np.testing.assert_allclose(ma, g["acceptance"], rtol=1e-13, equal_nan=True)


def test_sixteen_move_pool_all_generators():
    """ARIANNA_MAX_MOVES moves: the multi-move kernels keep 2 KB of counters per move in shared memory next to their
    tables, which passes the 48 KB default for 12+ moves (opt-in required) -- replay, XOSHIRO and native Philox."""
    M, K, beta = 3001, 23, 2.0
    sigma = [0.05 * (k + 1) for k in range(16)]
    weight = [1.0 / 16] * 16
    x0 = O.init_synthetic(3, 0, M)
    uc, z, ua = _xoshiro_draws(x0, beta, sigma, weight, K)
    ref = O.Ensemble(x0, beta, sigma, weight)
    dref, _, _ = ref.sweep_replay(uc, z, ua, want_decisions=True)
    with mb.CudaEnsemble(M, beta, sigma, weight, arith="exact") as eng:                    # replay
        eng.set_state(x0)
        assert np.array_equal(eng.sweep_replay(uc, z, ua, want_decisions=True), dref)
        assert np.array_equal(eng.get_state(), ref.x)
        acc, tot = eng.chain_counters()
        assert np.array_equal(acc.astype(np.int64), ref.acc) and np.array_equal(tot.astype(np.int64), ref.tot)
    with mb.CudaEnsemble(M, beta, sigma, weight, rng="xoshiro", arith="exact") as eng:     # device xoshiro256++
        gen = O.Ensemble(x0, beta, sigma, weight)
        gen.seed_xoshiro(42)
        eng.set_state(x0)
        eng.set_rng_state(gen.states)
        eng.set_ziggurat_tables(*O.ziggurat_tables())
        eng.sweep(K)
        assert np.max(np.abs(eng.get_state() - ref.x)) < 1e-12      # ziggurat tail samples go through log/exp (≤ 1 ulp)
        assert np.array_equal(eng.chain_counters()[0].astype(np.int64), ref.acc)
    uc, z, ua = O.draws_philox(3, 0, M, 0, K)
    ref = O.Ensemble(x0, beta, sigma, weight)
    ref.sweep_replay(uc, z, ua)
    with mb.CudaEnsemble(M, beta, sigma, weight, seed=3, arith="fast") as eng:             # native Philox
        eng.init_synthetic()
        eng.sweep(K)
        assert np.max(np.abs(eng.get_state() - ref.x)) < 1e-12
        acc, tot = eng.chain_counters()
        assert np.array_equal(acc.astype(np.int64), ref.acc) and np.array_equal(tot.astype(np.int64), ref.tot)


def test_replay_per_chain_beta_and_chunked_calls():
    M, K = 4099, 40
    x0 = O.init_synthetic(5, 0, M)
    betas = np.linspace(0.5, 4.0, M)                  # the β sweep {0.5,1,2,4} of config 5, in one ensemble
    uc, z, ua = _xoshiro_draws(x0, 2.0, [0.3], [1.0], K)
    ref = O.Ensemble(x0, 2.0, [0.3])
    dec_ref, _, _ = ref.sweep_replay(None, z, ua, want_decisions=True, betas=betas)
    with mb.CudaEnsemble(M, 2.0, [0.3], arith="exact") as eng:
        eng.set_state(x0)
        eng.set_betas(betas)
        d1 = eng.sweep_replay(None, z[:13], ua[:13], want_decisions=True)
        d2 = eng.sweep_replay(None, z[13:], ua[13:], want_decisions=True)
        assert np.array_equal(np.concatenate([d1, d2]), dec_ref)
        assert np.array_equal(eng.get_state(), ref.x)
        assert np.array_equal(eng.chain_counters()[0][0], ref.acc[0])


def test_replay_edge_cases():
    # M = 1, K = 1; u_acc = 0 (always accept unless α = 0/NaN); NaN / inf states reject (min(1, NaN) semantics)
    with mb.CudaEnsemble(1, 2.0, [0.1], arith="exact") as eng:
        eng.set_state(np.array([0.25]))
        assert eng.sweep_replay(None, np.zeros((0, 1)), np.zeros((0, 1)), want_decisions=True).shape == (0, 1)  # K = 0
        d = eng.sweep_replay(None, np.array([[1.0]]), np.array([[0.0]]), want_decisions=True)
        assert d[0, 0] == 1 and eng.get_state()[0] == 0.25 + 0.1
    x0 = np.array([np.inf, np.nan, 1e308, 0.1 + 3 * 2.0 ** -54, -0.0])
    z = np.array([[1.0, 1.0, 1e10, 3.0, 0.0]])
    ua = np.array([[0.5, 0.5, 0.5, 0.999999, 1 - 2.0 ** -53]])
    ref = O.Ensemble(x0, 2.0, [1.0])
    with np.errstate(all="ignore"):
        dref, _, _ = ref.sweep_replay(None, z, ua, want_decisions=True)
    with mb.CudaEnsemble(5, 2.0, [1.0], arith="exact") as eng:
        eng.set_state(x0)
        d = eng.sweep_replay(None, z, ua, want_decisions=True)
        assert np.array_equal(d, dref) and list(d[0]) == [0, 0, 0, 0, 1]
        x = eng.get_state()
        assert np.array_equal(x, ref.x, equal_nan=True)
        assert x[3] == (x0[3] + 3.0) - 3.0 and x[3] != x0[3]      # reject path is fl(fl(x+δ)−δ), not a restore


def test_replay_device_pointers():
    import torch
    M, K = 3000, 20
    x0 = O.init_synthetic(9, 0, M)
    uc, z, ua = _xoshiro_draws(x0, 2.0, [0.2, 0.4], [0.5, 0.5], K)
    ref = O.Ensemble(x0, 2.0, [0.2, 0.4], [0.5, 0.5])
    dref, _, _ = ref.sweep_replay(uc, z, ua, want_decisions=True)
    with mb.CudaEnsemble(M, 2.0, [0.2, 0.4], [0.5, 0.5], arith="exact") as eng:
        eng.set_state(x0)
        with torch.cuda.stream(eng.torch_stream()):
            duc, dz, dua = (torch.from_numpy(a).cuda() for a in (uc, z, ua))
            ddec = torch.empty((K, M), dtype=torch.uint8, device="cuda")
            eng.sweep_replay_device(K, duc.data_ptr(), dz.data_ptr(), dua.data_ptr(), ddec.data_ptr())
            eng.synchronize()
        assert np.array_equal(ddec.cpu().numpy(), dref) and np.array_equal(eng.get_state(), ref.x)


def test_error_behaviour():
    with mb.CudaEnsemble(8, 2.0, [0.2, 0.4], [0.5, 0.5]) as eng:
        with pytest.raises(mb.AriannaError):                      # multi-move replay needs u_cat
            eng.sweep_replay(None, np.zeros((1, 8)), np.zeros((1, 8)))
        with pytest.raises(mb.AriannaError):                      # Normal(0, σ ≤ 0) throws in the reference
            eng.set_params(0, -1.0)
        with pytest.raises(mb.AriannaError):
            eng.set_params(5, 0.1)
        with pytest.raises(mb.AriannaError):                      # XOSHIRO state on a PHILOX handle
            eng.set_rng_state(np.zeros((8, 4), dtype=np.uint64))
        with pytest.raises(mb.AriannaError):
            eng.pgmc_estimate(0, [1])
    with pytest.raises(mb.AriannaError):
        mb.CudaEnsemble(8, 2.0, [0.1, 0.1], [0.7, 0.7])


# ---------------------------------------------------------------------------------------------------------
# native Philox mode against the oracle fed the same counter-based draws
# ---------------------------------------------------------------------------------------------------------
def test_init_synthetic_bit_exact():
    with mb.CudaEnsemble(5001, 2.0, [0.1], seed=42, chain_offset=12345) as eng:
        eng.init_synthetic()
        assert np.array_equal(eng.get_state(), O.init_synthetic(42, 12345, 5001))
        eng.init_synthetic(7)
        assert np.array_equal(eng.get_state(), O.init_synthetic(7, 12345, 5001))


@pytest.mark.parametrize("arith", ["exact", "fast"])
@pytest.mark.parametrize("sigma,weight,pot,betas", [
    _case(f"sigma{i}-weight{i}", s, w, pot, b, pot=pot, betas=b)
    for i, (s, w) in enumerate([([0.1], [1.0]), ([0.2] * 7, [0.4] + [0.1] * 6)]) for pot in POTS for b in (False, True)])
def test_philox_native_matches_oracle(arith, sigma, weight, pot, betas):
    """Every plain native sweep -- sweep_philox_kernel<P, A, false, B> (one move) and sweep_multi_kernel<P, A, B> (seven
    moves) for the three potentials, both arithmetics, β a kernel constant (B = false) or read per chain (B = true) --
    against the oracle fed the same counter-based draws."""
    M, K, beta, seed, off = 6001, 101, 2.0, 42, 777     # odd K: exercises the half-used Box-Muller pair
    x0 = O.init_synthetic(seed, off, M)
    bl = _beta_ladder(M, seed) if betas else None
    uc, z, ua = O.draws_philox(seed, off, M, 0, K)
    ref = O.Ensemble(x0, beta, sigma, weight, potential=POTS[pot])
    ref.sweep_replay(uc, z, ua, betas=bl)
    _assert_sensitive(ref, pot, bl)
    with mb.CudaEnsemble(M, beta, sigma, weight, seed=seed, chain_offset=off, potential=pot, arith=arith) as eng:
        eng.init_synthetic()
        if betas:
            eng.set_betas(bl)
        eng.sweep(K)
        x = eng.get_state()
        acc, tot = eng.chain_counters()
    # Box-Muller on the device uses CUDA's log/sincospi, the oracle glibc's: normals agree to a few ulp, so x agrees
    # to ~1e-15 and a decision can only flip when |α − u| ≲ 1e-15
    _assert_native_parity(x, acc, tot, ref,
                          lambda bad: _flip_report(bad, x0, K, seed, off, sigma, weight, pot, arith, bl, beta))


@pytest.mark.parametrize("arith", ["exact", "fast"])
@pytest.mark.parametrize("nm", [1, 3])
def test_chunk_and_shard_invariance(arith, nm):
    M, seed = 5000, 3
    sigma, weight = [0.1, 0.3, 0.9][:nm], [[1.0], None, [0.5, 0.25, 0.25]][nm - 1]

    def run(chunks, offset=0, n=M):
        with mb.CudaEnsemble(n, 2.0, sigma, weight, seed=seed, chain_offset=offset, arith=arith) as eng:
            eng.init_synthetic()
            for k in chunks:
                eng.sweep(k, reduce=(k % 2 == 0))
            return eng.get_state(), eng.chain_counters()

    x_ref, (a_ref, t_ref) = run([20])
    for chunks in ([7, 12, 1], [1] * 20, [3, 17], [10, 10]):   # includes launches that start / end on odd steps
        x, (a, t) = run(chunks)
        assert np.array_equal(x, x_ref) and np.array_equal(a, a_ref) and np.array_equal(t, t_ref), chunks
    # sharding: two handles with chain offsets == one handle (global chain id keys the stream)
    xa, (aa, _) = run([20], 0, 1234)
    xb, (ab, _) = run([20], 1234, M - 1234)
    assert np.array_equal(np.concatenate([xa, xb]), x_ref)
    assert np.array_equal(np.concatenate([aa, ab], axis=1), a_ref)
    # seed + c − 1 (metropolis.jl:262): chain c+1 under `seed` == chain c under `seed + 1`
    with mb.CudaEnsemble(M - 1, 2.0, sigma, weight, seed=seed + 1, arith=arith) as eng:
        eng.set_state(O.init_synthetic(seed, 1, M - 1))
        eng.sweep(20)
        assert np.array_equal(eng.get_state(), x_ref[1:])


def test_callbacks_fused_and_standalone_match_oracle():
    M, seed = 100003, 42
    x0 = O.init_synthetic(seed, 0, M)
    ref = O.Ensemble(x0, 2.0, [0.1])
    with mb.CudaEnsemble(M, 2.0, [0.1], seed=seed, arith="exact") as eng:
        eng.init_synthetic()
        me, ma = eng.callbacks()                                  # t = 0 store_first record
        assert abs(me / ref.callback_energy() - 1) < 1e-13 and math.isnan(ma[0])
        done = 0
        for K in (10, 1, 33):
            _, z, ua = O.draws_philox(seed, 0, M, done, K, with_cat=False)
            ref.sweep_replay(None, z, ua)
            done += K
            eng.sweep(K, reduce=True)                             # fused tail reduction
            s_fused = eng.callback_sums()
            eng.sweep(0, reduce=True)                             # standalone kernel over the same state
            s_alone = eng.callback_sums()
            np.testing.assert_allclose(s_fused, s_alone, rtol=1e-13)
            assert s_fused[2] == M
            me, ma = eng.callbacks()
            assert abs(me / ref.callback_energy() - 1) < 1e-12
            assert abs(ma[0] / ref.callback_acceptance()[0] - 1) < 1e-12


# the other potentials and per-chain β (sweep_philox_kernel<P, A, true, B>, all ten instantiations the harmonic
# scalar-β cases leave out) each with both interval forms: odd intervals over launches of 3 stores, whole-pair
# intervals in one launch
_SERIES_EXTRA = [("harmonic", True), ("quartic", False), ("quartic", True), ("double_well", False), ("double_well", True)]


@pytest.mark.parametrize("even,per_launch,arith,pot,betas", [
    _case(f"{even}-{pl}-{arith}", even, pl, arith, "harmonic", False)
    for even in (False, True) for pl in (0, 3) for arith in ("exact", "fast")] + [
    _case(f"{even}-{pl}-{arith}", even, pl, arith, pot, b, pot=pot, betas=b)
    for pot, b in _SERIES_EXTRA for even, pl in ((False, 3), (True, 0)) for arith in ("exact", "fast")])
def test_series_equals_per_store_sweeps(even, per_launch, arith, pot, betas, monkeypatch):
    """arianna_sweep_series == the loop [arianna_sweep(K_i, REDUCE); arianna_callback_sums] it replaces: identical
    chain states and counters (the draws are a pure function of (chain, step)), records equal up to the summation
    order, and equal to the oracle's callback_energy / callback_acceptance after every interval.  Odd interval
    lengths exercise store boundaries that split a Box-Muller pair."""
    if per_launch:
        monkeypatch.setenv("ARIANNA_SERIES_PER_LAUNCH", str(per_launch))
    M, seed = (70001 if pot == "harmonic" and not betas else 30011), 11
    # 22 stores > 16 per launch; empty intervals (two stores with no Metropolis step between them: Metropolis every
    # 2 steps, StoreCallbacks every step) at an even (44) AND at odd (57, 141) cumulative steps
    Ks = [10, 1, 7, 10, 10, 3, 0, 12, 1, 0, 4, 10, 10, 10, 9, 10, 11, 10, 10, 0, 2, 10]
    pre = 3                                                         # the series starts on an odd step
    if even:                                                        # whole-pair intervals: the flat-loop fast path
        Ks, pre = [10, 2, 8, 10, 10, 4, 6, 12, 4, 10, 10, 10, 8, 10, 12, 10, 10, 2, 10, 10], 4
    x0 = O.init_synthetic(seed, 0, M)
    bl = _beta_ladder(M, seed) if betas else None
    ref = O.Ensemble(x0, 2.0, [0.1], potential=POTS[pot])
    with mb.CudaEnsemble(M, 2.0, [0.1], seed=seed, potential=pot, arith=arith) as a, \
            mb.CudaEnsemble(M, 2.0, [0.1], seed=seed, potential=pot, arith=arith) as b:
        a.init_synthetic(); b.init_synthetic()
        if betas:
            a.set_betas(bl); b.set_betas(bl)
        a.sweep(pre); b.sweep(pre)
        rec = a.sweep_series(Ks)
        assert rec.shape == (len(Ks), 3) and a.steps_done == pre + sum(Ks)
        _, z, ua = O.draws_philox(seed, 0, M, 0, pre, with_cat=False)
        ref.sweep_replay(None, z, ua, betas=bl)
        done = pre
        for i, K in enumerate(Ks):
            b.sweep(K, reduce=True)
            sb = b.callback_sums()
            np.testing.assert_allclose(rec[i], sb, rtol=1e-13, err_msg=f"store {i}")
            assert rec[i, 2] == M
            if K:
                _, z, ua = O.draws_philox(seed, 0, M, done, K, with_cat=False)
                ref.sweep_replay(None, z, ua, betas=bl)
                done += K
            assert abs(rec[i, 0] / M / ref.callback_energy() - 1) < 1e-12
            assert abs(rec[i, 1] / M / ref.callback_acceptance()[0] - 1) < 1e-12
        assert np.array_equal(a.get_state(), b.get_state())
        assert np.array_equal(a.chain_counters()[0], b.chain_counters()[0])
        _assert_native_parity(a.get_state(), *a.chain_counters(), ref,
                              lambda bad: _flip_report(bad, x0, done, seed, 0, [0.1], [1.0], pot, arith, bl))
        _assert_sensitive(ref, pot, bl)
        # the last record doubles as the current callback sums
        np.testing.assert_array_equal(a.callback_sums(), rec[-1])
        me, ma = a.callbacks()
        assert abs(me / ref.callback_energy() - 1) < 1e-12
        # records can stay on the device (one all-reduce for the whole stretch) and be fetched later
        a.sweep_series([4, 4], read=False)
        b.sweep(4, reduce=True); s1 = b.callback_sums(); b.sweep(4, reduce=True); s2 = b.callback_sums()
        np.testing.assert_allclose(a.series_global(2), np.stack([s1, s2]), rtol=1e-13)


_POOLS_7_3 = [([0.2] * 7, [0.4] + [0.1] * 6), ([0.1, 0.3, 0.9], [0.5, 0.25, 0.25])]


@pytest.mark.parametrize("sigma,weight,even,arith,pot,betas", [
    _case(f"sigma{i}-weight{i}-{even}-{arith}", s, w, even, arith, "harmonic", False)
    for i, (s, w) in enumerate(_POOLS_7_3) for even in (False, True) for arith in ("exact", "fast")] + [
    # the other potentials and per-chain β (sweep_multi_kernel<P, A, B> with records): both interval forms in both
    # arithmetics, the two pools taking turns
    _case(f"sigma{i}-weight{i}-{even}-{arith}", *_POOLS_7_3[i], even, arith, pot, b, pot=pot, betas=b)
    for n, (pot, b) in enumerate(_SERIES_EXTRA) for even in (False, True) for arith in ("exact", "fast")
    for i in [(n + even) % 2]])
def test_series_multi_move_pools(sigma, weight, even, arith, pot, betas, monkeypatch):
    """Series mode for multi-move pools: the record of every store carries callback_acceptance as the reference defines
    it -- one entry PER MOVE, the mean over chains of accepted_calls/total_calls, NaN while some chain never tried the
    move (metropolis.jl:319-321) -- and equals the standalone reduction over the same state and the oracle's callbacks;
    chains and per-move counters are bit-identical to the per-store sweeps.  C4's pool is the 7-move case
    (pgmc_test.jl:17-25)."""
    monkeypatch.setenv("ARIANNA_SERIES_PER_LAUNCH", "5")
    M, seed, nm = 30011, 13, len(sigma)
    Ks = [1, 10, 7, 0, 10, 3, 12, 1, 0, 4, 10, 9]
    pre = 3
    if even:
        Ks, pre = [2, 10, 8, 4, 10, 6, 12, 2, 2, 4, 10, 8], 2
    x0 = O.init_synthetic(seed, 0, M)
    bl = _beta_ladder(M, seed) if betas else None
    ref = O.Ensemble(x0, 2.0, sigma, weight, potential=POTS[pot])
    with mb.CudaEnsemble(M, 2.0, sigma, weight, seed=seed, potential=pot, arith=arith) as a, \
            mb.CudaEnsemble(M, 2.0, sigma, weight, seed=seed, potential=pot, arith=arith) as b:
        a.init_synthetic(); b.init_synthetic()
        if betas:
            a.set_betas(bl); b.set_betas(bl)
        a.sweep(pre); b.sweep(pre)
        rec = a.sweep_series(Ks)
        assert rec.shape == (len(Ks), 2 + nm) and a.steps_done == pre + sum(Ks)
        uc, z, ua = O.draws_philox(seed, 0, M, 0, pre)
        ref.sweep_replay(uc, z, ua, betas=bl)
        done = pre
        for i, K in enumerate(Ks):
            b.sweep(K, reduce=True)                                 # fused per-move record of ONE interval
            sb = b.callback_sums()
            np.testing.assert_allclose(rec[i], sb, rtol=1e-13, equal_nan=True, err_msg=f"store {i}")
            if K:
                uc, z, ua = O.draws_philox(seed, 0, M, done, K)
                ref.sweep_replay(uc, z, ua, betas=bl)
                done += K
            assert rec[i, -1] == M
            assert abs(rec[i, 0] / M / ref.callback_energy() - 1) < 1e-12
            np.testing.assert_allclose(rec[i, 1:-1] / M, ref.callback_acceptance(), rtol=1e-12, equal_nan=True)
        # early stores: some chain has not tried every move yet -> NaN entries, exactly like the reference's mean
        assert np.isnan(rec[0, 1:-1]).any()
        assert np.array_equal(a.get_state(), b.get_state())
        for u, v in zip(a.chain_counters(), b.chain_counters()):
            assert np.array_equal(u, v)
        acc, tot = a.chain_counters()
        _assert_native_parity(a.get_state(), acc, tot, ref,
                              lambda bad: _flip_report(bad, x0, done, seed, 0, sigma, weight, pot, arith, bl))
        _assert_sensitive(ref, pot, bl)
        # the last record doubles as the current callback sums; the standalone reduction agrees
        np.testing.assert_array_equal(a.callback_sums(), rec[-1])
        a.sweep(0, reduce=True)
        np.testing.assert_allclose(a.callback_sums(), rec[-1], rtol=1e-13)
        me, ma = a.callbacks()
        np.testing.assert_allclose(ma, ref.callback_acceptance(), rtol=1e-12, equal_nan=True)


@pytest.mark.parametrize("weight", [[0.1234567, 0.3, 0.0765433, 0.5],        # thresholds off the bucket grid
                                    [0.5, 1e-5, 2e-5, 0.49997],              # two thresholds inside ONE bucket
                                    [0.25, 0.25, 0.5, 0.0]])                 # on bucket edges; a move that is never picked
def test_multi_move_host_job_and_pick_table(weight):
    """The pipelined host job for a multi-move pool (slices keep the row pitch of the per-move counter arrays), and the
    categorical pick: thresholds that fall inside a bucket of the 4096-entry table take the exact-compare paths."""
    import torch
    M, seed = 50021, 4
    sigma = [0.1, 0.2, 0.4, 0.8]
    Ks = [10, 10, 5, 10]
    x0 = O.init_synthetic(seed, 0, M)
    xin = torch.from_numpy(x0.copy()).pin_memory()
    xout = torch.empty(M, dtype=torch.float64).pin_memory()
    ref = O.Ensemble(x0, 2.0, sigma, weight)
    uc, z, ua = O.draws_philox(seed, 0, M, 0, sum(Ks))
    _, mov, _ = ref.sweep_replay(uc, z, ua, want_decisions=True)
    with mb.CudaEnsemble(M, 2.0, sigma, weight, seed=seed) as a, mb.CudaEnsemble(M, 2.0, sigma, weight, seed=seed) as b:
        b.set_state(x0)
        rec_b = b.sweep_series(Ks)
        rec_a = a.run_host_job(Ks, x_in=xin.data_ptr(), x_out=xout.data_ptr(), n_slices=3)
        np.testing.assert_allclose(rec_a, rec_b, rtol=1e-13)
        assert np.array_equal(xout.numpy(), b.get_state())
        for u, v in zip(a.chain_counters(), b.chain_counters()):
            assert np.array_equal(u, v)
        acc, tot = a.chain_counters()
        # tot is the histogram of the picked moves: identical to the oracle's scan over the same 32-bit uniforms
        assert np.array_equal(tot.astype(np.int64), ref.tot) and np.array_equal(acc.astype(np.int64), ref.acc)
        assert np.array_equal(tot.sum(axis=0), np.full(M, sum(Ks)))
    frac = np.bincount(mov.ravel(), minlength=4) / mov.size
    assert np.max(np.abs(frac - np.array(weight))) < 5 * np.sqrt(0.25 / mov.size)


@pytest.mark.parametrize("n_slices,pot,sigma,weight,betas", [
    _case(str(n), n, "harmonic", [0.1], [1.0], False) for n in (1, 3, 8)] + [
    # per-chain β read at a non-zero slice start (series_range / launch_multi offset the β array with the chains)
    _case(str(n), n, pot, s, w, True, pot=pot, betas=True)
    for n in (3, 8) for pot, s, w in (("quartic", [0.1], [1.0]), ("double_well", [0.1, 0.3, 0.9], [0.5, 0.25, 0.25]))])
def test_host_job_pipelined_over_slices(n_slices, pot, sigma, weight, betas):
    """arianna_run_host_job == set_state + sweep_series + get_state: chains and counters bit-identical (chains are
    independent, slice-major order changes nothing), records equal up to the order of the slice sums and equal to the
    oracle's callbacks after every interval."""
    import torch
    M, seed = (100003 if not betas else 30011), 5                  # not a multiple of the slice / CTA size
    nm = len(sigma)
    Ks = [10] * 14 + [3, 7]
    x0 = O.init_synthetic(seed, 0, M)
    bl = _beta_ladder(M, seed) if betas else None
    xin = torch.from_numpy(x0.copy()).pin_memory()
    xout = torch.empty(M, dtype=torch.float64).pin_memory()
    with mb.CudaEnsemble(M, 2.0, sigma, weight, seed=seed, potential=pot) as a, \
            mb.CudaEnsemble(M, 2.0, sigma, weight, seed=seed, potential=pot) as b:
        if betas:
            a.set_betas(bl); b.set_betas(bl)
        b.set_state(x0)
        rec_b = b.sweep_series(Ks)
        rec_a = a.run_host_job(Ks, x_in=xin.data_ptr(), x_out=xout.data_ptr(), n_slices=n_slices)
        assert np.array_equal(xout.numpy(), b.get_state()) and np.array_equal(a.get_state(), b.get_state())
        for u, v in zip(a.chain_counters(), b.chain_counters()):
            assert np.array_equal(u, v)
        np.testing.assert_allclose(rec_a, rec_b, rtol=1e-13)
        assert np.array_equal(rec_a[:, -1], np.full(len(Ks), float(M))) and a.steps_done == b.steps_done == sum(Ks)
        ref = O.Ensemble(x0, 2.0, sigma, weight, potential=POTS[pot])
        done = 0
        for i, K in enumerate(Ks):
            uc, z, ua = O.draws_philox(seed, 0, M, done, K, with_cat=nm > 1)
            ref.sweep_replay(uc, z, ua, betas=bl)
            done += K
            assert abs(rec_a[i, 0] / M / ref.callback_energy() - 1) < 1e-12, i
            np.testing.assert_allclose(rec_a[i, 1:-1] / M, ref.callback_acceptance(), rtol=1e-12, err_msg=str(i))
        _assert_native_parity(a.get_state(), *a.chain_counters(), ref,
                              lambda bad: _flip_report(bad, x0, done, seed, 0, sigma, weight, pot, "fast", bl))
        _assert_sensitive(ref, pot, bl)
        np.testing.assert_array_equal(a.callback_sums(), rec_a[-1])
        jt = a.job_timing()
        assert jt["h2d_ms"] > 0 and jt["d2h_ms"] > 0 and jt["h2d_gbs"] > 0.05 and jt["d2h_gbs"] > 0.05
        # a second job continues from the resident state (x_in = None) and may skip the download
        rec_a2 = a.run_host_job([4, 4], n_slices=n_slices)
        rec_b2 = b.sweep_series([4, 4])
        np.testing.assert_allclose(rec_a2, rec_b2, rtol=1e-13)
        assert np.array_equal(a.get_state(), b.get_state())
        # PCIe view of the job (both directions were used by the first job, none by the second)
        jt = a.job_timing()
        assert all(math.isnan(v) for v in jt.values())
        # the asynchronous records route: snapshot + (all-reduce) + D2H on a side stream while the next sweep runs
        pinned = torch.empty((2, 2 + nm), dtype=torch.float64).pin_memory()
        a.sweep_series([4, 4], read=False)
        a.series_global_begin(2, pinned.data_ptr())
        a.sweep(6)                                                  # overlaps the copy; must not disturb the records
        a.series_global_wait()
        rec_b3 = b.sweep_series([4, 4])
        b.sweep(6)
        np.testing.assert_allclose(pinned.numpy(), rec_b3, rtol=1e-13)
        assert np.array_equal(a.get_state(), b.get_state())
        # the overlapped trajectory write-back shares the copy stream with the host job
        a.get_state_async(xout.data_ptr())
        a.synchronize()
        assert np.array_equal(xout.numpy(), b.get_state())
    uc, z, ua = O.draws_philox(seed, 0, M, done, 8, with_cat=nm > 1)
    ref.sweep_replay(uc, z, ua, betas=bl)
    assert abs(rec_a2[-1, 0] / M / ref.callback_energy() - 1) < 1e-12


def test_device_timers():
    """arianna_timing: CUDA-event brackets of the last sweep and estimator pass (SURVEY.md §8b's arianna_timing)."""
    import time
    with mb.CudaEnsemble(1 << 22, 2.0, [0.1], seed=1) as eng:
        eng.init_synthetic()
        s, p = eng.timing()
        assert math.isnan(s) and math.isnan(p)
        eng.sweep(100, reduce=True)
        t0 = time.perf_counter()
        s100, _ = eng.timing()                                      # synchronises with the sweep
        wall = (time.perf_counter() - t0) * 1e3
        assert 0.05 < s100 < 50.0
        eng.sweep(1000)
        s1000, p = eng.timing()
        assert 4 * s100 < s1000 < 25 * s100 and math.isnan(p)       # device time scales with the fused steps
        eng.sweep_series([10] * 30)                                 # (first call: lazy module load + buffer allocation)
        eng.sweep_series([10] * 30)
        s300, _ = eng.timing()
        assert 1.2 * s100 < s300 < 10 * s100                        # (wide margins: a timing assert must never flake)
        eng.pgmc_estimate(10, [0])
        _, p = eng.timing()
        assert 0.01 < p < 50.0
        del wall


def test_c_host_example(tmp_path):
    """examples/harmonic_oscillator.c: the reference's example script written against the C ABI alone (gcc, no
    Python in the process) -- the records it prints are the oracle's callbacks."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe, libdir = str(tmp_path / "harmonic_oscillator"), os.path.dirname(mb.LIB_PATH)
    subprocess.check_call(["gcc", "-O2", "-Wall", "-Werror", "-I", os.path.join(root, "include"),
                           os.path.join(root, "examples", "harmonic_oscillator.c"), "-L", libdir, "-larianna_cuda",
                           f"-Wl,-rpath,{libdir}", "-o", exe])
    M, steps = 20000, 1030
    out = subprocess.run([exe, str(M), str(steps)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    rows = [ln for ln in out.stdout.splitlines() if ln and ln[0].isdigit()]
    assert [int(r.split()[0]) for r in rows] == [1000, 1010, 1020, 1030]
    ref = O.Ensemble(O.init_synthetic(42, 0, M), 2.0, [0.1])
    done = 0
    for r in rows:
        t = int(r.split()[0])
        _, z, ua = O.draws_philox(42, 0, M, done, t - done, with_cat=False)
        ref.sweep_replay(None, z, ua)
        done = t
        assert abs(float(r.split()[1]) / ref.callback_energy() - 1) < 1e-12
        assert abs(float(r.split("[")[1].rstrip("]")) / ref.callback_acceptance()[0] - 1) < 1e-12
    assert "chain-steps/s" in out.stdout


def test_series_small_ensemble_and_errors():
    """M = 10 (BASELINE config 1's width): up to ARIANNA_MAX_SERIES stores per launch; the XOSHIRO generator refuses."""
    M, seed = 10, 42
    x0 = O.init_synthetic(seed, 0, M)
    ref = O.Ensemble(x0, 2.0, [0.1])
    Ks = [1000] + [10] * 150
    with mb.CudaEnsemble(M, 2.0, [0.1], seed=seed, arith="fast") as eng:
        eng.init_synthetic()
        n0 = eng.launch_count
        rec = eng.sweep_series(Ks)
        assert eng.launch_count - n0 == 2 * math.ceil(len(Ks) / 64)
        done = 0
        for i, K in enumerate(Ks):
            _, z, ua = O.draws_philox(seed, 0, M, done, K, with_cat=False)
            ref.sweep_replay(None, z, ua)
            done += K
            assert abs(rec[i, 0] / M / ref.callback_energy() - 1) < 1e-11
            assert abs(rec[i, 1] / M / ref.callback_acceptance()[0] - 1) < 1e-12
        assert eng.sweep_series([]).shape == (0, 3)
        with pytest.raises(mb.AriannaError):
            eng.sweep_series([-1])
        with pytest.raises(mb.AriannaError):
            eng.run_host_job([10], n_slices=0)
        assert eng.run_host_job([], n_slices=2).shape == (0, 3)      # nothing to do is not an error
    with mb.CudaEnsemble(M, 2.0, [0.1, 0.2], seed=seed) as eng:
        assert eng.sweep_series([10]).shape == (1, 4)               # multi-move pools: per-move records
    with mb.CudaEnsemble(M, 2.0, [0.1], seed=seed, rng="xoshiro") as eng:
        with pytest.raises(mb.AriannaError) as ei:
            eng.sweep_series([10])
        assert ei.value.code == 4                                   # ARIANNA_ERR_UNSUPPORTED


def test_multi_move_acceptance_is_mean_of_ratios_with_nan():
    M, seed, K = 5000, 8, 3                                       # after 3 steps some chain has never tried move 7
    sigma, weight = [0.2] * 7, [0.4] + [0.1] * 6
    x0 = O.init_synthetic(seed, 0, M)
    uc, z, ua = O.draws_philox(seed, 0, M, 0, K)
    ref = O.Ensemble(x0, 2.0, sigma, weight)
    ref.sweep_replay(uc, z, ua)
    with mb.CudaEnsemble(M, 2.0, sigma, weight, seed=seed) as eng:
        eng.init_synthetic()
        eng.sweep(K, reduce=True)
        me, ma = eng.callbacks()
        want = ref.callback_acceptance()
        assert np.all(np.isnan(want))                             # 0/0 somewhere in every move at K = 3
        assert np.all(np.isnan(ma))
        eng.sweep(200, reduce=True)
        uc, z, ua = O.draws_philox(seed, 0, M, K, 200)
        ref.sweep_replay(uc, z, ua)
        me, ma = eng.callbacks()
        np.testing.assert_allclose(ma, ref.callback_acceptance(), rtol=1e-12)
        assert abs(me / ref.callback_energy() - 1) < 1e-11


# ---------------------------------------------------------------------------------------------------------
# XOSHIRO mode: the reference's generator family on the device
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sigma,weight,pot,arith", [
    _case(f"sigma{i}-weight{i}", s, w, pot, arith, pot=pot, fast=arith == "fast")
    for i, (s, w) in enumerate([([0.1], [1.0]), ([0.2, 0.6], [0.6, 0.4])]) for pot in POTS for arith in ("exact", "fast")])
def test_xoshiro_mode_matches_oracle(sigma, weight, pot, arith):
    """sweep_xoshiro_kernel<P, A, MULTI> for every potential, arithmetic and pool kind against the oracle's own
    xoshiro256++ / ziggurat sweep."""
    M, K, seed = 4001, (300 if pot == "harmonic" and arith == "exact" else 101), 42
    x0 = O.init_synthetic(seed, 0, M)
    ref = O.Ensemble(x0, 2.0, sigma, weight, potential=POTS[pot])
    ref.seed_xoshiro(seed)
    states0 = ref.states.copy()
    ref.sweep_xoshiro(K)
    _assert_sensitive(ref, pot)
    with mb.CudaEnsemble(M, 2.0, sigma, weight, seed=seed, potential=pot, rng="xoshiro", arith=arith) as eng:
        eng.set_state(x0)
        eng.set_rng_state(states0)                                    # (the engine's own default ziggurat tables)
        eng.sweep(K)
        x = eng.get_state()
        acc, tot = eng.chain_counters()
        st = eng.get_rng_state()
    assert np.array_equal(st, ref.states)                         # same number of raw draws consumed by every chain
    assert np.array_equal(acc.astype(np.int64), ref.acc) and np.array_equal(tot.astype(np.int64), ref.tot)
    # fast-path normals are bit-identical; ziggurat tail/wedge samples go through log/exp (≤ 1 ulp apart)
    assert np.max(np.abs(x - ref.x)) < 1e-12
    if arith == "exact":                                          # (FAST restores x on reject, the oracle re-applies −δ)
        assert np.mean(x == ref.x) > 0.9


def _xoshiro_unstep(s):
    """The state BEFORE one xoshiro256++ draw (the engine is linear and invertible)."""
    m64 = (1 << 64) - 1
    s0, s1, s2, s3 = (int(v) for v in s)
    e = ((s3 >> 45) | (s3 << 19)) & m64                # d ^ b
    a = s0 ^ e
    m = (s1 ^ a) ^ (s2 ^ a)                            # b ^ (b << 17)
    b = (m ^ (m << 17) ^ (m << 34) ^ (m << 51)) & m64
    return np.array([a, b, (s1 ^ a) ^ b, e ^ b], dtype=np.uint64)


def test_xoshiro_device_draws_the_julia_manual_normals():
    """The device generator through the C ABI against the known answers printed in the Julia manual (randn docstring:
    `rng = Xoshiro(123); randn(rng, ComplexF64)` = -0.45660053706486897 - 1.0346749725929225im, tests/test_oracle.py).
    One EXACT step with beta = 0 (always accepted), sigma = 1, x0 = 0 leaves x = 0 + (0 + 1 z) = z, the step's normal
    draw; a step consumes rand (u_cat), randn, rand (u_acc) in the reference's order (metropolis.jl:206, particle_1d.jl:57,
    metropolis.jl:184).  Chain 0 starts one draw BEFORE Xoshiro(123), so its normal is the manual's first one; chain 1
    starts AT Xoshiro(123) (u_cat uses up the draw the first normal took), so its normal is the manual's second."""
    from montecarlo_b200 import julia_rng as J
    s123 = J.xoshiro_state(123)
    r, nxt = O.xoshiro_next(_xoshiro_unstep(s123))
    assert np.array_equal(nxt, s123)                   # the inverse step is right
    states = np.stack([_xoshiro_unstep(s123), s123])
    with mb.CudaEnsemble(2, 0.0, [1.0], seed=0, rng="xoshiro", arith="exact") as eng:
        eng.set_state(np.zeros(2))
        eng.set_rng_state(states)                      # default tables = Julia's literal ki / wi / fi
        eng.sweep(1)
        z = eng.get_state()
        acc, _ = eng.chain_counters()
    assert list(acc[0]) == [1, 1]
    assert [float(0.7071067811865476 * v) for v in z] == [-0.45660053706486897, -1.0346749725929225]


# ---------------------------------------------------------------------------------------------------------
# PGMC estimator
# ---------------------------------------------------------------------------------------------------------
def test_pgmc_replay_matches_oracle(golden_dir):
    g = np.load(os.path.join(golden_dir, "pgmc.npz"))
    ns = g["sigma"].size
    with mb.CudaEnsemble(g["x0"].size, float(g["beta"]), g["sigma"], [1.0 / ns] * ns, arith="exact") as eng:
        eng.set_state(g["x0"])
        eng.pgmc_estimate_replay(int(g["q_batch"]), list(g["learn_ids"]), g["z"])
        gd = eng.pgmc_read(len(g["learn_ids"]))
        np.testing.assert_allclose(gd, g["gd"], rtol=1e-12)       # tree sum vs sequential fold
        assert np.array_equal(eng.get_state(), g["x"])            # perform/undo rounding drift reproduced exactly
        eng.pgmc_estimate_replay(int(g["q_batch"]), list(g["learn_ids"]), g["z"])   # accumulates (estimator.jl:130)
        assert eng.pgmc_read(2)[0, 4] == 2 * g["gd"][0, 4]
        eng.pgmc_reset()
        assert np.all(eng.pgmc_read(2) == 0)


@pytest.mark.parametrize("arith,pot", [_case(arith, arith, pot, pot=pot) for pot in POTS for arith in ("exact", "fast")])
def test_pgmc_native_matches_oracle(arith, pot):
    """pgmc_kernel<P, A, false> on the estimator stream and, in EXACT, pgmc_kernel<P, 0, true> fed the same draws,
    against the oracle's pgmc_replay."""
    M, seed, q = 20011, 42, 5                                     # odd q: second call starts on an odd sample index
    sigma = [0.2, 0.5, 1.3]
    learn = [1, 2]
    x0 = O.init_synthetic(seed, 0, M)
    ref = O.Ensemble(x0, 2.0, sigma, [0.4, 0.3, 0.3], potential=POTS[pot])
    want = np.zeros((2, 5))
    zs = []
    for call in range(3):
        zs.append(O.draws_pgmc_philox(seed, 0, M, call * len(learn) * q, len(learn) * q).reshape(len(learn), q, M))
    # sensitivity: the same draws under another potential give gradients far outside the 1e-10 bar
    other = O.Ensemble(x0, 2.0, sigma, [0.4, 0.3, 0.3], potential=POTS["quartic" if pot == "harmonic" else "harmonic"])
    alt = sum(other.pgmc_replay(q, learn, z) for z in zs)
    with mb.CudaEnsemble(M, 2.0, sigma, [0.4, 0.3, 0.3], seed=seed, potential=pot, arith=arith) as eng:
        eng.init_synthetic()
        for z in zs:
            want += ref.pgmc_replay(q, learn, z)
            eng.pgmc_estimate(q, learn)
        gd = eng.pgmc_read(2)
        np.testing.assert_allclose(gd, want, rtol=1e-10)          # the reference's own AD-parity tolerance is 1e-10
        assert gd[0, 4] == 3 * q * M
        assert np.all(np.abs(alt[:, :2] / want[:, :2] - 1) > 1e-3), (alt, want)
        if arith == "exact":
            assert np.max(np.abs(eng.get_state() - ref.x)) < 1e-13
        else:
            assert np.array_equal(eng.get_state(), x0)            # FAST never perturbs the chains
    if arith == "exact":                                          # the replay kernel on the same draws
        with mb.CudaEnsemble(M, 2.0, sigma, [0.4, 0.3, 0.3], potential=pot, arith="exact") as eng:
            eng.set_state(x0)
            for z in zs:
                eng.pgmc_estimate_replay(q, learn, z)
            np.testing.assert_allclose(eng.pgmc_read(2), want, rtol=1e-10)
            assert np.max(np.abs(eng.get_state() - ref.x)) < 1e-13


# ---------------------------------------------------------------------------------------------------------
# statistical acceptance tests of the reference (3σ bars), native mode
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("beta", [2.0, 2.5, 3.0])
@pytest.mark.parametrize("arith", ["fast", "exact"])
def test_harmonic_distribution(beta, arith):
    """test/distribution_test.jl:9-39 with M = 2^20 chains: ⟨x⟩ = 0, std = 1/√(2β), ⟨E⟩ = 1/(2β), acceptance."""
    M = 1 << 20
    with mb.CudaEnsemble(M, beta, [0.1], seed=42, arith=arith) as eng:
        eng.init_synthetic()
        eng.sweep(3000)                                           # x0 ~ U[−2,2) is far from stationary: burn
        x = eng.get_state()
        me, ma = eng.callbacks()
    s = 1 / math.sqrt(2 * beta)
    assert abs(x.mean()) < 3 * s / math.sqrt(M)
    assert abs(x.std() - s) < 3 * s / math.sqrt(2 * M)
    assert abs(me - 1 / (2 * beta)) < 3 * math.sqrt(1 / (2 * beta ** 2) / M)
    # cumulative acceptance since t = 0 includes the burn-in transient: loose window around (2/π)·atan(2s/σ)
    assert abs(ma[0] - 2 / math.pi * math.atan(2 * s / 0.1)) < 3e-3


def test_pgmc_learns_sigma_through_the_driver(tmp_path):
    """test/pgmc_test.jl:10-52 at M = 2^16 with faster learning rates: Static keeps σ₀, learners reach ≈1.2±0.2,
    ⟨energy⟩ ≈ 0.25 ± 0.05."""
    M, steps, burn = 1 << 16, 600, 50
    chains = mb.ParticleEnsemble(n_chains=M, beta=2.0)
    mk = lambda w: mb.Move(mb.Displacement(0.0), mb.StandardGaussian(), mb.ComponentArray(σ=0.2), w)
    pool = (mk(0.4), mk(0.1), mk(0.1), mk(0.1), mk(0.1), mk(0.1), mk(0.1))
    optimisers = (PG.Static(), PG.VPG(0.05), PG.BLPG(0.05), PG.BLAPG(2e-3, 1e-6), PG.NPG(0.5, 1e-6),
                  PG.ANPG(2e-3, 1e-6), PG.BLANPG(2e-3, 1e-6))
    sampletimes = mb.build_schedule(steps, burn, [0, 10])
    algorithm_list = (
        dict(algorithm=mb.Metropolis, pool=pool, seed=42, parallel=False),
        dict(algorithm=PG.PolicyGradientEstimator, dependencies=(mb.Metropolis,), optimisers=optimisers,
             q_batch_size=10, parallel=True),
        dict(algorithm=PG.PolicyGradientUpdate, dependencies=(PG.PolicyGradientEstimator,),
             scheduler=mb.build_schedule(steps, burn, 2)),
        dict(algorithm=mb.StoreCallbacks, callbacks=(mb.callback_energy, mb.callback_acceptance), scheduler=sampletimes),
        dict(algorithm=mb.StoreParameters, dependencies=(mb.Metropolis,), scheduler=sampletimes),
    )
    sim = mb.Simulation(chains, algorithm_list, steps, path=str(tmp_path))
    mb.run(sim)
    energies = np.loadtxt(tmp_path / "energy.dat")[:, 1]
    assert abs(energies[len(energies) // 2:].mean() - 0.25) < 5e-2
    sig = [m.parameters.σ for m in pool]
    assert sig[0] == 0.2
    assert all(abs(s - 1.2) < 0.2 for s in sig[1:]), sig


def test_on_device_optimiser_matches_host_updates(tmp_path):
    """PolicyGradientUpdate(on_device=True): averaging + learning_step! + reset in one device kernel, σ kept in a
    device-resident block read by the sweeps and the estimator -- against the host path (read-back, Python
    learning_step, set_params) on the same seeds: identical chains, identical counters, σ histories equal to the last
    bit (the six rules are restated operation by operation, IEEE sqrt / division), and each rule equal to the oracle's
    ao_learning_step on the same averaged record."""
    M, steps, burn = 1 << 14, 120, 20
    optimisers = (PG.Static(), PG.VPG(0.05), PG.BLPG(0.05), PG.BLAPG(2e-3, 1e-6), PG.NPG(0.5, 1e-6),
                  PG.ANPG(2e-3, 1e-6), PG.BLANPG(2e-3, 1e-6))

    def run(path, on_device):
        chains = mb.ParticleEnsemble(n_chains=M, beta=2.0)
        mk = lambda w: mb.Move(mb.Displacement(0.0), mb.StandardGaussian(), mb.ComponentArray(σ=0.2), w)
        pool = (mk(0.4), mk(0.1), mk(0.1), mk(0.1), mk(0.1), mk(0.1), mk(0.1))
        sim = mb.Simulation(chains, (
            dict(algorithm=mb.Metropolis, pool=pool, seed=42),
            dict(algorithm=PG.PolicyGradientEstimator, dependencies=(mb.Metropolis,), optimisers=optimisers, q_batch_size=10),
            dict(algorithm=PG.PolicyGradientUpdate, dependencies=(PG.PolicyGradientEstimator,),
                 scheduler=mb.build_schedule(steps, burn, 2), on_device=on_device),
            dict(algorithm=mb.StoreParameters, dependencies=(mb.Metropolis,), scheduler=mb.build_schedule(steps, burn, 10)),
        ), steps, path=str(path))
        mb.run(sim)
        hist = [open(path / "parameters" / str(k + 1) / "parameters.dat").read() for k in range(7)]
        return chains.x, chains.engine.chain_counters(), [m.parameters.σ for m in pool], hist, chains.engine.launch_count

    xh, ch, sh, hh, _ = run(tmp_path / "host", False)
    xd, cd, sd, hd, _ = run(tmp_path / "dev", True)
    assert sh[0] == sd[0] == 0.2 and all(s != 0.2 for s in sd[1:])
    assert sd == sh                                               # final σ, bit for bit
    assert hd == hh                                               # every stored σ along the way, byte for byte
    assert np.array_equal(xd, xh)
    for u, v in zip(cd, ch):
        assert np.array_equal(u, v)
    # every rule against the oracle on one hand-made record (sums over n = 1000 samples)
    rec = np.array([[310.5, 44.25, -120.75, 5120.0, 1000.0]])
    for name, kind, p1, p2 in [("VPG", O.OPT_VPG, 0.05, 0.0), ("BLPG", O.OPT_BLPG, 0.05, 0.0), ("BLAPG", O.OPT_BLAPG, 2e-3, 1e-6),
                               ("NPG", O.OPT_NPG, 0.5, 1e-6), ("ANPG", O.OPT_ANPG, 2e-3, 1e-6), ("BLANPG", O.OPT_BLANPG, 2e-3, 1e-6)]:
        with mb.CudaEnsemble(256, 2.0, [0.3, 0.7], [0.5, 0.5], seed=1) as eng:
            import torch
            with torch.cuda.stream(eng.torch_stream()):
                eng.pgmc_sums_tensor()[:5].copy_(torch.from_numpy(rec[0]))
            eng.pgmc_update_device([1], [(name, p1, p2)])
            want = O.learning_step(kind, p1, p2, rec[0, :4] / rec[0, 4], 0.7)
            assert eng.get_params(1) == want and eng.get_params(0) == 0.3, name
            assert np.all(eng.pgmc_read(1) == 0)                  # accumulators zeroed (update.jl:55)
    # an update that drives σ out of (0, ∞) is reported when the parameters are pulled (Normal(0, σ) throws in the reference)
    with mb.CudaEnsemble(256, 2.0, [0.3, 0.7], [0.5, 0.5], seed=1) as eng:
        with torch.cuda.stream(eng.torch_stream()):
            eng.pgmc_sums_tensor()[:5].copy_(torch.tensor([1.0, -1e6, 0.0, 1.0, 1.0], dtype=torch.float64))
        eng.pgmc_update_device([1], [("VPG", 1.0, 0.0)])
        with pytest.raises(mb.AriannaError):
            eng.get_params(1)


@pytest.mark.parametrize("arith", ["exact", "fast"])
@pytest.mark.parametrize("sigma,weight,learn", [([0.3], [1.0], [0]), ([0.2, 0.5, 1.3], [0.4, 0.3, 0.3], [0, 2])])
def test_device_sigma_sweeps_match_oracle(sigma, weight, learn, arith):
    """After an on-device optimiser step the sweeps read σ (and log-norm, 1/(2σ²)) from the device-resident parameter
    block: the single-move sweep_philox_kernel<0, A, *, true> and sweep_multi_kernel<0, A, false>, plain and series,
    against the oracle built on the σ that arianna_get_params returns.  σ is fetched only after the sweeps, so until
    then the host copy of the pool still holds the old values."""
    M, K, seed, off, q = 20011, 101, 21, 333, 5
    Ks = [11, 0, 7, 0, 0, 13, 1]                                  # odd and empty intervals
    nm = len(sigma)
    with mb.CudaEnsemble(M, 2.0, sigma, weight, seed=seed, chain_offset=off, arith=arith) as eng:
        eng.init_synthetic()
        eng.pgmc_estimate(q, learn)
        eng.pgmc_update_device(learn, [("VPG", 0.05, 0.0)] * len(learn))
        eng.sweep(K)
        rec = eng.sweep_series(Ks)
        x = eng.get_state()
        acc, tot = eng.chain_counters()
        new = [eng.get_params(k) for k in range(nm)]
    assert all((new[k] != sigma[k]) == (k in learn) for k in range(nm)), new
    x0 = O.init_synthetic(seed, off, M)
    if arith == "exact":                                          # the estimator's perform/undo drift of x
        est = O.Ensemble(x0, 2.0, sigma, weight)
        est.pgmc_replay(q, learn, O.draws_pgmc_philox(seed, off, M, 0, len(learn) * q).reshape(len(learn), q, M))
        x0 = est.x
    ref = O.Ensemble(x0, 2.0, new, weight)
    uc, z, ua = O.draws_philox(seed, off, M, 0, K, with_cat=nm > 1)
    ref.sweep_replay(uc, z, ua)
    done = K
    for i, k in enumerate(Ks):
        if k:
            uc, z, ua = O.draws_philox(seed, off, M, done, k, with_cat=nm > 1)
            ref.sweep_replay(uc, z, ua)
            done += k
        assert rec[i, -1] == M
        assert abs(rec[i, 0] / M / ref.callback_energy() - 1) < 1e-12, i
        np.testing.assert_allclose(rec[i, 1:-1] / M, ref.callback_acceptance(), rtol=1e-12, equal_nan=True, err_msg=str(i))
    # (an EXACT flip that the host rerun does not show: compare the device's log-norm, CUDA's log, with O.lognorm(new))
    _assert_native_parity(x, acc, tot, ref,
                          lambda bad: _flip_report(bad, x0, done, seed, off, new, weight, "harmonic", arith, None))
    _assert_sensitive(ref, "harmonic")


def test_driver_matches_oracle_on_gpu(tmp_path):
    """Simulation / run! through the real engine == the stepwise oracle (same check as the CPU test double)."""
    M, steps, burn, seed = 2048, 300, 100, 42
    x0 = O.init_synthetic(seed, 0, M)
    chains = mb.ParticleEnsemble(x0, 2.0, arith="exact")
    pool = (mb.Move(mb.Displacement(0.0), mb.StandardGaussian(), mb.ComponentArray(σ=0.1), 1.0),)
    sched = mb.build_schedule(steps, burn, [0, 10])
    sim = mb.Simulation(chains, (dict(algorithm=mb.Metropolis, pool=pool, seed=seed),
                                 dict(algorithm=mb.StoreCallbacks, callbacks=(mb.callback_energy, mb.callback_acceptance),
                                      scheduler=sched),
                                 dict(algorithm=mb.StoreTrajectories, scheduler=sched)), steps, path=str(tmp_path))
    mb.run(sim)
    assert chains.engine.steps_done == steps
    ref = O.Ensemble(x0, 2.0, [0.1])
    rows = np.loadtxt(tmp_path / "energy.dat")
    assert rows[0, 0] == 0 and abs(rows[0, 1] / ref.callback_energy() - 1) < 1e-13
    done = 0
    for row, t in zip(rows[1:], sched):
        _, z, ua = O.draws_philox(seed, 0, M, done, t - done, with_cat=False)
        ref.sweep_replay(None, z, ua)
        done = t
        assert row[0] == t and abs(row[1] / ref.callback_energy() - 1) < 1e-11
    t, x = mb.StoreTrajectories.read_binary(str(tmp_path / "trajectories" / "rank0.bin"), M)
    assert list(t) == [0] + sched and np.max(np.abs(x[-1] - ref.x)) < 1e-12
    chains.sync_move_counters()
    assert pool[0].total_calls == steps * M and pool[0].accepted_calls == int(ref.acc.sum())


# ---------------------------------------------------------------------------------------------------------
# BASELINE.json full sizes through size-independent properties
# ---------------------------------------------------------------------------------------------------------
def test_config2_replay_full_width():
    """Config 2 width (M = 2^24) in replay mode on a K = 6 chunk of the Julia-like xoshiro stream: decisions,
    counters and positions bit-identical to the oracle for ALL 2^24 chains."""
    M, K, beta = 1 << 24, 6, 2.0
    x0 = O.init_synthetic(42, 0, M)
    gen = O.Ensemble(x0, beta, [0.1])
    gen.seed_xoshiro(42)
    _, z, ua = gen.draws_xoshiro(K)
    ref = O.Ensemble(x0, beta, [0.1])
    dref, _, _ = ref.sweep_replay(None, z, ua, want_decisions=True)
    with mb.CudaEnsemble(M, beta, [0.1], arith="exact") as eng:
        eng.set_state(x0)
        dec = eng.sweep_replay(None, z, ua, want_decisions=True)
        assert np.array_equal(dec, dref)
        assert np.array_equal(eng.get_state(), ref.x)
        assert np.array_equal(eng.chain_counters()[0][0].astype(np.int64), ref.acc[0])


def test_config2_xoshiro_full_length_subset():
    """Config 2 length (10^4 steps) with the reference's generator family on the device: a shard of 2^14 chains run
    for the FULL 10^4 steps must reproduce the oracle's counters and generator states exactly, positions ≤1e-12."""
    M, K, seed = 1 << 14, 10 ** 4, 42
    x0 = O.init_synthetic(seed, 0, M)
    ref = O.Ensemble(x0, 2.0, [0.1])
    ref.seed_xoshiro(seed)
    st0 = ref.states.copy()
    ref.sweep_xoshiro(K)
    with mb.CudaEnsemble(M, 2.0, [0.1], seed=seed, rng="xoshiro", arith="exact") as eng:
        eng.set_state(x0)
        eng.set_rng_state(st0)
        eng.set_ziggurat_tables(*O.ziggurat_tables())
        eng.sweep(K)
        assert np.array_equal(eng.get_rng_state(), ref.states)
        assert np.array_equal(eng.chain_counters()[0][0].astype(np.int64), ref.acc[0])
        assert np.max(np.abs(eng.get_state() - ref.x)) < 1e-12


def test_config3_full_size_properties():
    """Config 3 (M = 2^27, callbacks every 10 steps): determinism, chunk invariance and the analytic averages at
    full size; a random subset of chains is checked against the oracle."""
    M, seed = 1 << 27, 42
    with mb.CudaEnsemble(M, 2.0, [0.1], seed=seed, arith="fast") as eng:
        eng.init_synthetic()
        for _ in range(100):
            eng.sweep(10, reduce=True)                            # 1000 steps = burn
        s1 = eng.callback_sums()
        x1 = eng.get_state()
        assert s1[2] == M
        assert abs(s1[0] / M - 0.25) < 3 * math.sqrt(1 / 8 / M) + 2e-4   # + residual burn-in bias at t = 1000
    # a slice of 4096 chains from the middle of the ensemble against the oracle (1000 steps)
    off, n = (1 << 26) + 12345, 4096
    x0 = O.init_synthetic(seed, off, n)
    ref = O.Ensemble(x0, 2.0, [0.1])
    _, z, ua = O.draws_philox(seed, off, n, 0, 1000, with_cat=False)
    ref.sweep_replay(None, z, ua)
    assert np.max(np.abs(x1[off:off + n] - ref.x)) < 1e-12
    # determinism + chunk invariance at full size: one launch of 1000 steps == 100 launches of 10
    with mb.CudaEnsemble(M, 2.0, [0.1], seed=seed, arith="fast") as eng:
        eng.init_synthetic()
        eng.sweep(1000, reduce=True)
        s2 = eng.callback_sums()
        x2 = eng.get_state()
    assert np.array_equal(x1, x2)
    np.testing.assert_allclose(s1, s2, rtol=1e-13)
    # the series path and the pipelined host job at full size: 100 store intervals of 10 steps == the above, and the
    # records inside the stretch carry the analytic acceptance (2/π)·atan(2s/σ) = 0.9365 of the stationary chain
    import torch
    xout = torch.empty(M, dtype=torch.float64).pin_memory()
    with mb.CudaEnsemble(M, 2.0, [0.1], seed=seed, arith="fast") as eng:
        eng.init_synthetic()
        rec = eng.run_host_job([10] * 100, x_out=xout.data_ptr(), n_slices=8)
        np.testing.assert_allclose(rec[-1], s1, rtol=1e-12)
        assert np.array_equal(xout.numpy(), x1)
        rec2 = eng.sweep_series([10] * 22)                         # 2 full launches of 11 stores, t = 1010 .. 1220
        assert np.all(rec2[:, 2] == M)
        assert np.all(np.abs(rec2[:, 0] / M - 0.25) < 3 * math.sqrt(1 / 8 / M) + 1e-4)
        acc_inc = (rec2[-1, 1] * 1220 - rec2[0, 1] * 1010) / M / 210   # mean acceptance over steps 1010 .. 1220
        assert abs(acc_inc - 2 / math.pi * math.atan(2 * 0.5 / 0.1)) < 1e-4


# ---------------------------------------------------------------------------------------------------------
# config 5 shape: β sweep in ONE ensemble, fused K = 100 sweeps with trajectory frames
# ---------------------------------------------------------------------------------------------------------
def test_config5_beta_sweep_with_trajectories(tmp_path):
    """BASELINE config 5 shrunk: β ∈ {0.5, 1, 2, 4} as per-chain β of one ensemble, StoreTrajectories on
    build_schedule(steps, burn, 100): every β group must sample its own N(0, 1/(2β)) (3σ bars)."""
    G = 1 << 16
    betas = np.repeat([0.5, 1.0, 2.0, 4.0], G)
    M, steps, burn = betas.size, 2000, 1000
    chains = mb.ParticleEnsemble(n_chains=M, beta=betas)
    pool = (mb.Move(mb.Displacement(0.0), mb.StandardGaussian(), mb.ComponentArray(σ=0.3), 1.0),)
    sched = mb.build_schedule(steps, burn, 100)
    sim = mb.Simulation(chains, (dict(algorithm=mb.Metropolis, pool=pool, seed=42),
                                 dict(algorithm=mb.StoreTrajectories, scheduler=sched, store_first=False)),
                        steps, path=str(tmp_path))
    mb.run(sim)
    assert chains.engine.launch_count <= len(sched) + 2          # one fused K = 100 launch per store interval
    t, x = mb.StoreTrajectories.read_binary(str(tmp_path / "trajectories" / "rank0.bin"), M)
    assert list(t) == sched and x.shape == (len(sched), M)
    last = x[-1].reshape(4, G)
    for g, b in enumerate([0.5, 1.0, 2.0, 4.0]):
        s = 1 / math.sqrt(2 * b)
        assert abs(last[g].mean()) < 3 * s / math.sqrt(G)
        assert abs(last[g].std() - s) < 3 * s / math.sqrt(2 * G)


# ---------------------------------------------------------------------------------------------------------
# multi-GPU: the Simulation path under torchrun + NCCL (skipped on single-GPU boxes)
# ---------------------------------------------------------------------------------------------------------
_NCCL_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch, torch.distributed as dist
rank = int(os.environ["RANK"]); torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
import montecarlo_b200 as mb
from montecarlo_b200 import policy_guided as PG
M, steps = 100003, 60
chains = mb.ParticleEnsemble(n_chains=M, beta=2.0, arith="exact")
pool = (mb.Move(mb.Displacement(0.0), mb.StandardGaussian(), mb.ComponentArray(σ=0.3), 0.5),
        mb.Move(mb.Displacement(0.0), mb.StandardGaussian(), mb.ComponentArray(σ=0.05), 0.5))
sched = mb.build_schedule(steps, 10, 10)
sim = mb.Simulation(chains, (dict(algorithm=mb.Metropolis, pool=pool, seed=7),
                             dict(algorithm=PG.PolicyGradientEstimator, dependencies=(mb.Metropolis,),
                                  optimisers=(PG.Static(), PG.VPG(0.05)), q_batch_size=3),
                             dict(algorithm=PG.PolicyGradientUpdate, dependencies=(PG.PolicyGradientEstimator,),
                                  scheduler=mb.build_schedule(steps, 10, 4)),
                             dict(algorithm=mb.StoreCallbacks, callbacks=(mb.callback_energy, mb.callback_acceptance),
                                  scheduler=sched)), steps, path={path!r})
mb.run(sim)
np.save(os.path.join({path!r}, f"x_rank{{rank}}.npy"), chains.x)
if rank == 0:
    np.save(os.path.join({path!r}, "sigma.npy"), np.array([m.parameters.σ for m in pool]))
dist.barrier(); dist.destroy_process_group()
"""


def test_two_gpu_nccl_simulation_matches_one_gpu(tmp_path):
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
                            "--master-addr", "127.0.0.1", "--master-port", str(29600 + n), str(script)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        outs[n] = (np.concatenate([np.load(d / f"x_rank{k}.npy") for k in range(n)]), np.load(d / "sigma.npy"),
                   np.loadtxt(d / "energy.dat"))
    np.testing.assert_allclose(outs[2][0], outs[1][0], rtol=0, atol=1e-12)     # per-chain results independent of sharding
    np.testing.assert_allclose(outs[2][1], outs[1][1], rtol=1e-12)
    np.testing.assert_allclose(outs[2][2], outs[1][2], rtol=1e-12)
    assert outs[1][1][0] == 0.3 and outs[1][1][1] != 0.05


_NCCL_SERIES_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch, torch.distributed as dist
rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"]); torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
import montecarlo_b200 as mb
M, steps = 100003, 400
chains = mb.ParticleEnsemble(n_chains=M, beta=2.0)
pool = (mb.Move(mb.Displacement(0.0), mb.StandardGaussian(), mb.ComponentArray(σ=0.1), 1.0),)
sim = mb.Simulation(chains, (dict(algorithm=mb.Metropolis, pool=pool, seed=7),
                             dict(algorithm=mb.StoreCallbacks, callbacks=(mb.callback_energy, mb.callback_acceptance),
                                  scheduler=mb.build_schedule(steps, 100, 10)),
                             dict(algorithm=mb.StoreLastFrames, scheduler=[steps])), steps, path={path!r})
mb.run(sim)                                           # look-ahead: ONE series call + ONE NCCL all-reduce per stretch
np.save(os.path.join({path!r}, f"x_rank{{rank}}.npy"), chains.x)
np.save(os.path.join({path!r}, f"launches_rank{{rank}}.npy"), np.array([chains.engine.launch_count]))
# the library-side path a Julia host uses: arianna_comm_init + arianna_series_global
ids = [mb.CudaEnsemble.nccl_unique_id() if rank == 0 else None]
dist.broadcast_object_list(ids, src=0)
off, n = mb.shard_bounds(M, rank, world)
with mb.CudaEnsemble(n, 2.0, [0.1], seed=7, chain_offset=off, n_chains_total=M) as eng:
    eng.comm_init(ids[0], rank, world)
    eng.init_synthetic()
    eng.sweep_series([100] + [10] * 30, read=False)
    np.save(os.path.join({path!r}, f"lib_rank{{rank}}.npy"), eng.series_global(31))
dist.barrier(); dist.destroy_process_group()
"""


def test_two_gpu_series_allreduce(tmp_path):
    """The series path sharded over 2 GPUs: torch.distributed all-reduce of the whole stretch in the host mirror,
    arianna_series_global inside the library; both equal the single-GPU records."""
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
        script.write_text(_NCCL_SERIES_WORKER.format(root=root, path=str(d)))
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                            "--master-addr", "127.0.0.1", "--master-port", str(29700 + n), str(script)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        outs[n] = (np.concatenate([np.load(d / f"x_rank{k}.npy") for k in range(n)]), np.loadtxt(d / "energy.dat"),
                   [np.load(d / f"lib_rank{k}.npy") for k in range(n)], np.load(d / "launches_rank0.npy")[0])
    assert np.array_equal(outs[2][0], outs[1][0])                               # chains independent of the sharding
    np.testing.assert_allclose(outs[2][1], outs[1][1], rtol=1e-12)              # energy.dat
    assert np.array_equal(outs[2][2][0], outs[2][2][1])                         # every rank holds the global records
    np.testing.assert_allclose(outs[2][2][0], outs[1][2][0], rtol=1e-12)
    assert outs[2][2][0][0, 2] == 100003 and outs[1][3] <= 2 + 2 * 3 + 2        # init + t=0 record + 3 series launches
    M = 100003
    ref = O.Ensemble(O.init_synthetic(7, 0, M), 2.0, [0.1])
    _, z, ua = O.draws_philox(7, 0, M, 0, 400, with_cat=False)
    ref.sweep_replay(None, z, ua)
    assert np.max(np.abs(outs[2][0] - ref.x)) < 1e-12
    assert abs(outs[2][1][-1, 1] / ref.callback_energy() - 1) < 1e-12


def test_config1_verbatim(tmp_path):
    """BASELINE config 1 = example/particle_1d/harmonic_oscillator/MC_harmonic_oscillator.jl verbatim: β = 2, M = 10,
    10^5 steps, burn 1000, σ = 0.1, Metropolis + StoreCallbacks energy/acceptance + StoreTrajectories + StoreLastFrames
    on build_schedule(steps, burn, [0, 10]).  Every one of the 9 902 records must match the stepwise oracle."""
    seed, beta, M, steps, burn = 42, 2.0, 10, 10 ** 5, 1000
    x0 = O.init_synthetic(seed, 0, M)
    chains = [mb.System(x, beta) for x in x0]                      # the reference's `chains` vector
    pool = (mb.Move(mb.Displacement(0.0), mb.StandardGaussian(), mb.ComponentArray(σ=0.1), 1.0),)
    sampletimes = mb.build_schedule(steps, burn, [0, 10])
    algorithm_list = (
        dict(algorithm=mb.Metropolis, pool=pool, seed=seed, parallel=False),
        dict(algorithm=mb.StoreCallbacks, callbacks=(mb.callback_energy, mb.callback_acceptance), scheduler=sampletimes),
        dict(algorithm=mb.StoreTrajectories, scheduler=sampletimes),
        dict(algorithm=mb.StoreLastFrames, scheduler=[steps]),
        dict(algorithm=mb.PrintTimeSteps, scheduler=mb.build_schedule(steps, burn, steps // 10)),
    )
    simulation = mb.Simulation(chains, algorithm_list, steps, path=str(tmp_path), verbose=False)
    mb.run(simulation)
    energies = np.loadtxt(tmp_path / "energy.dat")
    assert energies.shape == (1 + len(sampletimes), 2) and len(sampletimes) == 9901
    ref = O.Ensemble(x0, beta, [0.1])
    want, done = [ref.callback_energy()], 0
    for t in sampletimes:
        _, z, ua = O.draws_philox(seed, 0, M, done, t - done, with_cat=False)
        ref.sweep_replay(None, z, ua)
        done = t
        want.append(ref.callback_energy())
    np.testing.assert_allclose(energies[:, 1], want, rtol=1e-10)
    assert list(energies[:, 0]) == [0] + sampletimes
    trj = np.loadtxt(tmp_path / "trajectories" / "10" / "trajectory.dat")
    assert trj.shape == (1 + len(sampletimes), 2) and abs(trj[-1, 1] - ref.x[9]) < 1e-12
    # the example's own sanity print: mean(energies) ≈ 1/(2β) (10 chains x 9 901 correlated samples: loose window)
    assert abs(energies[1:, 1].mean() - 0.25) < 0.03
    acc = open(tmp_path / "acceptance.dat").read().split("\n")
    assert acc[0] == "0 [NaN]" and abs(float(acc[-2].split("[")[1][:-1]) - ref.callback_acceptance()[0]) < 1e-12


def test_config1_julia_mode_matches_the_prediction(tmp_path, golden_dir):
    """BASELINE config 1 run the way Julia runs it: the initial condition from Xoshiro(42), the chains on the DEVICE
    generator (XOSHIRO mode: Julia's own Xoshiro(seed + c - 1) states, Julia's ziggurat tables) in EXACT arithmetic,
    through the mirror's Simulation / run.  It must land on tests/golden/julia_prediction_config1.json, the oracle's
    prediction of what the real reference writes for its example script: the same number of raw draws consumed by
    every chain (final generator states), the same accept counts, energies to 1e-12."""
    import importlib.util
    import json
    spec = importlib.util.spec_from_file_location("make_julia_prediction", os.path.join(golden_dir, "make_julia_prediction.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    gold = json.load(open(os.path.join(golden_dir, "julia_prediction_config1.json")))
    x0, ens_ref, energy_ref, accept_ref = mod.predict()                     # the full predicted files (2 s of oracle)
    assert energy_ref[:20] == gold["energy_head"] and accept_ref[-5:] == gold["acceptance_tail"]
    seed, beta, steps, burn = gold["seed"], gold["beta"], gold["steps"], gold["burn"]
    chains = mb.ParticleEnsemble(x0, beta, rng="xoshiro", arith="exact")
    pool = (mb.Move(mb.Displacement(0.0), mb.StandardGaussian(), mb.ComponentArray(σ=gold["sigma"]), 1.0),)
    sampletimes = mb.build_schedule(steps, burn, [0, 10])
    algorithm_list = (
        dict(algorithm=mb.Metropolis, pool=pool, seed=seed, parallel=False),
        dict(algorithm=mb.StoreCallbacks, callbacks=(mb.callback_energy, mb.callback_acceptance), scheduler=sampletimes),
    )
    simulation = mb.Simulation(chains, algorithm_list, steps, path=str(tmp_path), verbose=False)
    mb.run(simulation)
    eng = chains.engine
    assert np.array_equal(eng.get_rng_state(), np.array(gold["rng_states_final"], dtype=np.uint64))
    acc, _ = eng.chain_counters()
    assert list(acc[0]) == gold["accepted_calls"]
    x_ref = np.array([float.fromhex(h) for h in gold["x_final_hex"]])
    assert np.max(np.abs(eng.get_state() - x_ref)) < 1e-12
    got = open(tmp_path / "energy.dat").read().split("\n")[:-1]
    assert len(got) == gold["records"] and [ln.split()[0] for ln in got] == [ln.split()[0] for ln in energy_ref]
    e_got = np.array([float(ln.split()[1]) for ln in got])
    e_ref = np.array([float(ln.split()[1]) for ln in energy_ref])
    np.testing.assert_allclose(e_got, e_ref, rtol=1e-12)
    a_got = open(tmp_path / "acceptance.dat").read().split("\n")[:-1]
    assert a_got[0] == "0 [NaN]"
    np.testing.assert_allclose([float(ln.split("[")[1][:-1]) for ln in a_got[1:]],
                               [float(ln.split("[")[1][:-1]) for ln in accept_ref[1:]], rtol=1e-12)


_LIBNCCL_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch, torch.distributed as dist
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
dist.init_process_group("gloo")                      # only used to hand the 128-byte NCCL id around
import montecarlo_b200 as mb
from montecarlo_b200.arianna import shard_bounds
M = 100003
off, n = shard_bounds(M, rank, world)
ids = [mb.CudaEnsemble.nccl_unique_id() if rank == 0 else None]
dist.broadcast_object_list(ids, src=0)
eng = mb.CudaEnsemble(n, 2.0, [0.2, 0.6], [0.5, 0.5], seed=11, chain_offset=off, n_chains_total=M, arith="exact",
                      device=int(os.environ["LOCAL_RANK"]))
eng.comm_init(ids[0], rank, world)
eng.init_synthetic()
eng.sweep(25, reduce=True)
me, ma = eng.callbacks_global()                      # NCCL all-reduce inside libarianna_cuda.so
eng.pgmc_estimate(3, [0, 1])
gd = eng.pgmc_read_global(2)
np.save(os.path.join({path!r}, f"out_rank{{rank}}.npy"), np.concatenate([[me], ma, gd.ravel()]))
eng.close(); dist.barrier(); dist.destroy_process_group()
"""


def test_two_gpu_allreduce_inside_the_library(tmp_path):
    """arianna_comm_init / arianna_callbacks_global / arianna_pgmc_read_global: the NCCL path a Julia host would use."""
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "worker.py"
    script.write_text(_LIBNCCL_WORKER.format(root=root, path=str(tmp_path)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29650", str(script)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    a, b = (np.load(tmp_path / f"out_rank{k}.npy") for k in range(2))
    assert np.array_equal(a, b)                                   # every rank holds the ensemble-wide values
    M = 100003
    with mb.CudaEnsemble(M, 2.0, [0.2, 0.6], [0.5, 0.5], seed=11, arith="exact") as eng:   # one GPU, whole ensemble
        eng.init_synthetic()
        eng.sweep(25, reduce=True)
        me, ma = eng.callbacks_global()                           # no communicator: equals the local call
        eng.pgmc_estimate(3, [0, 1])
        want = np.concatenate([[me], ma, eng.pgmc_read(2).ravel()])
    np.testing.assert_allclose(a, want, rtol=1e-12)


def test_replay_host_staging_is_chunked_over_steps(monkeypatch):
    """Host-pointer replay streams the draws through a bounded device buffer: force 3-step chunks."""
    M, K = 2049, 20
    monkeypatch.setenv("ARIANNA_REPLAY_STAGE_BYTES", str(3 * 8 * M))
    x0 = O.init_synthetic(4, 0, M)
    uc, z, ua = _xoshiro_draws(x0, 2.0, [0.2, 0.7], [0.3, 0.7], K)
    ref = O.Ensemble(x0, 2.0, [0.2, 0.7], [0.3, 0.7])
    dref, _, _ = ref.sweep_replay(uc, z, ua, want_decisions=True)
    with mb.CudaEnsemble(M, 2.0, [0.2, 0.7], [0.3, 0.7], arith="exact") as eng:
        eng.set_state(x0)
        l0 = eng.launch_count
        dec = eng.sweep_replay(uc, z, ua, want_decisions=True)
        assert eng.launch_count - l0 == 7                          # ceil(20 / 3) launches
        assert np.array_equal(dec, dref) and np.array_equal(eng.get_state(), ref.x)
        assert np.array_equal(eng.chain_counters()[1].astype(np.int64), ref.tot)
