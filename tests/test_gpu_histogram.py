"""GPU tests of the on-device histograms and moments (arianna_set_histogram / _accumulate / _read / _reset): counts
bit-identical to the numpy restatement of the bin rule on every kind of handle, accumulation over time, no side
effects, sharding invariance, agreement with the per-rung ladder sums, the distribution of harmonic chains, argument
errors, the StoreHistograms mirror, and a ledger of the histogram_kernel instantiations."""
import math
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

import montecarlo_b200 as mb
from montecarlo_b200 import _lib as L_
from montecarlo_b200._build import LIB_PATH
from montecarlo_b200.julia_rng import xoshiro_states

from test_histogram_host import bin_cells, inv_width, np_histogram

pytestmark = pytest.mark.gpu

M_ODD = 3 * 4099                      # not a multiple of the 512-thread block
OFFSET = 1003                         # = 17 · 59: no G below divides it
GROUPS = (1, 2, 7, 32, 256)
BINS = 37                             # 256 · (37 + 3) cells fit ARIANNA_MAX_HISTOGRAM_CELLS
RANGES = {"x": (-1.5, 1.7), "e": (0.0, 2.5)}

CASES = [   # dtype, rng, σ per move, potential
    ("f64", "philox", [0.5], "harmonic"),
    ("f64", "philox", [0.5, 0.1, 0.05], "double_well"),
    ("f64", "philox", [0.4], "quartic"),
    ("f64", "xoshiro", [0.5], "quartic"),
    ("f64", "xoshiro", [0.5, 0.2, 0.1], "double_well"),
    ("f32", "philox", [0.5], "harmonic"),
    ("f32", "philox", [0.5], "quartic"),
    ("f32", "philox", [0.5], "double_well"),
]


def _engine(dtype, rng, sigma, pot, M=M_ODD, offset=OFFSET, seed=9):
    eng = mb.CudaEnsemble(M, 1.5, sigma, seed=seed, chain_offset=offset, n_chains_total=M + offset + 17,
                          potential=pot, rng=rng, dtype=dtype)
    if rng == "xoshiro":
        eng.set_rng_state(xoshiro_states(np.arange(seed + offset, seed + offset + M, dtype=np.int64)))
    return eng


def _values(eng, obs):
    """What the accumulate sees, restated from get_state / get_state_f32 (F32: the Float32 values, widened)."""
    if eng.dtype == "f32":
        x, e = eng.get_state_f32(with_energy=True)
        return (x if obs == "x" else e).astype(np.float64)
    x, e = eng.get_state(with_energy=True)
    return x if obs == "x" else e


def _crafted(M, lo, hi, n, f32, rng):
    """lo, hi, every nominal edge, ±0, ±inf, NaN, subnormals, values just below hi that bin to n (overflow), random rest."""
    inv_w = inv_width(lo, hi, n)
    special = [lo, hi, 0.0, -0.0, np.inf, -np.inf, np.nan, 5e-324, -5e-324, 2.2250738585072014e-308,
               np.nextafter(lo, -np.inf), np.nextafter(hi, np.inf)]
    special += [lo + k * (hi - lo) / n for k in range(n + 1)]
    x = np.nextafter(hi, -np.inf)
    for _ in range(64):                                     # (v − lo)·inv_w rounds up to n although v < hi
        if (x - lo) * inv_w >= n:
            special.append(x)
        x = np.nextafter(x, -np.inf)
    v = rng.uniform(lo - 0.3, hi + 0.3, M)
    if f32:
        special += [np.float32(1e-45), np.float32(-1e-45), np.float32(1.1754942e-38)]
    v[:len(special)] = special
    v[len(special):2 * len(special)] = special              # twice, in other groups
    return v.astype(np.float32) if f32 else v


def _check(eng, obs, lo, hi, n, G, offset, samples):
    """Counts bit-identical to the numpy restatement; n exact; Σv and Σv² within 1e-12 of math.fsum (relative to Σ|.|)."""
    counts, mom, k = eng.histogram()
    want = np.zeros((G, n + 3), np.int64)
    per_group = [[] for _ in range(G)]
    for v in samples:
        grp = (offset + np.arange(v.size)) % G
        want += np.bincount(grp * (n + 3) + bin_cells(v, lo, hi, n), minlength=G * (n + 3)).reshape(G, n + 3)
        fin = np.isfinite(v)
        order = np.argsort(grp[fin], kind="stable")
        bounds = np.searchsorted(grp[fin][order], np.arange(G + 1))
        vf = v[fin][order]
        for g in range(G):
            per_group[g].append(vf[bounds[g]:bounds[g + 1]])
    assert k == len(samples)
    assert np.array_equal(counts, want), np.argwhere(counts != want)[:5]
    vals = [np.concatenate(p) for p in per_group]
    assert np.array_equal(mom[:, 0], [a.size for a in vals])
    for g, a in enumerate(vals):
        for q, w in ((1, a), (2, a * a)):
            ref = math.fsum(w)
            assert abs(mom[g, q] - ref) <= 1e-12 * math.fsum(np.abs(w)), (g, q, mom[g, q], ref)


@pytest.mark.parametrize("obs", ["x", "e"])
@pytest.mark.parametrize("dtype,rng,sigma,pot", CASES)
def test_counts_equal_the_numpy_restatement(dtype, rng, sigma, pot, obs):
    lo, hi = RANGES[obs]
    g = np.random.default_rng(len(sigma) * 7 + len(pot))
    with _engine(dtype, rng, sigma, pot) as eng:
        eng.init_synthetic()
        eng.sweep(20)
        for G in GROUPS:                                    # the chains after Metropolis steps
            eng.set_histogram(obs, lo, hi, BINS, G)
            eng.histogram_accumulate()
            _check(eng, obs, lo, hi, BINS, G, OFFSET, [_values(eng, obs)])
        crafted = _crafted(M_ODD, *RANGES["x"], BINS, dtype == "f32", g)
        if dtype == "f32":
            eng.set_state_f32(crafted)
        else:
            eng.set_state(crafted)
        v = _values(eng, obs)
        assert np.isnan(v).any() and np.isinf(v).any()
        for G in GROUPS:                                    # crafted states: edges, specials, round-up to n_bins
            eng.set_histogram(obs, *RANGES["x"], BINS, G)
            eng.histogram_accumulate()
            _check(eng, obs, *RANGES["x"], BINS, G, OFFSET, [v])
            if obs == "x" and G == 1:
                c = eng.histogram()[0][0]
                assert c[BINS] > 0 and c[BINS + 1] > 0 and c[BINS + 2] > 0 and c[0] > 0


@pytest.mark.parametrize("dtype", ["f64", "f32"])
def test_counts_equal_the_numpy_restatement_at_full_grid(dtype):
    """M far above the 8 loads per thread of one resident wave (2 × 148 CTAs × 512 threads on a B200): every thread runs
    the unrolled loop and the tail over many chains of ONE group, so the group of the 2nd, 3rd, ... chain of a thread,
    the per-thread runs and moments over many chains, and the flush of every CTA of the wave are all compared exactly.
    States: after Metropolis steps (broad), every chain at 0 (one cell per group), and a few-bin state."""
    M, offset = 3 * (1 << 20) + 1001, 1003
    with mb.CudaEnsemble(M, 1.5, [0.5], seed=3, chain_offset=offset, n_chains_total=M + offset, potential="double_well",
                         dtype=dtype) as eng:
        assert M > 8 * 2 * eng.device_info()["sm_count"] * 512
        eng.init_synthetic()
        eng.sweep(30)
        few = np.random.default_rng(5).choice([-1.0, 0.25, 0.3, 1.0], M)
        for state in ("broad", "zeros", "few"):
            if state == "zeros":
                eng.set_state(np.zeros(M))
            elif state == "few":
                eng.set_state(few)
            for obs in ("x", "e"):
                lo, hi = RANGES[obs]
                v = _values(eng, obs)
                for G in (1, 7, 32, 256):
                    eng.set_histogram(obs, lo, hi, BINS, G)
                    eng.histogram_accumulate()
                    eng.histogram_accumulate()                  # twice: the counts accumulate
                    _check(eng, obs, lo, hi, BINS, G, offset, [v, v])


def test_accumulation_over_time_reset_and_replace():
    lo, hi, n, G = -1.0, 1.0, 50, 7
    with _engine("f64", "philox", [0.3], "harmonic") as eng:
        eng.init_synthetic()
        eng.set_histogram("x", lo, hi, n, G)
        samples = []
        for step in (lambda: eng.sweep(5), lambda: eng.sweep_series([3, 4]), lambda: eng.sweep(2, reduce=True),
                     lambda: None, lambda: eng.sweep_series([1, 1, 6], read=False)):
            step()
            eng.histogram_accumulate()
            samples.append(_values(eng, "x"))
        _check(eng, "x", lo, hi, n, G, OFFSET, samples)
        eng.histogram_reset()
        c, m, k = eng.histogram()
        assert k == 0 and not c.any() and not m.any() and c.shape == (G, n + 3)
        eng.histogram_accumulate()
        _check(eng, "x", lo, hi, n, G, OFFSET, samples[-1:])
        eng.set_histogram("e", 0.0, 0.5, 11, 3)             # replaces the binning and zeroes the accumulators
        c, m, k = eng.histogram()
        assert c.shape == (3, 14) and k == 0 and not c.any()
        eng.histogram_accumulate()
        _check(eng, "e", 0.0, 0.5, 11, 3, OFFSET, [_values(eng, "e")])


def test_no_side_effects():
    L = 8
    with _engine("f64", "philox", [0.4, 0.1, 0.05], "double_well", M=8 * 2048, offset=8 * 3) as eng:
        eng.init_synthetic()
        eng.set_ladder(np.geomspace(0.5, 4.0, L))
        eng.sweep(7)
        eng.replica_exchange()
        rec = eng.sweep_series([3, 5], read=False)
        assert rec is None

        def snapshot():
            return [eng.get_state(), *eng.chain_counters(), np.array([eng.steps_done]),
                    np.array([eng.get_params(k) for k in range(3)]), np.array([eng.callbacks()[0]]),
                    eng.callbacks()[1], eng.series_global(2), eng.ladder_sums(), eng.exchange_counters()[0]]
        before = snapshot()
        n0 = eng.launch_count
        eng.set_histogram("e", 0.0, 3.0, 64, L)
        eng.histogram_accumulate()
        eng.histogram_accumulate()
        assert eng.launch_count == n0 + 4                   # at most 2 launches per accumulate
        after = snapshot()
        for a, b in zip(before, after):
            assert a.tobytes() == b.tobytes()
    with _engine("f32", "philox", [0.5], "harmonic") as eng:
        eng.init_synthetic()
        eng.sweep(5)
        x0 = eng.get_state_f32()
        me = eng.callbacks()
        eng.set_histogram("x", -2.0, 2.0, 10)
        eng.histogram_accumulate()
        assert eng.get_state_f32().tobytes() == x0.tobytes() and eng.callbacks()[0] == me[0]


def test_sharding_invariance():
    M, G, cut, lo, hi, n = 20000, 7, 9001, -1.2, 1.2, 90

    def run(off, m):
        with mb.CudaEnsemble(m, 1.0, [0.4], seed=5, chain_offset=off, n_chains_total=M, potential="quartic") as eng:
            eng.init_synthetic()
            eng.set_histogram("x", lo, hi, n, G)
            for K in (4, 9, 1):
                eng.sweep(K)
                eng.histogram_accumulate()
            return eng.histogram()
    c, m, k = run(0, M)
    ca, ma, _ = run(0, cut)
    cb, mb_, _ = run(cut, M - cut)
    assert k == 3 and c.sum() == 3 * M
    assert np.array_equal(ca + cb, c)
    assert np.array_equal(ma[:, 0] + mb_[:, 0], m[:, 0])
    np.testing.assert_allclose(ma + mb_, m, rtol=1e-12)


def test_energy_moments_equal_the_ladder_sums():
    L, M = 16, 16 * 4096
    with mb.CudaEnsemble(M, 1.0, [0.3], seed=4, potential="double_well") as eng:
        eng.init_synthetic()
        eng.set_ladder(np.geomspace(0.25, 8.0, L))
        for _ in range(12):
            eng.sweep(10)
            eng.replica_exchange()
        assert eng.exchange_counters()[0].sum() > 0
        eng.set_histogram("e", 0.0, 4.0, 100, L)
        eng.histogram_accumulate()
        _, mom, _ = eng.histogram()
        s = eng.ladder_sums()
    assert np.array_equal(mom[:, 0], s[:, -1])
    np.testing.assert_allclose(mom[:, 1], s[:, 0], rtol=1e-12)


def test_harmonic_distribution():
    from scipy import stats
    M, beta, lo, hi, n = 1 << 22, 2.0, -2.5, 2.5, 50
    sd = math.sqrt(1 / (2 * beta))
    with mb.CudaEnsemble(M, beta, [1.0], seed=21) as eng:
        eng.init_synthetic()
        eng.sweep(2000)
        eng.set_histogram("x", lo, hi, n)
        eng.histogram_accumulate()
        c, m, _ = eng.histogram()
    c = c[0]
    assert c[n + 2] == 0 and c.sum() == M
    edges = np.array([lo + k * (hi - lo) / n for k in range(n + 1)])
    p = np.diff(stats.norm.cdf(edges, scale=sd))
    obs = np.concatenate([c[:n], [c[n] + c[n + 1]]])
    exp = M * np.concatenate([p, [1 - p.sum()]])
    keep = exp >= 5
    chi2 = (((obs - exp) ** 2 / exp)[keep]).sum() + (obs[~keep].sum() - exp[~keep].sum()) ** 2 / max(exp[~keep].sum(), 1)
    dof = int(keep.sum())
    assert stats.chi2.sf(chi2, dof) > 1e-4, (chi2, dof)
    cnt, s1, s2 = m[0]
    mean = s1 / cnt
    var = s2 / cnt - mean * mean
    assert cnt == M
    assert abs(mean) < 3 * sd / math.sqrt(M)
    assert abs(math.sqrt(var) - sd) < 3 * sd / math.sqrt(2 * M)


def test_errors_leave_the_handle_usable():
    with mb.CudaEnsemble(1000, 1.0, [0.4]) as eng:
        codes = []
        for fn in (eng.histogram_accumulate, eng.histogram, eng.histogram_reset):   # before set
            with pytest.raises(mb.AriannaError) as e:
                fn()
            codes.append(e.value.code)
        bad = [(2, -1.0, 1.0, 10, 1), ("v", -1.0, 1.0, 10, 1), ("x", -1.0, 1.0, 0, 1), ("x", -1.0, 1.0, 10, 0), ("x", -1.0, 1.0, 10, 257),
               ("x", -1.0, 1.0, 16382, 1), ("x", -1.0, 1.0, 509, 33), ("x", np.nan, 1.0, 10, 1),
               ("x", -1.0, np.inf, 10, 1), ("x", 1.0, 1.0, 10, 1), ("x", 1.0, -1.0, 10, 1),
               ("x", 0.0, 1e-320, 10, 1),                   # inv_w overflows
               ("x", -1e308, 1e308, 10, 1)]                 # hi − lo overflows: inv_w = 0
        for i, args in enumerate(bad):
            with pytest.raises(mb.AriannaError) as e:
                eng.set_histogram(*args)
            codes.append(e.value.code)
            if i == 4:                                      # a valid set in between: a failed set keeps it
                eng.set_histogram("x", -1.0, 1.0, 16381, 1)
        assert codes == [L_.ERR_INVALID] * len(codes)
        eng.histogram_accumulate()
        c, _, k = eng.histogram()
        assert k == 1 and c.shape == (1, 16384) and c.sum() == 1000
        eng.set_histogram("x", -1.0, 1.0, 509, 32)          # 32 · 512 = the cell limit
        n0 = eng.launch_count
        eng.histogram_accumulate()
        assert eng.launch_count == n0 + 2
        assert eng.histogram()[0].sum() == 1000


def _mirror(path, M, steps, lookahead=True):
    chains = mb.ParticleEnsemble(n_chains=M, beta=1.0, potential="double_well")
    pool = (mb.Move(mb.Displacement(0.0), mb.StandardGaussian(), mb.ComponentArray(σ=0.4), 1.0),)
    sim = mb.Simulation(chains, (
        dict(algorithm=mb.Metropolis, pool=pool, seed=13),
        dict(algorithm=mb.StoreCallbacks, callbacks=(mb.callback_energy, mb.callback_acceptance),
             scheduler=list(range(0, steps + 1, 5))),
        dict(algorithm=mb.StoreHistograms, observable="x", range=(-2.0, 2.0), bins=40, groups=5,
             scheduler=list(range(0, steps + 1, 20))),
        dict(algorithm=mb.StoreTrajectories, scheduler=list(range(20, steps + 1, 20)), store_first=False),
    ), steps, path=str(path))
    sim.lookahead = lookahead
    mb.run(sim)
    return chains, sim


def test_through_the_mirror(tmp_path):
    M, steps = 3 * 4096 + 5, 100
    chains, sim = _mirror(tmp_path / "look", M, steps)
    plain, psim = _mirror(tmp_path / "plain", M, steps, lookahead=False)
    hist = sim.algorithms[2]
    t, frames = mb.StoreTrajectories.read_binary(str(tmp_path / "look" / "trajectories" / "rank0.bin"), M)
    assert t.tolist() == [20, 40, 60, 80, 100]
    want = sum(np_histogram(x, -2.0, 2.0, 40, 5)[0] for x in frames)
    assert np.array_equal(hist.counts, want) and hist.samples == 5
    body = [ln for ln in open(tmp_path / "look" / "histogram_x.dat").read().split("\n")[:-1] if not ln.startswith("#")]
    assert [[int(v) for v in ln.split()[2:]] for ln in body[:40]] == want[:, :40].T.tolist()
    assert open(tmp_path / "look" / "histogram_x.dat").read() == open(tmp_path / "plain" / "histogram_x.dat").read()
    # the four callback-only stores of every 20-step stretch run as ONE series call: fewer launches than per-store sweeps
    assert chains.engine.launch_count <= plain.engine.launch_count - steps // 20, \
        (chains.engine.launch_count, plain.engine.launch_count)
    np.testing.assert_allclose(np.loadtxt(tmp_path / "look" / "energy.dat"), np.loadtxt(tmp_path / "plain" / "energy.dat"),
                               rtol=1e-12)


_NCCL_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch, torch.distributed as dist
rank = int(os.environ["RANK"]); torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
import montecarlo_b200 as mb
M, steps = 16 * 4096 + 3, 200
chains = mb.ParticleEnsemble(n_chains=M, beta=1.0, potential="double_well")
pool = (mb.Move(mb.Displacement(0.0), mb.StandardGaussian(), mb.ComponentArray(σ=0.3), 1.0),)
sim = mb.Simulation(chains, (dict(algorithm=mb.Metropolis, pool=pool, seed=7),
                             dict(algorithm=mb.StoreHistograms, observable="e", range=(0.0, 2.0), bins=64, groups=7,
                                  scheduler=list(range(25, steps + 1, 25)))),
                    steps, path={path!r})
mb.run(sim)
dist.barrier(); dist.destroy_process_group()
"""


def test_two_gpu_histogram_matches_one_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    files = {}
    for n in (1, 2):
        d = tmp_path / f"n{n}"
        d.mkdir()
        script = d / "worker.py"
        script.write_text(_NCCL_WORKER.format(root=root, path=str(d)))
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                            "--master-addr", "127.0.0.1", "--master-port", str(29800 + n), str(script)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        files[n] = open(d / "histogram_e.dat").read().split("\n")
    for a, b in zip(files[1], files[2]):
        if a.startswith("moments"):
            assert a.split()[:2] == b.split()[:2]
            np.testing.assert_allclose([float(v) for v in b.split()[2:]], [float(v) for v in a.split()[2:]], rtol=1e-12)
        else:
            assert a == b                                   # counts: int64 all-reduce, exact
    assert len(files[1]) == len(files[2])


# ---- ledger of the histogram kernel family ------------------------------------------------------------------------
COUNTS = "counts bit-identical to the numpy restatement; moments within 1e-12 of math.fsum"
ALL = "test_gpu_histogram::test_counts_equal_the_numpy_restatement"
FULL = "test_gpu_histogram::test_counts_equal_the_numpy_restatement_at_full_grid"
HIST_LEDGER = {   # histogram_kernel<element type, SRC>: SRC -1 the position, 0 / 1 / 2 the harmonic / quartic / double-well energy
    "histogram_kernel<double, -1>": ((ALL, FULL, "test_gpu_histogram::test_through_the_mirror"), COUNTS),
    "histogram_kernel<double, 0>": ((ALL, "test_gpu_histogram::test_accumulation_over_time_reset_and_replace"), COUNTS),
    "histogram_kernel<double, 1>": ((ALL,), COUNTS),
    "histogram_kernel<double, 2>": ((ALL, FULL, "test_gpu_histogram::test_energy_moments_equal_the_ladder_sums"), COUNTS),
    "histogram_kernel<float, -1>": ((ALL, FULL, "test_gpu_histogram::test_no_side_effects"), COUNTS),
    "histogram_kernel<float, 0>": ((ALL,), COUNTS),
    "histogram_kernel<float, 1>": ((ALL,), COUNTS),
    "histogram_kernel<float, 2>": ((ALL, FULL), COUNTS),
}


def test_every_histogram_kernel_instantiation_has_a_ledger_row():
    if shutil.which("nm") is None:
        pytest.skip("nm (binutils) is not installed")
    out = subprocess.run(["nm", "-C", LIB_PATH], capture_output=True, text=True, check=True).stdout
    found = {f"histogram_kernel<{m.group(1)}>" for m in re.finditer(r"\bhistogram_kernel<([^<>]*)>\(", out)}
    assert found == set(HIST_LEDGER), (sorted(found), sorted(HIST_LEDGER))
    names = set(re.findall(r"^def (test_\w+)", open(__file__).read(), flags=re.M))
    for kernel, (tests, bar) in HIST_LEDGER.items():
        assert bar == COUNTS and tests, kernel
        for t in tests:
            assert t.split("::")[1] in names, (kernel, t)
