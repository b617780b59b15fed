"""CPU tests of the on-device histograms: the numpy restatement of the bin rule, argument errors of the C ABI without a
device, the StoreHistograms file format and its int64 all-reduce over an oracle-backed test double (one process and
two gloo ranks write identical files), the look-ahead around histogram times, and the Julia shim's bindings."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import montecarlo_b200 as mb
from montecarlo_b200 import _lib as L
from montecarlo_b200 import arianna as A
from oracle import oracle as O

from fake_engine import OracleEngine
import test_julia_shim_abi as SHIM

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- the bin rule, restated -------------------------------------------------------------------------------------
def inv_width(lo, hi, n_bins):
    return np.float64(n_bins) / (np.float64(hi) - np.float64(lo))


def bin_cells(v, lo, hi, n_bins):
    """Cell of every value: floor((v − lo)·inv_w) in binary64 (two IEEE operations, numpy never contracts them); NaN ->
    n_bins + 2, k < 0 -> n_bins (underflow), k >= n_bins -> n_bins + 1 (overflow)."""
    v = np.asarray(v, dtype=np.float64)
    with np.errstate(all="ignore"):
        k = np.floor((v - np.float64(lo)) * inv_width(lo, hi, n_bins))
    cell = np.where(np.isnan(k), n_bins + 2, np.where(k < 0, n_bins, np.where(k >= n_bins, n_bins + 1, k)))
    return cell.astype(np.int64)


def np_histogram(v, lo, hi, n_bins, groups=1, offset=0):
    """(counts int64 [groups][n_bins + 3], moments [groups][3] = (n, fsum v, fsum v²) over the finite v) of one sample
    of the chains offset, offset + 1, ... (chain g in group g % groups)."""
    v = np.asarray(v, dtype=np.float64)
    grp = (offset + np.arange(v.size, dtype=np.int64)) % groups
    cells = n_bins + 3
    counts = np.bincount(grp * cells + bin_cells(v, lo, hi, n_bins), minlength=groups * cells).reshape(groups, cells)
    moments = np.zeros((groups, 3))
    fin = np.isfinite(v)
    for g in range(groups):
        s = v[fin & (grp == g)]
        with np.errstate(over="ignore"):
            moments[g] = (s.size, math.fsum(s), math.fsum(s * s))
    return counts.astype(np.int64), moments


def test_bin_rule_edges():
    lo, hi, n = -1.0, 2.0, 3
    v = np.array([-1.0, 2.0, 0.0, -0.0, 1.0, np.nextafter(-1.0, -2), np.nextafter(2.0, 3), np.inf, -np.inf, np.nan,
                  5e-324, -5e-324])
    assert bin_cells(v, lo, hi, n).tolist() == [0, 4, 1, 1, 2, 3, 1 + 3, 4, 3, 5, 1, 1]
    # a value just below hi whose (v − lo)·inv_w rounds up to n_bins lands in overflow, as the formula says
    lo, hi, n = -1.0, 0.1, 11
    below = np.nextafter(np.nextafter(hi, 0), 0)
    assert below < hi and (below - lo) * inv_width(lo, hi, n) == n
    assert bin_cells([below], lo, hi, n).tolist() == [n + 1]
    c, m = np_histogram([1.0, np.nan, np.inf, 2.0, 3.0], 0.0, 4.0, 4, groups=2, offset=1)
    assert c.tolist() == [[0, 0, 1, 0, 0, 0, 1], [0, 1, 0, 1, 0, 1, 0]]
    assert m.tolist() == [[1.0, 2.0, 4.0], [2.0, 4.0, 10.0]]


def test_null_handle_is_invalid_without_a_device():
    lib = L.load()
    assert lib.arianna_set_histogram(None, 0, -1.0, 1.0, 10, 1) == L.ERR_INVALID
    assert lib.arianna_histogram_accumulate(None) == L.ERR_INVALID
    assert lib.arianna_histogram_read(None, None, None, None) == L.ERR_INVALID
    assert lib.arianna_histogram_reset(None) == L.ERR_INVALID
    assert L.MAX_HISTOGRAM_CELLS == 16384
    hdr = open(os.path.join(ROOT, "include", "arianna_cuda.h")).read()
    assert "#define ARIANNA_MAX_HISTOGRAM_CELLS 16384" in hdr and "ARIANNA_OBS_E = 1" in hdr


def test_shim_binds_the_histogram_calls():
    calls = {c[0]: c for c in SHIM.julia_ccalls(SHIM.SHIM)}
    for name in ("arianna_set_histogram", "arianna_histogram_accumulate", "arianna_histogram_read",
                 "arianna_histogram_reset"):
        assert name in calls, name
    assert calls["arianna_histogram_read"][2] == ["Ptr{Cvoid}", "Ptr{Int64}", "Ptr{Float64}", "Ref{Int64}"]
    src = open(SHIM.SHIM).read()
    for fn in ("set_histogram!", "accumulate_histogram!", "histogram"):
        assert f"function {fn}(" in src, fn


# ---- the host mirror over an oracle-backed engine ----------------------------------------------------------------
class HistogramEngine(OracleEngine):
    """OracleEngine + the histogram entry points, restated with numpy."""

    def set_histogram(self, observable, lo, hi, n_bins, n_groups=1):
        self.hist = (observable, float(lo), float(hi), int(n_bins), int(n_groups))
        self.histogram_reset()

    def histogram_reset(self):
        _, _, _, n, G = self.hist
        self.h_counts, self.h_moments, self.h_samples = np.zeros((G, n + 3), np.int64), np.zeros((G, 3)), 0

    def histogram_accumulate(self):
        obs, lo, hi, n, G = self.hist
        c, m = np_histogram(self.ens.x if obs == "x" else self.ens.e, lo, hi, n, G, self.chain_offset)
        self.h_counts += c
        self.h_moments += m
        self.h_samples += 1
        self.launch_count += 2

    def histogram(self):
        return self.h_counts.copy(), self.h_moments.copy(), self.h_samples


@pytest.fixture
def histogram_engine(monkeypatch):
    monkeypatch.setattr(A, "CudaEnsemble", HistogramEngine)


POOL = lambda: (mb.Move(mb.Displacement(0.0), mb.StandardGaussian(), mb.ComponentArray(σ=0.5), 1.0),)   # noqa: E731


def _sim(path, M=30, steps=60, observable="x", groups=3, lookahead=True, traj=True):
    chains = mb.ParticleEnsemble(O.init_synthetic(3, 0, M), 1.5, potential="double_well")
    hist_times = list(range(0, steps + 1, 15))                      # t = 0 is not sampled (no store_first)
    algs = [dict(algorithm=mb.Metropolis, pool=POOL(), seed=3),
            dict(algorithm=mb.StoreCallbacks, callbacks=(mb.callback_energy, mb.callback_acceptance),
                 scheduler=list(range(0, steps + 1, 5))),
            dict(algorithm=mb.StoreHistograms, observable=observable, range=(-2.0, 2.0), bins=16, groups=groups,
                 scheduler=hist_times)]
    if traj:
        algs.append(dict(algorithm=mb.StoreTrajectories, scheduler=hist_times, store_first=False))
    sim = mb.Simulation(chains, tuple(algs), steps, path=str(path))
    sim.lookahead = lookahead
    return chains, sim


@pytest.mark.parametrize("observable", ["x", "e"])
def test_file_equals_the_histogram_of_the_trajectory_frames(tmp_path, histogram_engine, observable):
    chains, sim = _sim(tmp_path, observable=observable)
    mb.run(sim)
    hist = sim.algorithms[2]
    t, frames = mb.StoreTrajectories.read_binary(str(tmp_path / "trajectories" / "rank0.bin"), 30)
    assert t.tolist() == [15, 30, 45, 60]
    want_c, want_m = np.zeros((3, 19), np.int64), np.zeros((3, 3))
    for x in frames:
        v = x if observable == "x" else O.Ensemble(x, 1.5, [0.5], potential=O.POT_DOUBLE_WELL).e
        c, m = np_histogram(v, -2.0, 2.0, 16, 3)
        want_c += c
        want_m += m
    assert np.array_equal(hist.counts, want_c) and hist.samples == 4
    np.testing.assert_allclose(hist.moments, want_m, rtol=1e-14)
    lines = open(tmp_path / f"histogram_{observable}.dat").read().split("\n")[:-1]
    assert lines[1] == "# lo = -2.0, hi = 2.0, bins = 16, groups = 3, samples = 4"
    body = [ln for ln in lines if not ln.startswith("#")]
    assert len(body) == 16 + 3 + 3
    assert body[0] == "-2.0 -1.75 " + " ".join(str(c) for c in want_c[:, 0])
    assert body[15].startswith("1.75 2.0 ")
    assert [ln.split()[0] for ln in body[16:]] == ["underflow", "overflow", "nan"] + ["moments"] * 3
    assert body[18] == "nan 0 0 0"
    for g, ln in enumerate(body[19:]):
        assert ln == f"moments {int(hist.moments[g, 0])} {A._jl(hist.moments[g, 1])} {A._jl(hist.moments[g, 2])}"
        assert int(ln.split()[1]) == 4 * 10                          # 30 chains in 3 groups, 4 samples
    assert "\tStoreHistograms\n\t\tCalls: 4\n\t\tObservable: " + observable + "\n\t\tRange: [-2.0, 2.0]\n\t\tBins: 16\n" \
        "\t\tGroups: 3\n" in open(tmp_path / "summary.log").read()


def test_histogram_times_are_lookahead_barriers(tmp_path, histogram_engine):
    """Callback-only stores between histogram times still run as series calls; files equal those without look-ahead."""
    ca, sa = _sim(tmp_path / "look", traj=False)
    plan = A._make_lookahead(sa)
    mb.run(sa)
    cb, sb = _sim(tmp_path / "plain", traj=False, lookahead=False)
    mb.run(sb)
    for name in ("energy.dat", "acceptance.dat", "histogram_x.dat"):
        assert open(tmp_path / "look" / name).read() == open(tmp_path / "plain" / name).read(), name
    assert ca.engine.series_calls >= 4 and ca.engine.launch_count < cb.engine.launch_count
    for t, want in ((5, [5, 5]), (15, []), (16, [4, 5, 5]), (55, [5])):
        sa.t = t
        assert plan() == want, t


def test_arguments_are_checked_before_the_run(tmp_path, histogram_engine):
    for bad in (dict(observable="v", range=(0, 1), bins=4), dict(range=(0, 1)), dict(bins=4)):
        chains = mb.ParticleEnsemble(np.zeros(8), 1.0)
        with pytest.raises((ValueError, TypeError)):
            mb.Simulation(chains, (dict(algorithm=mb.Metropolis, pool=POOL()),
                                   dict(algorithm=mb.StoreHistograms, **bad)), 10, path=str(tmp_path))


_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
import numpy as np, torch.distributed as dist
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=int(sys.argv[2]))
import montecarlo_b200 as mb
from montecarlo_b200 import arianna as A
from test_histogram_host import HistogramEngine, _sim
import pathlib
A.CudaEnsemble = HistogramEngine
chains, sim = _sim(pathlib.Path({path!r}), M={M}, observable="e", groups=4, traj=False)
mb.run(sim)
h = sim.algorithms[2]
assert h.counts.dtype == np.int64
np.save(os.path.join({path!r}, f"counts_rank{{chains.rank}}.npy"), h.counts)
dist.barrier(); dist.destroy_process_group()
"""


def _gloo_run(path, world, M=30):
    port = 29500 + (os.getpid() + 11 * world + 977) % 2000
    path.mkdir()
    script = path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT, port=port, path=str(path), M=M))
    procs = [subprocess.Popen([sys.executable, str(script), str(r), str(world)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT) for r in range(world)]
    outs = [p.communicate(timeout=240)[0].decode() for p in procs]
    return [p.returncode for p in procs], outs


def test_two_gloo_ranks_write_the_one_rank_file(tmp_path):
    """Shards of 15 chains each: rank 1 starts at chain 15, not a multiple of the 4 groups.  Everything but the moment
    sums is byte-identical (the counts are all-reduced as int64); Σv and Σv² are split across ranks, so they agree to
    the rounding of the split sums."""
    rc1, o1 = _gloo_run(tmp_path / "n1", 1)
    rc2, o2 = _gloo_run(tmp_path / "n2", 2)
    assert rc1 == [0] and rc2 == [0, 0], "\n".join(o1 + o2)
    a = open(tmp_path / "n1" / "histogram_e.dat").read().split("\n")
    b = open(tmp_path / "n2" / "histogram_e.dat").read().split("\n")
    assert len(a) == len(b) == 4 + 16 + 3 + 4 + 1
    for la, lb in zip(a, b):
        if la.startswith("moments"):
            fa, fb = la.split(), lb.split()
            assert fa[:2] == fb[:2]                                   # n: exact
            np.testing.assert_allclose([float(v) for v in fb[2:]], [float(v) for v in fa[2:]], rtol=1e-13)
        else:
            assert la == lb
    c1 = np.load(tmp_path / "n1" / "counts_rank0.npy")
    assert np.array_equal(np.load(tmp_path / "n2" / "counts_rank1.npy"), c1) and c1.sum() == 4 * 30
