"""bench.py's JSON contract on a real GPU, at a reduced size (the driver runs the default size)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--log2-chains", "22", "--steps", "25",
                          "--warmup", "3", "--ref-log2-chains", "12", "--cpu-seconds", "1", *extra], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    def strict(name):                    # Python's json would accept NaN / Infinity; a strict parser does not
        raise AssertionError(f"bench.py printed the non-JSON constant {name}")
    return json.loads(out.stdout.strip().splitlines()[-1], parse_constant=strict)


@pytest.mark.parametrize("series", ["0", "1"])
def test_bench_line_contract(series):
    d = _run("--series", series)
    assert d["metric"] == "metropolis_chain_steps_per_sec" and d["unit"] == "chain-steps/s"
    assert d["n_gpus"] == 1 and d["steps"] == 25 and d["warmup"] == 3 and d["higher_is_better"] is True
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert "C3" in d["config"]["workload"] and d["config"]["chains_per_gpu"] == 1 << 22
    assert d["value"] > 1e10 and abs(d["value"] - (1 << 22) * 10 * 25 / (d["ms_per_step"] * 25e-3)) < 1e-6 * d["value"]
    assert d["gpu_launches"] >= 25 // max(1, d["engine"]["stores_per_launch"])
    assert "stores_per_launch" not in d["config"] and sum(d["engine"]["launch_plan"]) == 25
    assert d["roofline"]["kernel_launches_averaged"] >= 2
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    r = d["roofline"]
    assert r["bound"] in ("fp64", "hbm", "tensor") and r["unit"] == "TFLOP/s" and "traffic" in r
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0.2 < r["frac"] < 2.0
    assert abs(r["hbm"]["frac"] - r["hbm"]["achieved"] / r["hbm"]["peak"]) < 1e-9
    e = d["e2e"]
    assert e["unit"] == d["unit"] and 0 < e["value"] <= 1.3 * d["value"]      # (tiny job: timing noise)
    assert e["h2d_bytes_per_step"] >= 8 * (1 << 22) // 25 and e["d2h_bytes_per_step"] == 24
    w = e["with_final_state_download"]
    assert 0 < w["value"] <= 1.3 * d["value"] and w["d2h_bytes_per_step"] >= 8 * (1 << 22) // 25
    assert abs(d["mean_energy"] - e["energy"]) < 0.02          # both runs sample the same ensemble a little later
    if series == "0":
        assert e["pcie"]["h2d_gbs"] > 1 and w["pcie"]["d2h_gbs"] > 1 and e["pcie"]["sweep_ms"] > 0
    assert d["strong"]["chains_total"] == 1 << 22 and d["strong"]["value"] == d["value"]
    p = d["parity"]
    assert p["ok"] is True and p["accepted_sums_equal_oracle"] is True and p["energy_sum_max_rel_err_vs_oracle"] <= 1e-12
    assert p["x_bits_checksum_equals_1gpu"] in (True, None)
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["cores"] >= 1 and c["value"] > 0 and c["unit"] == d["unit"] and c["sample"]


def test_bench_dump_outputs_are_reproducible(tmp_path):
    """--dump-outputs writes the timed run's outputs (one record per timed step, a 2^20-chain sample of the final
    state) in float64, under 64 MB; the inputs are seeded, so a second run with the same arguments writes the same."""
    names = ["accepted.npy", "records.npy", "x.npy"]
    dumps = []
    for run in ("a", "b"):
        d = _run("--no-e2e", "--no-strong", "--no-parity", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / run))
        assert sorted(os.listdir(tmp_path / run)) == names
        assert sum(os.path.getsize(tmp_path / run / n) for n in names) <= 64 << 20
        dumps.append({n: np.load(tmp_path / run / n) for n in names})
        rec = dumps[-1]["records.npy"]
        assert rec.shape == (25, 3) and np.all(rec[:, 2] == 1 << 22)           # one record per step of --steps 25
        assert rec[-1, 0] / rec[-1, 2] == d["mean_energy"]
    for n in names:
        assert dumps[0][n].dtype == np.float64 and np.array_equal(dumps[0][n], dumps[1][n]), n
    x, acc = dumps[0]["x.npy"], dumps[0]["accepted.npy"]
    assert x.shape == acc.shape == (1 << 20,) and np.all(np.isfinite(x))
    assert np.all((acc >= 0) & (acc <= 10 * (3 + 25)))         # 3 warm-up + 25 timed intervals of 10 steps
