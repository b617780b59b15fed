"""Coverage ledger of the CUDA kernel templates.  Every instantiation of the sweep, estimator, exchange and replay kernel
templates that `nm -C` finds in libarianna_cuda.so has a row below naming the GPU tests that compare it with an exact
CPU reference (oracle/ or tests/exchange_oracle) and the bar they hold it to.  An instantiation added without such a
row, a row left behind by a removed one, or a row that names a test which no longer exists fails here, on a machine
without a GPU."""
import ast
import os
import re
import shutil
import subprocess

import pytest

from montecarlo_b200._build import LIB_PATH

TESTS = os.path.dirname(os.path.abspath(__file__))

# bars (DESIGN.md §3)
EXACT = "bit-exact: decisions, positions and counters identical to the reference"
NATIVE = "identical accept / total counters, max |dx| < 1e-12, records within rtol 1e-12"
PGMC = "gradient sums within rtol 1e-10, EXACT positions within 1e-13"
RECORDS = "per-rung records within rtol 1e-12"
STATISTICAL = "statistical: 3-sigma averages, loose agreement with the oracle's libm restatement"

# pinning tests, as <module>::<function> under tests/
NAT = "test_gpu_parity::test_philox_native_matches_oracle"
SER = "test_gpu_parity::test_series_equals_per_store_sweeps"
MSER = "test_gpu_parity::test_series_multi_move_pools"
DEV = "test_gpu_parity::test_device_sigma_sweeps_match_oracle"
HOST = "test_gpu_parity::test_host_job_pipelined_over_slices"
XCH = "test_gpu_exchange::test_parity_with_the_oracle"
PGMC_T = "test_gpu_parity::test_pgmc_native_matches_oracle"
PGMC_GOLD = "test_gpu_parity::test_pgmc_replay_matches_oracle"
XOSH = "test_gpu_parity::test_xoshiro_mode_matches_oracle"
REPLAY = "test_gpu_parity::test_replay_bit_exact"
F32_REPLAY = "test_gpu_f32::test_f32_replay_bit_exact"
F32_NAT = "test_gpu_f32::test_f32_native_follows_the_oracle_restatement"
F32_STAT = "test_gpu_f32::test_f32_native_distribution_and_invariance"

# template arguments: POT 0 harmonic, 1 quartic, 2 double well; ARITH 0 EXACT, 1 FAST;
# sweep_philox_kernel<POT, ARITH, SERIES, BETAS>, sweep_multi_kernel<POT, ARITH, BETAS>, pgmc_kernel<POT, ARITH, REPLAY>,
# sweep_xoshiro_kernel<POT, ARITH, MULTI>, sweep_f32_kernel<POT, ARITH>, exchange_kernel<POT>,
# ladder_reduce_kernel<MOVES>, sweep_replay_kernel / sweep_replay_tma_kernel<POT, MULTI>, sweep_replay_f32_kernel<POT>
LEDGER = {
    "sweep_philox_kernel<0, 0, false, false>": ((NAT,), NATIVE),
    "sweep_philox_kernel<0, 0, false, true>": ((NAT, DEV), NATIVE),
    "sweep_philox_kernel<0, 0, true, false>": ((SER,), NATIVE),
    "sweep_philox_kernel<0, 0, true, true>": ((SER, DEV), NATIVE),
    "sweep_philox_kernel<0, 1, false, false>": ((NAT,), NATIVE),
    "sweep_philox_kernel<0, 1, false, true>": ((NAT, DEV, XCH), NATIVE),
    "sweep_philox_kernel<0, 1, true, false>": ((SER, HOST), NATIVE),
    "sweep_philox_kernel<0, 1, true, true>": ((SER, DEV), NATIVE),
    "sweep_philox_kernel<1, 0, false, false>": ((NAT,), NATIVE),
    "sweep_philox_kernel<1, 0, false, true>": ((NAT,), NATIVE),
    "sweep_philox_kernel<1, 0, true, false>": ((SER,), NATIVE),
    "sweep_philox_kernel<1, 0, true, true>": ((SER,), NATIVE),
    "sweep_philox_kernel<1, 1, false, false>": ((NAT,), NATIVE),
    "sweep_philox_kernel<1, 1, false, true>": ((NAT, XCH), NATIVE),
    "sweep_philox_kernel<1, 1, true, false>": ((SER,), NATIVE),
    "sweep_philox_kernel<1, 1, true, true>": ((SER, HOST), NATIVE),
    "sweep_philox_kernel<2, 0, false, false>": ((NAT,), NATIVE),
    "sweep_philox_kernel<2, 0, false, true>": ((NAT,), NATIVE),
    "sweep_philox_kernel<2, 0, true, false>": ((SER,), NATIVE),
    "sweep_philox_kernel<2, 0, true, true>": ((SER,), NATIVE),
    "sweep_philox_kernel<2, 1, false, false>": ((NAT,), NATIVE),
    "sweep_philox_kernel<2, 1, false, true>": ((NAT, XCH), NATIVE),
    "sweep_philox_kernel<2, 1, true, false>": ((SER,), NATIVE),
    "sweep_philox_kernel<2, 1, true, true>": ((SER,), NATIVE),
    "sweep_multi_kernel<0, 0, false>": ((NAT, MSER, DEV), NATIVE),
    "sweep_multi_kernel<0, 0, true>": ((NAT, MSER), NATIVE),
    "sweep_multi_kernel<0, 1, false>": ((NAT, MSER, DEV), NATIVE),
    "sweep_multi_kernel<0, 1, true>": ((NAT, MSER, XCH), NATIVE),
    "sweep_multi_kernel<1, 0, false>": ((NAT, MSER), NATIVE),
    "sweep_multi_kernel<1, 0, true>": ((NAT, MSER), NATIVE),
    "sweep_multi_kernel<1, 1, false>": ((NAT, MSER), NATIVE),
    "sweep_multi_kernel<1, 1, true>": ((NAT, MSER), NATIVE),
    "sweep_multi_kernel<2, 0, false>": ((NAT, MSER), NATIVE),
    "sweep_multi_kernel<2, 0, true>": ((NAT, MSER), NATIVE),
    "sweep_multi_kernel<2, 1, false>": ((NAT, MSER), NATIVE),
    "sweep_multi_kernel<2, 1, true>": ((NAT, MSER, HOST, XCH), NATIVE),
    "pgmc_kernel<0, 0, false>": ((PGMC_T,), PGMC),
    "pgmc_kernel<0, 1, false>": ((PGMC_T,), PGMC),
    "pgmc_kernel<0, 0, true>": ((PGMC_T, PGMC_GOLD), PGMC),
    "pgmc_kernel<1, 0, false>": ((PGMC_T,), PGMC),
    "pgmc_kernel<1, 1, false>": ((PGMC_T,), PGMC),
    "pgmc_kernel<1, 0, true>": ((PGMC_T,), PGMC),
    "pgmc_kernel<2, 0, false>": ((PGMC_T,), PGMC),
    "pgmc_kernel<2, 1, false>": ((PGMC_T,), PGMC),
    "pgmc_kernel<2, 0, true>": ((PGMC_T,), PGMC),
    "sweep_xoshiro_kernel<0, 0, false>": ((XOSH,), NATIVE),
    "sweep_xoshiro_kernel<0, 0, true>": ((XOSH,), NATIVE),
    "sweep_xoshiro_kernel<0, 1, false>": ((XOSH,), NATIVE),
    "sweep_xoshiro_kernel<0, 1, true>": ((XOSH,), NATIVE),
    "sweep_xoshiro_kernel<1, 0, false>": ((XOSH,), NATIVE),
    "sweep_xoshiro_kernel<1, 0, true>": ((XOSH,), NATIVE),
    "sweep_xoshiro_kernel<1, 1, false>": ((XOSH,), NATIVE),
    "sweep_xoshiro_kernel<1, 1, true>": ((XOSH,), NATIVE),
    "sweep_xoshiro_kernel<2, 0, false>": ((XOSH,), NATIVE),
    "sweep_xoshiro_kernel<2, 0, true>": ((XOSH,), NATIVE),
    "sweep_xoshiro_kernel<2, 1, false>": ((XOSH,), NATIVE),
    "sweep_xoshiro_kernel<2, 1, true>": ((XOSH,), NATIVE),
    "sweep_f32_kernel<0, 0>": ((F32_NAT, F32_STAT), STATISTICAL),
    "sweep_f32_kernel<0, 1>": ((F32_NAT, F32_STAT), STATISTICAL),
    "sweep_f32_kernel<1, 0>": ((F32_NAT,), STATISTICAL),
    "sweep_f32_kernel<1, 1>": ((F32_NAT,), STATISTICAL),
    "sweep_f32_kernel<2, 0>": ((F32_NAT,), STATISTICAL),
    "sweep_f32_kernel<2, 1>": ((F32_NAT,), STATISTICAL),
    "exchange_kernel<0>": ((XCH,), EXACT),
    "exchange_kernel<1>": ((XCH,), EXACT),
    "exchange_kernel<2>": ((XCH,), EXACT),
    "ladder_reduce_kernel<1>": ((XCH,), RECORDS),
    "ladder_reduce_kernel<16>": ((XCH,), RECORDS),
    "sweep_replay_kernel<0, false>": ((REPLAY,), EXACT),
    "sweep_replay_tma_kernel<0, false>": ((REPLAY,), EXACT),
    "sweep_replay_kernel<0, true>": ((REPLAY,), EXACT),
    "sweep_replay_tma_kernel<0, true>": ((REPLAY,), EXACT),
    "sweep_replay_f32_kernel<0>": ((F32_REPLAY,), EXACT),
    "sweep_replay_kernel<1, false>": ((REPLAY,), EXACT),
    "sweep_replay_tma_kernel<1, false>": ((REPLAY,), EXACT),
    "sweep_replay_kernel<1, true>": ((REPLAY,), EXACT),
    "sweep_replay_tma_kernel<1, true>": ((REPLAY,), EXACT),
    "sweep_replay_f32_kernel<1>": ((F32_REPLAY,), EXACT),
    "sweep_replay_kernel<2, false>": ((REPLAY,), EXACT),
    "sweep_replay_tma_kernel<2, false>": ((REPLAY,), EXACT),
    "sweep_replay_kernel<2, true>": ((REPLAY,), EXACT),
    "sweep_replay_tma_kernel<2, true>": ((REPLAY,), EXACT),
    "sweep_replay_f32_kernel<2>": ((F32_REPLAY,), EXACT),
}

FAMILIES = ("sweep_philox_kernel", "sweep_multi_kernel", "pgmc_kernel", "sweep_xoshiro_kernel", "sweep_f32_kernel",
            "exchange_kernel", "ladder_reduce_kernel", "sweep_replay_kernel", "sweep_replay_tma_kernel",
            "sweep_replay_f32_kernel")


def _instantiations():
    if shutil.which("nm") is None:
        pytest.skip("nm (binutils) is not installed: the library's kernel instantiations cannot be listed")
    out = subprocess.run(["nm", "-C", LIB_PATH], capture_output=True, text=True, check=True).stdout
    pat = re.compile(r"\b(" + "|".join(FAMILIES) + r")<([^<>]*)>\(")
    return {f"{m.group(1)}<{m.group(2)}>" for m in pat.finditer(out)}


def test_every_kernel_instantiation_has_a_ledger_row():
    found = _instantiations()
    assert found, f"no kernel instantiation found in {LIB_PATH}"
    assert not found - LEDGER.keys(), f"instantiations without a pinning test: {sorted(found - LEDGER.keys())}"
    assert not LEDGER.keys() - found, f"ledger rows the library no longer has: {sorted(LEDGER.keys() - found)}"


def test_every_ledger_row_names_existing_tests_and_a_bar():
    functions = {}
    for mod in {t.split("::")[0] for tests, _ in LEDGER.values() for t in tests}:
        with open(os.path.join(TESTS, mod + ".py")) as f:
            tree = ast.parse(f.read())
        functions[mod] = {n.name for n in tree.body if isinstance(n, ast.FunctionDef) and n.name.startswith("test_")}
    for kernel, (tests, bar) in LEDGER.items():
        assert tests, kernel
        assert bar in (EXACT, NATIVE, PGMC, RECORDS, STATISTICAL), kernel
        for t in tests:
            mod, fn = t.split("::")
            assert fn in functions[mod], f"{kernel}: {t} does not exist"
