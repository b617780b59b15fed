"""Replica exchange on one B200 (through the C ABI): the exchange kernel and arianna_ladder_sums at M = 2^27 chains for
L = 8, 32, 256 rungs, against the device-to-device copy bandwidth measured in the same run, and the overhead of one
exchange round per store interval on a C3-shaped run (harmonic, σ = 0.1, K = 10 steps per interval, 32-rung ladder).
Prints one JSON line per case with the card name, its power limit and the NVML clock record of the timed region
(bench.py's ClockSampler).  CUDA events on the engine's stream after warm-up; every working set is larger than L2."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import montecarlo_b200 as mb  # noqa: E402
from bench import ClockSampler  # noqa: E402

M = 1 << 27
SAMPLER = ClockSampler(0)
LAST_CLOCKS = [None]


def card():
    info = {"device": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(0)
        info["power_limit_w"] = pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
    except Exception:
        pass
    return info


CARD = None


def emit(**kw):
    kw.update(CARD)
    kw["clocks"] = LAST_CLOCKS[0]
    print(json.dumps(kw), flush=True)


def timed(stream, fn, reps, warm=4):
    """Device milliseconds per call of fn (CUDA events on `stream`, after `warm` untimed calls)."""
    with torch.cuda.stream(stream):
        for _ in range(warm):
            fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stream.synchronize()
        SAMPLER.start()
        a.record(stream)
        for _ in range(reps):
            fn()
        b.record(stream)
        b.synchronize()
        LAST_CLOCKS[0] = SAMPLER.stop()
    return a.elapsed_time(b) / reps


def copy_bandwidth():
    """Device-to-device copy of 2 GiB (read + write counted), the yardstick of the HBM-bound kernels."""
    src = torch.empty(1 << 28, dtype=torch.float64, device="cuda").fill_(1.0)
    dst = torch.empty_like(src)
    s = torch.cuda.current_stream()
    ms = timed(s, lambda: dst.copy_(src), reps=20)
    del src, dst
    torch.cuda.empty_cache()
    return 2 * 8 * (1 << 28) / (ms * 1e-3) / 1e9, ms


def main():
    global CARD
    CARD = card()
    copy_gbs, copy_ms = copy_bandwidth()
    emit(case="copy", bytes=2 * 8 * (1 << 28), ms=copy_ms, gbs=copy_gbs)
    for L in (8, 32, 256):
        with mb.CudaEnsemble(M, 1.0, [0.1], seed=42, arith="fast") as eng:
            eng.init_synthetic()
            eng.set_ladder(np.geomspace(0.5, 4.0, L))
            eng.sweep(10)
            s = eng.torch_stream()
            reps = 50
            for _ in range(4):                                 # warm-up rounds (even and odd)
                eng.replica_exchange()
            a0 = eng.exchange_counters()[0].sum()
            ms = timed(s, eng.replica_exchange, reps=reps, warm=0)
            swaps = int(eng.exchange_counters()[0].sum() - a0)
            # read x and β of every chain, write x of both chains of every swapped pair
            nbytes = 16 * M + 16 * swaps / reps
            gbs = nbytes / (ms * 1e-3) / 1e9
            emit(case="exchange_kernel", M=M, L=L, rounds=reps, ms_per_round=ms, bytes_per_round=nbytes, gbs=gbs,
                 copy_share=gbs / copy_gbs, swaps_per_round=swaps / reps)
            ms = timed(s, eng.ladder_sums, reps=20)
            nbytes = 12 * M                                   # x (8 B) + the accepted counter (4 B) of every chain
            gbs = nbytes / (ms * 1e-3) / 1e9
            emit(case="ladder_sums", M=M, L=L, calls=20, ms_per_call=ms, bytes_per_call=nbytes, gbs=gbs,
                 copy_share=gbs / copy_gbs, note="includes the fold and the [L][3] download")
    # C3-shaped run: 100 store intervals of K = 10 steps with the callback record after each
    n_int, K = 100, 10
    with mb.CudaEnsemble(M, 1.0, [0.1], seed=42, arith="fast") as eng:
        eng.init_synthetic()
        eng.set_ladder(np.geomspace(0.5, 4.0, 32))
        s = eng.torch_stream()
        ms_series = timed(s, lambda: eng.sweep_series([K] * n_int, read=False), reps=2, warm=1)

        def with_exchange():
            for _ in range(n_int):
                eng.sweep(K, reduce=True)
                eng.replica_exchange()

        def without_exchange():
            for _ in range(n_int):
                eng.sweep(K, reduce=True)

        ms_plain = timed(s, without_exchange, reps=2, warm=1)
        ms_pt = timed(s, with_exchange, reps=2, warm=1)
    steps = M * K * n_int
    emit(case="c3_parallel_tempering", M=M, L=32, K=K, intervals=n_int,
         series_no_exchange_chain_steps_per_s=steps / (ms_series * 1e-3),
         per_interval_no_exchange_chain_steps_per_s=steps / (ms_plain * 1e-3),
         with_exchange_chain_steps_per_s=steps / (ms_pt * 1e-3),
         overhead_vs_series=ms_pt / ms_series - 1, overhead_vs_per_interval=ms_pt / ms_plain - 1)


if __name__ == "__main__":
    if not torch.cuda.is_available():
        raise SystemExit("bench_exchange.py measures on a CUDA device; none is visible")
    main()
