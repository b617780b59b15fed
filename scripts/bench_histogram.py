"""On-device histograms on one B200 (through the C ABI): one arianna_histogram_accumulate at M = 2^27 chains (the working
set is larger than L2) for Float64 and Float32 handles, observables x and e, G = 1 with 64 / 1024 / 16381 bins and G = 32
with 509 bins, on a broad state (harmonic equilibrium, range ±4 std) and on the worst case (every chain in one bin), against
the device-to-device copy bandwidth measured in the same run.  Context: what a user does without it (get_state +
np.histogram) and a C3-shaped run (harmonic, σ = 0.1, a store every 10 steps) with and without one accumulate per store.
Prints one JSON line per case with the card name, its power limit and the NVML clock record of the timed region."""
import json
import math
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import montecarlo_b200 as mb  # noqa: E402
from bench_exchange import LAST_CLOCKS, card, copy_bandwidth, timed  # noqa: E402
import bench_exchange  # noqa: E402

M = 1 << 27
BETA = 1.0
SD = math.sqrt(1 / (2 * BETA))                  # harmonic equilibrium: x ~ N(0, 1/(2β))
SHAPES = [(1, 64), (1, 1024), (1, 16381), (32, 509)]


def emit(**kw):
    kw.update(bench_exchange.CARD)
    kw["clocks"] = LAST_CLOCKS[0]
    print(json.dumps(kw), flush=True)


def main():
    bench_exchange.CARD = card()
    copy_gbs, copy_ms = copy_bandwidth()
    emit(case="copy", bytes=2 * 8 * (1 << 28), ms=copy_ms, gbs=copy_gbs)
    for dtype, width in (("f64", 8), ("f32", 4)):
        with mb.CudaEnsemble(M, BETA, [1.0], seed=42, arith="fast", dtype=dtype) as eng:
            s = eng.torch_stream()
            for state in ("broad", "one_bin"):
                if state == "broad":
                    eng.init_synthetic()
                    eng.sweep(300)
                else:
                    eng.set_state(np.zeros(M))
                for obs, rng in (("x", (-4 * SD, 4 * SD)), ("e", (0.0, (4 * SD) ** 2))):
                    for G, bins in SHAPES:
                        eng.set_histogram(obs, rng[0], rng[1], bins, G)
                        reps = 20
                        ms = timed(s, eng.histogram_accumulate, reps=reps, warm=3)
                        counts, _, n = eng.histogram()
                        assert counts.sum() == n * M
                        nbytes = width * M                  # the kernel reads x once; the fold reads a few KB
                        gbs = nbytes / (ms * 1e-3) / 1e9
                        emit(case="histogram_accumulate", dtype=dtype, observable=obs, state=state, M=M, groups=G,
                             bins=bins, calls=reps, ms_per_call=ms, bytes_per_call=nbytes, gbs=gbs,
                             copy_share=gbs / copy_gbs, max_cell_share=float(counts.max() / counts.sum()))
        # what a user does without it: download the positions, bin them on the host
        if dtype == "f64":
            with mb.CudaEnsemble(M, BETA, [1.0], seed=42, arith="fast") as eng:
                eng.init_synthetic()
                eng.sweep(300)
                eng.synchronize()
                t0 = time.perf_counter()
                x = eng.get_state()
                t1 = time.perf_counter()
                np.histogram(x, bins=64, range=(-4 * SD, 4 * SD))
                t2 = time.perf_counter()
                LAST_CLOCKS[0] = None
                emit(case="get_state_np_histogram", M=M, bins=64, get_state_ms=(t1 - t0) * 1e3,
                     np_histogram_ms=(t2 - t1) * 1e3, total_ms=(t2 - t0) * 1e3, note="host wall clock, pageable buffer")
                del x
    # C3-shaped run: 100 store intervals of K = 10 steps, the callback record after each; with StoreHistograms on the
    # same schedule every store time is a barrier, so the intervals run as per-store sweeps plus one accumulate each
    n_int, K = 100, 10
    with mb.CudaEnsemble(M, BETA, [0.1], seed=42, arith="fast") as eng:
        eng.init_synthetic()
        eng.set_histogram("x", -4 * SD, 4 * SD, 64)
        s = eng.torch_stream()
        ms_series = timed(s, lambda: eng.sweep_series([K] * n_int, read=False), reps=2, warm=1)

        def per_interval():
            for _ in range(n_int):
                eng.sweep(K, reduce=True)

        def with_histogram():
            for _ in range(n_int):
                eng.sweep(K, reduce=True)
                eng.histogram_accumulate()

        ms_plain = timed(s, per_interval, reps=2, warm=1)
        ms_hist = timed(s, with_histogram, reps=2, warm=1)
    steps = M * K * n_int
    emit(case="c3_store_histograms", M=M, K=K, intervals=n_int, bins=64,
         series_no_histogram_chain_steps_per_s=steps / (ms_series * 1e-3),
         per_interval_no_histogram_chain_steps_per_s=steps / (ms_plain * 1e-3),
         with_histogram_chain_steps_per_s=steps / (ms_hist * 1e-3),
         overhead_vs_series=ms_hist / ms_series - 1, overhead_vs_per_interval=ms_hist / ms_plain - 1)


if __name__ == "__main__":
    if not torch.cuda.is_available():
        raise SystemExit("bench_histogram.py measures on a CUDA device; none is visible")
    main()
