#!/usr/bin/env python
"""bench.py -- Metropolis chain-steps/sec of the fused sweep on B200 (BASELINE.json metric).

Workload (BASELINE.json configs[2], "C3"): particle_1d harmonic, β = 2, Gaussian displacement σ = 0.1, Float64,
M = 2^27 chains per GPU, StoreCallbacks energy/acceptance every 10 MC steps.  One bench "step" = one store
interval = 10 Metropolis steps over every local chain + its callback record (Σe, Σacc/tot, count).  The engine fuses
up to `series_per_launch` (11 on B200) store intervals into ONE launch (arianna_sweep_series: chains stay in
registers across the intervals, the records are reduced on the device); the K steps are cut into equal launches
(K = 20 -> 2 launches of 10 stores, K = 110 -> 10 of 11).  `--series 1` is the one-launch-per-store path
(arianna_sweep with the reduction fused at its tail).  The all-reduce (N > 1) of a launch's records and their copy to
the host run on a side stream while the next launch already executes: the next sweep does not depend on callback means.
Chains are independent, so they shard over ranks with no data-path collective: weak scaling, per-GPU work fixed; the
line also carries a `strong` object (2^27 chains IN TOTAL, as configs[2] words it) and a `parity` object (a
2^20-chain strong-sharded mini-run checked against committed oracle / N = 1 values, tests/golden/bench_parity.json).

  python bench.py [--gpus N --steps K --warmup W]                  # our arm (one process per GPU under torchrun)
  python bench.py --impl reference [...]                           # the CPU restatement of the reference path
  python bench.py --dump-outputs DIR [...]                         # + the timed run's outputs as DIR/*.npy

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.  The inputs are seeded, so two builds
run with the same arguments can be compared output for output through --dump-outputs (see dump_outputs).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "metropolis_chain_steps_per_sec"
UNIT = "chain-steps/s"
FLOPS_PER_CHAIN_STEP = 110.0          # SURVEY.md §8d convention (12 plain + exp 36 + ½(log 44 + sqrt 12 + sincos 70))
BYTES_PER_CHAIN_PER_LAUNCH = 24.0     # x f64 read+write, acc u32 read+write
PARITY_GOLDEN = os.path.join(ROOT, "tests", "golden", "bench_parity.json")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=110)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2-chains", type=int, default=27, help="chains per GPU (weak) or in total (strong), log2")
    ap.add_argument("--mc-steps", type=int, default=10, help="Metropolis steps per store interval")
    ap.add_argument("--series", type=int, default=0,
                    help="store intervals fused per launch (0 = the engine's preferred count, 1 = one launch per store)")
    ap.add_argument("--slices", type=int, default=8, help="regular chain slices of the pipelined end-to-end job")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--arith", default="fast", choices=["fast", "exact"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--ref-log2-chains", type=int, default=0,
                    help="chains of the CPU arm's sample, log2 (0 = the full per-GPU ensemble when it fits --ref-seconds, "
                         "else the largest power of two that does; cpu_baseline leg: 2^20)")
    ap.add_argument("--ref-seconds", type=float, default=120.0, help="time budget of the --impl reference run")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="time budget of the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what they computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ---------------------------------------------------------------------------------------------------------
# clocks: NVML sampled in a thread DURING the timed region
# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index: int, period_s: float = 0.002):
        """nvmlInit happens HERE (tens of ms): construct the sampler before the barrier that precedes the timed region."""
        self.samples, self.reasons, self.power = [], set(), []
        self.max_mhz = None
        self.period = period_s
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self._reasons_fn = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = self._reasons_fn(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        self.samples, self.reasons, self.power = [], set(), []
        self._stop.clear()
        if self.nv is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()

    def stop(self):
        if self._thr is not None:
            self._stop.set()
            self._thr.join()
            self._thr = None
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples), "power_w_max": max(self.power) if self.power else None}


# ---------------------------------------------------------------------------------------------------------
# CPU arm: the oracle's restatement of Metropolis.make_step! with parallel=true (OpenMP over chains)
# ---------------------------------------------------------------------------------------------------------
def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_reference_rate(log2_chains: int, mc_steps: int, steps: int, warmup: int, budget_s: float = 20.0, threads: int = 0):
    """chain-steps/s of the reference path on the host cores, on a bounded sample of the workload: 2^log2_chains
    chains, `steps` store intervals of mc_steps Metropolis steps + the energy/acceptance callbacks.  `threads` > 0
    forces the OpenMP team size (torchrun exports OMP_NUM_THREADS=1, which would void the arm)."""
    from oracle import oracle as O
    if threads > 0:
        O.set_num_threads(threads)
    M = 1 << log2_chains
    ens = O.Ensemble(O.init_synthetic(42, 0, M), 2.0, [0.1])
    ens.seed_xoshiro(42)
    for _ in range(max(1, warmup)):
        ens.sweep_xoshiro(mc_steps)
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        ens.sweep_xoshiro(mc_steps)
        ens.callback_energy()
        ens.callback_acceptance()
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return M * mc_steps * done / dt, done, dt, O.num_threads()


def run_reference(args):
    """The reference arm: rank 0 alone, ALL host cores, on the arm's own config.  The sample is the full per-GPU
    ensemble (2^27 chains) when K + W store intervals of it fit --ref-seconds at the calibrated rate, else the largest
    power of two that does; the line says which."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # other ranks exit 0 without work
    cores = host_cores()
    m_log2 = args.ref_log2_chains
    if m_log2 <= 0:
        rate0, _, _, _ = cpu_reference_rate(min(20, args.log2_chains), args.mc_steps, 3, 1, 5.0, threads=cores)
        fit = rate0 * args.ref_seconds / (args.mc_steps * (args.steps + max(1, args.warmup)))
        m_log2 = max(10, min(args.log2_chains, int(math.floor(math.log2(max(fit, 1024.0))))))
    while True:
        try:
            rate, done, dt, threads = cpu_reference_rate(m_log2, args.mc_steps, args.steps, args.warmup,
                                                         2.0 * args.ref_seconds, threads=cores)
            break
        except MemoryError:
            m_log2 -= 1
    full = m_log2 == args.log2_chains
    sample = (f"2^{m_log2} chains ({'the full per-GPU ensemble' if full else 'bounded sample of the 2^%d per GPU' % args.log2_chains}) "
              f"x {done} store intervals of {args.mc_steps} MC steps + both callbacks, {threads} OpenMP threads "
              f"(C restatement of mc_sweep!/Metropolis.make_step! parallel=true, xoshiro256++/ziggurat; Julia is absent)")
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": done,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / done,
        "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "sample": {"chains": 1 << m_log2, "store_intervals": done, "seconds": dt, "full_per_gpu_ensemble": full},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def workload_config(args, world):
    """The WORKLOAD, identical in both arms (engine tuning such as stores per launch lives in the line's `engine`)."""
    m_local = chains_per_rank(args, world)
    return {
        "workload": "C3: particle_1d harmonic beta=2, Gaussian Displacement sigma=0.1, Metropolis + StoreCallbacks "
                    "energy/acceptance every 10 steps (BASELINE.json configs[2])",
        "chains_per_gpu": m_local, "chains_total": m_local * world, "mc_steps_per_store": args.mc_steps,
        "l2_policy": "inputs larger than L2 (x + counters = %.0f MiB per GPU vs 126 MB L2)" % (m_local * 12 / 2 ** 20),
        "parallelism": f"chains sharded x{world}, all-reduce of 3 doubles per store",
    }


def _finite(o):
    """JSON has no NaN / Infinity: non-finite floats become null (strict parsers reject Python's `NaN` literal)."""
    if isinstance(o, float):
        return o if math.isfinite(o) else None
    if isinstance(o, dict):
        return {k: _finite(v) for k, v in o.items()}
    if isinstance(o, (list, tuple)):
        return [_finite(v) for v in o]
    return o


def emit(line):
    print(json.dumps(_finite(line), allow_nan=False), flush=True)


def _profile():
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return None


def ncu_issue(m_local, mc_steps, series, chain_steps_per_s, sm_count=148, smsp=4, ghz=1.965):
    """Issue-slot view of the same launch: warp instructions per warp-step from the committed ncu capture x the
    measured step rate, against one instruction per SMSP per clock.  (The sweep is issue-bound: an IMAD.WIDE holds
    the dispatch port for ~4.5 cycles, profiles/microbench.)"""
    t = _profile()
    if not t or t.get("mc_steps") != mc_steps:
        return None
    ach = t["warp_inst_per_warp_step"] * chain_steps_per_s / 32.0
    peak = sm_count * smsp * ghz * 1e9
    return {"achieved": ach / 1e9, "peak": peak / 1e9, "unit": "G warp-inst/s", "frac": ach / peak,
            "warp_inst_per_warp_step": t["warp_inst_per_warp_step"],
            "ncu_issue_active_pct": t.get("issue_active_pct"), "source": t["source"]}


def ncu_executed_flops(mc_steps, chain_steps_per_s, fp64_peak):
    """FP64 flops the kernel actually EXECUTES per chain-step (ncu smsp__sass_thread_inst_executed_op_{dfma,dmul,dadd}
    _pred_on, DFMA = 2) x the measured step rate: the hardware-side FP64 fraction beside the F = 110 convention."""
    t = _profile()
    if not t or t.get("mc_steps") != mc_steps or "fp64_flop_per_chain_step" not in t:
        return None
    ach = t["fp64_flop_per_chain_step"] * chain_steps_per_s
    return {"flop_per_chain_step": t["fp64_flop_per_chain_step"], "achieved": ach / 1e12, "unit": "TFLOP/s",
            "frac": ach / fp64_peak, "fp64_pipe_pct_ncu": t.get("fp64_pipe_pct"), "source": t["source"]}


def ncu_traffic(m_local, mc_steps, series=1):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the sweep kernel from the committed `ncu --set full`
    capture (profiles/traffic.json, written by scripts/summarise_profile.py); only valid for the captured shape."""
    t = _profile()
    if t and t["chains"] == m_local and t["mc_steps"] == mc_steps:
        return {"bytes_per_launch": t["dram_bytes_per_launch"], "algorithmic_bytes_per_launch": 24 * m_local,
                "captured_stores_per_launch": t.get("series", 1), "source": t["source"]}
    return None


def chains_per_rank(args, world):
    total = 1 << args.log2_chains
    return total if args.scaling == "weak" else total // world


def launch_plan(K, g_max):
    """K store intervals in equal launches of at most g_max: K = 20, g_max = 11 -> [10, 10]."""
    n = max(1, math.ceil(K / max(1, g_max)))
    g = math.ceil(K / n)
    return [min(g, K - s) for s in range(0, K, g)]


DUMP_SAMPLE_CHAINS = 1 << 20          # 2 per-chain arrays x 8 B x 2^20 = 16 MiB: the whole dump stays under 64 MB


def dump_outputs(out_dir, eng, records):
    """Writes what the timed store intervals handed their caller, as float64 arrays in out_dir:
      records.npy            [K][3] the callback record of every timed store interval (Σe, Σ acc/tot, chain count),
                             summed over the ranks
      x.npy, accepted.npy    position and accepted-move count after the last timed interval of a fixed sample of this
                             rank's chains: DUMP_SAMPLE_CHAINS chain indices drawn with numpy's default_rng(0) without
                             replacement, in ascending order (every chain when there are fewer).
    The energies are not written: the engine derives them from the positions."""
    os.makedirs(out_dir, exist_ok=True)
    x = eng.get_state()
    acc = eng.chain_counters()[0][0]
    n = x.size
    idx = np.arange(n) if n <= DUMP_SAMPLE_CHAINS else \
        np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLE_CHAINS, replace=False))
    for name, a in (("records", records), ("x", x[idx]), ("accepted", acc[idx])):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


# ---------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    import montecarlo_b200 as mb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    K, W, S = args.steps, max(3, args.warmup), args.mc_steps
    stream = torch.cuda.Stream(device=local_rank)      # torch owns the compute stream; the engine launches on it
    side = torch.cuda.Stream(device=local_rank)        # all-reduce + D2H of a launch's records, beside the next launch
    sampler = ClockSampler(local_rank)                 # nvmlInit now, not between the barrier and the first event

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_engine(m_local, offset, total):
        return mb.CudaEnsemble(m_local, 2.0, [0.1], [1.0], seed=42, chain_offset=offset, n_chains_total=total,
                               arith=args.arith, device=local_rank, stream=stream.cuda_stream)

    def timed_run(eng, m_local, K, W, want_clocks):
        """W warm-up + K timed store intervals; returns device ms (max over ranks), per-launch ms, records, launches."""
        g_max = args.series if args.series > 0 else eng.series_per_launch
        g_max = max(1, min(g_max, 64))
        plan = launch_plan(K, g_max)
        host = torch.empty((len(plan), 3 * max(plan)), dtype=torch.float64).pin_memory()
        pending = []

        def one_launch(i, n, ev=None):
            """n store intervals: one fused launch (+ the record fold) on the compute stream; the all-reduce (N > 1) and
            the D2H of the 3n sums follow on the side stream and overlap the next launch."""
            if ev is not None:
                ev[0].record(stream)
            if g_max == 1:
                eng.sweep(S, reduce=True)
            else:
                eng.sweep_series([S] * n, read=False)
            if ev is not None:
                ev[1].record(stream)
            t = (eng.callback_sums_tensor() if g_max == 1 else eng.series_tensor()).clone()   # snapshot: the buffer is reused
            t.record_stream(side)
            snap = torch.cuda.Event()
            snap.record(stream)
            with torch.cuda.stream(side):
                side.wait_event(snap)
                if world > 1:
                    dist.all_reduce(t)
                if i is not None:
                    host[i, :3 * n].copy_(t, non_blocking=True)
            pending.append(t)

        with torch.cuda.stream(stream):
            for n in launch_plan(W, g_max):
                one_launch(None, n)
            stream.wait_stream(side)
            barrier()
            launches0 = eng.launch_count
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in plan]
            start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            if want_clocks:
                sampler.start()
            barrier()                                   # re-barrier immediately before the first timed event
            start.record(stream)
            for i, (n, e) in enumerate(zip(plan, ev)):
                one_launch(i, n, e)
            stream.wait_stream(side)                    # the K steps are done when their records are on the host
            stop.record(stream)
            stop.synchronize()
            torch.cuda.synchronize()
            clocks = sampler.stop() if want_clocks else None
            barrier()
        launches = eng.launch_count - launches0
        ms_total = start.elapsed_time(stop)
        full = [a.elapsed_time(b) for n, (a, b) in zip(plan, ev) if n == plan[0]]
        tmax = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        rec = np.concatenate([host[i, :3 * n].numpy().reshape(n, 3) for i, n in enumerate(plan)])
        return {"ms": float(tmax.item()), "kern_ms": float(np.mean(full)), "n_full": len(full), "plan": plan,
                "records": rec, "launches": int(launches), "clocks": clocks, "g_max": g_max}

    # ---- the headline run: weak scaling by default (2^27 chains per GPU) --------------------------------------
    m_local = chains_per_rank(args, world)
    eng = make_engine(m_local, rank * m_local, m_local * world)
    with torch.cuda.stream(stream):
        eng.init_synthetic()
        fp64_peak = eng.measure_fp64_peak()
    main = timed_run(eng, m_local, K, W, True)
    rec = main["records"]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, rec)           # before the e2e leg moves the chains on
    energy = float(rec[-1, 0] / rec[-1, 2])
    value = m_local * world * S * K / (main["ms"] * 1e-3)

    # ---- e2e: the same job through the C ABI with HOST buffers inside the timed region ----------------------------
    e2e = None
    if not args.no_e2e:
        with torch.cuda.stream(stream):
            x_in = torch.empty(m_local, dtype=torch.float64).pin_memory()
            x_out = torch.empty(m_local, dtype=torch.float64).pin_memory()
            eng.get_state_to_ptr(x_in.data_ptr())
            if world > 1:
                # the collective of this leg runs INSIDE the library (arianna_comm_init / arianna_series_global over
                # dlopen'ed NCCL), the route a host without torch.distributed (the Julia shim) takes
                ids = [mb.CudaEnsemble.nccl_unique_id() if rank == 0 else None]
                dist.broadcast_object_list(ids, src=0)
                eng.comm_init(ids[0], rank, world)
            # W untimed warm-up store intervals through the SAME route: the first host job creates the copy streams and
            # events, the first in-library all-reduce connects the NCCL communicator (about a second)
            if main["g_max"] == 1:
                eng.sweep(S, reduce=True)
                _ = eng.callbacks_global() if world > 1 else eng.callback_sums()
            else:
                eng.run_host_job([S] * W, x_in=x_in.data_ptr(), x_out=x_out.data_ptr(), n_slices=args.slices, read=False)
                _ = eng.series_global(W)
            def timed_job(download):
                """One end-to-end job: x0 pinned host -> HBM, K store intervals, the K records -> host (all-reduced
                inside the library when N > 1) and, with `download`, the final chains -> pinned host."""
                barrier()
                barrier()
                t0 = time.perf_counter()
                if main["g_max"] == 1:
                    eng.set_state_from_ptr(x_in.data_ptr())            # H2D: the job's chains, pinned host -> HBM
                    for _ in range(K):
                        eng.set_params(0, 0.1)                         # the launch's input: policy parameters θ = (σ)
                        eng.sweep(S, reduce=True)
                        if world > 1:
                            ev = float(eng.callbacks_global()[0])      # in-library all-reduce + D2H: the step's result
                        else:
                            vals = eng.callback_sums()                 # D2H: the step's result (3 doubles)
                            ev = float(vals[0] / vals[2])
                    if download:
                        eng.get_state_to_ptr(x_out.data_ptr())         # D2H: final chains (StoreLastFrames)
                else:
                    # the whole job in ONE C-ABI call: chains in, K store intervals, records out (chains out); the library
                    # pipelines slices of chains so that the copies (one stream per PCIe direction) overlap the sweeps
                    eng.set_params(0, 0.1)
                    r = eng.run_host_job([S] * K, x_in=x_in.data_ptr(), x_out=x_out.data_ptr() if download else None,
                                         n_slices=args.slices, read=(world == 1))
                    t_job = time.perf_counter() - t0
                    if world > 1:
                        r = eng.series_global(K)                       # in-library NCCL all-reduce + D2H of the K records
                    ev = float(r[-1, 0] / r[-1, 2])
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                detail = None
                if main["g_max"] > 1:
                    detail = dict(eng.job_timing(), job_ms=1e3 * t_job, sweep_ms=eng.timing()[0], total_ms=1e3 * dt)
                    if world > 1:                                      # every rank's view (the slowest one sets the time)
                        rows = [None] * world
                        dist.all_gather_object(rows, detail)
                        detail = {"per_rank": rows}
                tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
                if world > 1:
                    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                return float(tt.item()), ev, detail

            dt, evals, pcie = timed_job(False)
            dt_dl, _, pcie_dl = timed_job(True)
        total_steps = m_local * world * S * K
        e2e = {"value": total_steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": int(8 * m_local / K + 8), "d2h_bytes_per_step": 24,
               "seconds": dt, "collective": "in-library NCCL (arianna_series_global)" if world > 1 else None,
               "pcie": pcie,
               "note": ("timed: ONE arianna_run_host_job call = pinned-host x0 -> HBM, K store intervals, the K callback "
                        f"records -> host, pipelined over ramped slices of chains ({args.slices} regular ones); the chains "
                        "stay resident in HBM like the shim's CudaEnsemble (C3 has no StoreLastFrames)"
                        if main["g_max"] > 1 else
                        "timed: pinned-host x0 -> HBM once, per step sigma in + callback sums out; the one-off upload is "
                        "amortised over the K steps"),
               "with_final_state_download": {
                   "value": total_steps / dt_dl, "seconds": dt_dl, "d2h_bytes_per_step": int(8 * m_local / K + 24),
                   "pcie": pcie_dl,
                   "note": "the same job + the final chains -> pinned host (StoreLastFrames), uploads and downloads on "
                           "separate streams"},
               "energy": evals}
        del x_in, x_out

    eng.close()

    # ---- strong scaling: BASELINE configs[2] as worded, 2^27 chains IN TOTAL over the N GPUs ------------------------
    strong = None
    if not args.no_strong:
        total = 1 << args.log2_chains
        if world == 1 or args.scaling == "strong":
            strong = {"chains_total": total, "value": value, "ms_per_step": main["ms"] / K,
                      "note": "identical to the headline run"}
        else:
            ms = total // world
            es = make_engine(ms, rank * ms, total)
            with torch.cuda.stream(stream):
                es.init_synthetic()
            sr = timed_run(es, ms, K, W, False)
            strong = {"chains_total": total, "chains_per_gpu": ms, "value": total * S * K / (sr["ms"] * 1e-3),
                      "ms_per_step": sr["ms"] / K, "kernel_ms": sr["kern_ms"], "stores_per_launch": sr["plan"][0]}
            es.close()

    # ---- parity: a strong-sharded 2^20-chain mini-run against committed values (shard invariance under the driver) ---
    parity = None
    if not args.no_parity:
        parity = parity_check(mb, torch, dist, make_engine, stream, rank, world)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        kern_ms, steps_per_launch = main["kern_ms"], S * main["plan"][0]
        rate = m_local * steps_per_launch / (kern_ms * 1e-3)            # chain-steps/s of one GPU inside the kernel
        ach_tf = FLOPS_PER_CHAIN_STEP * rate / 1e12
        ach_gb = BYTES_PER_CHAIN_PER_LAUNCH * m_local / (kern_ms * 1e-3) / 1e9
        roofline = {
            "bound": "fp64", "kernel": "sweep_philox_kernel<HARMONIC,%s,single-move%s>" % (
                args.arith.upper(), ",series" if main["g_max"] > 1 else ""),
            "achieved": ach_tf, "peak": fp64_peak / 1e12, "unit": "TFLOP/s", "frac": ach_tf / (fp64_peak / 1e12),
            "peak_source": "DFMA microbenchmark in this run (arianna_measure_fp64_peak; MEASURED_PEAKS.json has no "
                           "FP64 entry); nominal 148 SM x 64 DFMA/clk x 2 x 1.965 GHz = 37.2",
            "note": "issue-bound FP64/integer kernel, no tensor-core work: neither 'hbm' nor 'tensor' applies. achieved = "
                    "110 conventional FP64 flop per chain-step (SURVEY.md 8d, fixed before the build) x steps/s; the "
                    "kernel executes far fewer (tables, FP32 filter), so frac may exceed 1 -- 'executed' is the FP64 work "
                    "the kernel really issues, 'issue' the hardware-side issue-slot fraction, 'hbm' the memory view",
            "flops_per_chain_step": FLOPS_PER_CHAIN_STEP, "kernel_ms": kern_ms, "kernel_launches_averaged": main["n_full"],
            "mc_steps_per_launch": steps_per_launch,
            "traffic": ncu_traffic(m_local, S, main["plan"][0]),
            "executed": ncu_executed_flops(S, rate, fp64_peak),
            "issue": ncu_issue(m_local, S, main["plan"][0], rate),
            "hbm": {"achieved": ach_gb, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gb / hbm_peak,
                    "bytes_per_chain_step": BYTES_PER_CHAIN_PER_LAUNCH / steps_per_launch,
                    "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"},
        }
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": main["ms"] / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(args, world),
            "engine": {"stores_per_launch": main["plan"][0], "mc_steps_per_launch": steps_per_launch,
                       "launch_plan": main["plan"], "rng": "philox4x32-10 + box-muller (native mode)", "arith": args.arith,
                       "collective": "torch.distributed NCCL all-reduce of 3 doubles per store, one per launch, on a "
                                     "side stream (overlaps the next launch)" if world > 1 else None},
            "clocks": main["clocks"], "gpu_launches": main["launches"], "roofline": roofline, "mean_energy": energy,
        }
        if e2e:
            line["e2e"] = e2e
        if strong:
            line["strong"] = strong
        if parity:
            line["parity"] = parity
        if world == 1 and not args.no_cpu_baseline:
            lg = args.ref_log2_chains if args.ref_log2_chains > 0 else 20
            rate, done, dt, cores = cpu_reference_rate(lg, S, 10 ** 9, 2, args.cpu_seconds, threads=host_cores())
            line["cpu_baseline"] = {
                "value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"2^{lg} chains x {done} store intervals of {S} MC steps in {dt:.1f} s "
                          "(oracle: C restatement of mc_sweep! with xoshiro256++/ziggurat, OpenMP over chains)"}
        emit(line)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def parity_check(mb, torch, dist, make_engine, stream, rank, world):
    """2^20 chains IN TOTAL, sharded over the N ranks like any ensemble (contiguous global chain ids), 5 store
    intervals of 10 steps in one series launch.  The all-reduced records must equal the committed ones
    (tests/golden/bench_parity.json: computed by the CPU oracle; Σe to 1e-12, the integer Σacc exactly), and the
    order-independent 64-bit checksum of the final positions (sum of the bit patterns mod 2^64, all-reduced) must equal
    the one a single GPU produced -- i.e. the N-rank run is bit for bit the 1-rank run."""
    try:
        gold = json.load(open(PARITY_GOLDEN))
    except Exception as exc:
        return {"ok": None, "error": f"no golden file: {exc}"}
    total, Ks, seed = int(gold["chains"]), [int(k) for k in gold["Ks"]], int(gold["seed"])
    off, m = mb.shard_bounds(total, rank, world)
    eng = mb.CudaEnsemble(m, float(gold["beta"]), [float(gold["sigma"])], [1.0], seed=seed, chain_offset=off,
                          n_chains_total=total, arith="fast", device=torch.cuda.current_device(),
                          stream=stream.cuda_stream)
    with torch.cuda.stream(stream):
        eng.init_synthetic()
        eng.sweep_series(Ks, read=False)
        rec = eng.series_tensor().clone()
        if world > 1:
            dist.all_reduce(rec)
        rec = rec.cpu().numpy().reshape(len(Ks), 3)
        x = eng.get_state()
        acc = eng.chain_counters()[0][0]
        chk = torch.tensor([int(x.view(np.uint64).sum(dtype=np.uint64).astype(np.int64)),
                            int(acc.sum(dtype=np.int64))], dtype=torch.int64, device="cuda")
        if world > 1:
            dist.all_reduce(chk)                        # int64 sums wrap modulo 2^64: order-independent, exact
        chk = chk.cpu().numpy()
    eng.close()
    g = np.array(gold["records"], dtype=np.float64)
    t_done = np.cumsum(Ks)
    err_e = float(np.max(np.abs(rec[:, 0] / g[:, 0] - 1.0)))
    acc_sums = np.rint(rec[:, 1] * t_done).astype(np.int64)
    acc_exact = bool(np.array_equal(acc_sums, np.array(gold["acc_sums"], dtype=np.int64)))
    count_ok = bool(np.all(rec[:, 2] == total))
    x_chk = int(np.uint64(chk[0].astype(np.uint64)))
    want = gold.get("x_bits_checksum_gpu_n1")
    ok = err_e <= 1e-12 and acc_exact and count_ok and int(chk[1]) == int(gold["acc_sums"][-1]) and \
        (want is None or x_chk == int(want, 16))
    return {"ok": bool(ok), "chains_total": total, "ranks": world, "stores": len(Ks),
            "energy_sum_max_rel_err_vs_oracle": err_e, "accepted_sums_equal_oracle": acc_exact,
            "x_bits_checksum": f"{x_chk:#018x}",
            "x_bits_checksum_equals_1gpu": None if want is None else bool(x_chk == int(want, 16)),
            "golden": "tests/golden/bench_parity.json (oracle records; 1-GPU checksum of the final positions)"}


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
