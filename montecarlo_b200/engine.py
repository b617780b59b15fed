"""CudaEnsemble -- Python owner of one arianna_handle (one GPU, one contiguous shard of the global ensemble).

This is the Python twin of the Julia shim's `CudaEnsemble <: AriannaSystem` (INTEGRATION.md): every method is a
1:1 call through the C ABI of libarianna_cuda.so (include/arianna_cuda.h).  numpy arrays in, numpy arrays out;
torch is only used (optionally) to wrap the engine's stream / reduction buffers for torch.distributed.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import _lib as L


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class _DeviceBuffer:
    """Minimal __cuda_array_interface__ carrier so torch.as_tensor can alias an engine-owned f64 buffer."""

    def __init__(self, ptr: int, n: int, stream: int):
        self.__cuda_array_interface__ = {
            "shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 3, "strides": None,
            "stream": None,  # ordering is the caller's job: use the tensor on the engine's own stream
        }


class HostBuffer:
    """Page-locked host memory from the library (arianna_host_alloc), viewed as a float64 numpy array.
    write_combined=True: for buffers the host only writes and the GPU reads (uploads)."""

    def __init__(self, n: int, write_combined: bool = False):
        self._lib = L.load()
        p = C.c_void_p()
        L.check(None, self._lib.arianna_host_alloc(8 * int(n), 1 if write_combined else 0, C.byref(p)))
        self.ptr = p.value
        self.array = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_double)), shape=(int(n),))

    def close(self):
        if getattr(self, "ptr", None):
            self.array = None
            self._lib.arianna_host_free(C.c_void_p(self.ptr))
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class CudaEnsemble:
    """M Metropolis chains of the particle_1d system resident in the HBM of one B200.

    Parameters mirror the reference objects they replace:
      n_chains, chain_offset, n_chains_total -- shard of `chains::Vector{Particle}` (simulation.jl:17)
      beta                                   -- Particle.β (particle_1d.jl:11)
      sigma, weight                          -- Move(Displacement(0.0), StandardGaussian(), ComponentArray(σ=σ), w)
      seed                                   -- Metropolis(...; seed) (metropolis.jl:288)
    """

    def __init__(self, n_chains: int, beta: float, sigma: Sequence[float], weight: Optional[Sequence[float]] = None,
                 *, seed: int = 1, chain_offset: int = 0, n_chains_total: int = 0, potential: str = "harmonic",
                 rng: str = "philox", arith: str = "fast", device: int = -1, stream: int = 0, dtype: str = "f64"):
        self._lib = L.load()
        sigma = [float(s) for s in np.atleast_1d(sigma)]
        weight = [1.0 / len(sigma)] * len(sigma) if weight is None else [float(w) for w in np.atleast_1d(weight)]
        if len(sigma) != len(weight):
            raise ValueError("sigma and weight must have the same length")
        if len(sigma) > L.MAX_MOVES:
            raise ValueError(f"at most {L.MAX_MOVES} moves per pool")
        cfg = L.Config()
        cfg.struct_size = C.sizeof(L.Config)
        cfg.device = device
        cfg.n_chains = int(n_chains)
        cfg.chain_offset = int(chain_offset)
        cfg.n_chains_total = int(n_chains_total)
        cfg.seed = int(seed)
        cfg.beta = float(beta)
        cfg.potential = L.POTENTIALS[potential]
        cfg.n_moves = len(sigma)
        for k, (s, w) in enumerate(zip(sigma, weight)):
            cfg.sigma[k] = s
            cfg.weight[k] = w
        cfg.rng_mode = L.RNG_MODES[rng]
        cfg.arith_mode = L.ARITH_MODES[arith]
        cfg.stream = stream or None
        cfg.dtype = L.DTYPES[dtype]
        self.dtype = dtype
        self._h = C.c_void_p()
        L.check(None, self._lib.arianna_create(C.byref(cfg), C.byref(self._h)))
        self.n_chains = int(n_chains)
        self.chain_offset = int(chain_offset)
        self.n_chains_total = int(n_chains_total) or int(n_chains)
        self.n_moves = len(sigma)
        self.seed = int(seed)
        self.beta = float(beta)
        self.rng, self.arith, self.potential = rng, arith, potential
        self.ladder = None

    # -- lifecycle ----------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.arianna_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _ck(self, code):
        L.check(self._h, code)

    # -- chain state --------------------------------------------------------------------------------------
    def set_state(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        if x.shape != (self.n_chains,):
            raise ValueError(f"x must have shape ({self.n_chains},)")
        self._ck(self._lib.arianna_set_state(self._h, _ptr(x)))

    def init_synthetic(self, seed: Optional[int] = None):
        self._ck(self._lib.arianna_init_synthetic(self._h, self.seed if seed is None else int(seed)))

    def get_state(self, with_energy: bool = False):
        x = np.empty(self.n_chains, dtype=np.float64)
        e = np.empty(self.n_chains, dtype=np.float64) if with_energy else None
        self._ck(self._lib.arianna_get_state(self._h, _ptr(x), _ptr(e)))
        return (x, e) if with_energy else x

    def set_state_f32(self, x):
        """Float32 ensembles: positions in their own element type (arianna_set_state_f32)."""
        x = np.ascontiguousarray(x, dtype=np.float32)
        if x.shape != (self.n_chains,):
            raise ValueError(f"x must have shape ({self.n_chains},)")
        self._ck(self._lib.arianna_set_state_f32(self._h, _ptr(x)))

    def get_state_f32(self, with_energy: bool = False):
        x = np.empty(self.n_chains, dtype=np.float32)
        e = np.empty(self.n_chains, dtype=np.float32) if with_energy else None
        self._ck(self._lib.arianna_get_state_f32(self._h, _ptr(x), _ptr(e)))
        return (x, e) if with_energy else x

    def get_state_async(self, x_pinned_ptr: int):
        self._ck(self._lib.arianna_get_state_async(self._h, C.c_void_p(x_pinned_ptr)))

    def copy_wait(self):
        """Wait for the last get_state_async frame only (arianna_copy_wait)."""
        self._ck(self._lib.arianna_copy_wait(self._h))

    def set_state_from_ptr(self, host_ptr: int):
        """set_state from a raw (e.g. pinned) host pointer holding n_chains float64."""
        self._ck(self._lib.arianna_set_state(self._h, C.c_void_p(host_ptr)))

    def get_state_to_ptr(self, host_ptr: int):
        self._ck(self._lib.arianna_get_state(self._h, C.c_void_p(host_ptr), None))

    def set_beta(self, beta: float):
        self._ck(self._lib.arianna_set_beta(self._h, float(beta)))
        self.beta = float(beta)

    def set_betas(self, betas):
        b = np.ascontiguousarray(betas, dtype=np.float64)
        if b.shape != (self.n_chains,):
            raise ValueError(f"betas must have shape ({self.n_chains},)")
        self._ck(self._lib.arianna_set_betas(self._h, _ptr(b)))

    # -- replica exchange across β ladders ----------------------------------------------------------------
    def set_ladder(self, betas):
        """β ladder of L = len(betas) rungs: chain g (global) gets betas[g % L] (arianna_set_ladder).  The shard must
        hold whole ladders."""
        b = np.ascontiguousarray(betas, dtype=np.float64)
        if b.ndim != 1:
            raise ValueError("betas must be a 1-d ladder")
        self._ck(self._lib.arianna_set_ladder(self._h, int(b.size), b.ctypes.data_as(C.POINTER(C.c_double))))
        self.ladder = b.copy()

    def _rungs(self) -> int:
        # without a ladder the library refuses the call; the buffer only has to be large enough until it does
        return self.ladder.size if self.ladder is not None else L.MAX_LADDER

    def replica_exchange(self):
        """One exchange round between neighbouring rungs, even/odd pairs alternating (asynchronous)."""
        self._ck(self._lib.arianna_replica_exchange(self._h))

    def exchange_counters(self):
        """(accepted[L-1], attempted[L-1], rounds) of the local shard; pair k is attempted in rounds R ≡ k (mod 2)."""
        n = self._rungs()
        acc = (C.c_int64 * (n - 1))()
        rounds = C.c_int64()
        self._ck(self._lib.arianna_exchange_counters(self._h, acc, C.byref(rounds)))
        R = rounds.value
        per_round = np.array([(R + 1) // 2 if k % 2 == 0 else R // 2 for k in range(n - 1)], dtype=np.int64)
        return np.array(acc[:], dtype=np.int64), (self.n_chains // n) * per_round, R

    def ladder_sums(self):
        """Per-rung callback records [L][2 + n_moves] = (Σe, Σ acc/tot per move, count) over the local shard."""
        out = np.empty((self._rungs(), 2 + self.n_moves), dtype=np.float64)
        self._ck(self._lib.arianna_ladder_sums(self._h, out.ctypes.data_as(C.POINTER(C.c_double))))
        return out

    # -- policy parameters --------------------------------------------------------------------------------
    def set_params(self, move_id: int, sigma: float, log_norm: Optional[float] = None):
        th = C.c_double(float(sigma))
        ln = C.c_double(float(log_norm)) if log_norm is not None else None
        self._ck(self._lib.arianna_set_params(self._h, int(move_id), C.byref(th), 1,
                                              C.byref(ln) if ln is not None else None))

    def get_params(self, move_id: int) -> float:
        th = C.c_double()
        self._ck(self._lib.arianna_get_params(self._h, int(move_id), C.byref(th), 1))
        return th.value

    # -- the hot path -------------------------------------------------------------------------------------
    def sweep(self, K: int, reduce: bool = False):
        """K fused mc steps per chain (asynchronous)."""
        self._ck(self._lib.arianna_sweep(self._h, int(K), L.SWEEP_REDUCE if reduce else 0))

    def sweep_series(self, Ks: Sequence[int], read: bool = True):
        """len(Ks) consecutive store intervals of Ks[i] mc steps, the callback record taken after each ON THE DEVICE
        (arianna_sweep_series).  read=True returns the local-shard records [n][2 + n_moves] = (Σe, Σ acc/tot per move,
        count); read=False leaves them on the device (series_tensor / series_global)."""
        ks = np.ascontiguousarray(Ks, dtype=np.int64)
        rec = np.empty((ks.size, 2 + self.n_moves), dtype=np.float64) if read else None
        self._ck(self._lib.arianna_sweep_series(self._h, int(ks.size), ks.ctypes.data_as(C.POINTER(C.c_int64)),
                                                _ptr(rec)))
        return rec

    def run_host_job(self, Ks: Sequence[int], x_in=None, x_out=None, n_slices: int = 8, read: bool = True):
        """A complete callbacks-only job with host buffers, pipelined over slices of the chains
        (arianna_run_host_job): chains in, len(Ks) store intervals, records out, chains out.  x_in / x_out: numpy
        arrays or raw pointers of page-locked host memory ([n_chains] f64), or None."""
        ks = np.ascontiguousarray(Ks, dtype=np.int64)
        rec = np.empty((ks.size, 2 + self.n_moves), dtype=np.float64) if read else None

        def ptr(a):
            if a is None:
                return None
            if isinstance(a, np.ndarray):
                assert a.dtype == np.float64 and a.size == self.n_chains and a.flags.c_contiguous
                return a.ctypes.data_as(C.c_void_p)
            return C.c_void_p(int(a))
        self._ck(self._lib.arianna_run_host_job(self._h, ptr(x_in), int(ks.size), ks.ctypes.data_as(C.POINTER(C.c_int64)),
                                                _ptr(rec), ptr(x_out), int(n_slices)))
        return rec

    def job_timing(self):
        """PCIe view of the last run_host_job: {"h2d_ms", "h2d_gbs", "d2h_ms", "d2h_gbs"} (arianna_job_timing)."""
        v = [C.c_double() for _ in range(4)]
        self._ck(self._lib.arianna_job_timing(self._h, *[C.byref(x) for x in v]))
        return dict(zip(("h2d_ms", "h2d_gbs", "d2h_ms", "d2h_gbs"), (x.value for x in v)))

    @property
    def series_per_launch(self) -> int:
        """Store intervals one sweep_series launch fuses for this ensemble (arianna_series_per_launch)."""
        n = C.c_int32()
        self._ck(self._lib.arianna_series_per_launch(self._h, C.byref(n)))
        return n.value

    def series_tensor(self):
        """torch view (no copy) of the device records of the last sweep_series call, for ONE in-place all_reduce."""
        import torch
        p = C.c_void_p()
        n = C.c_int32()
        self._ck(self._lib.arianna_series_device(self._h, C.byref(p), C.byref(n)))
        return torch.as_tensor(_DeviceBuffer(p.value, n.value, self.stream_ptr), device="cuda")

    def series_global(self, n_stores: int):
        """Records of the last sweep_series call all-reduced inside the library (arianna_comm_init)."""
        rec = np.empty((int(n_stores), 2 + self.n_moves), dtype=np.float64)
        self._ck(self._lib.arianna_series_global(self._h, int(n_stores), _ptr(rec)))
        return rec

    def series_global_begin(self, n_stores: int, records_pinned_ptr: int):
        """Asynchronous series_global: all-reduce + D2H into page-locked memory on a side stream, overlapping the next
        sweep (arianna_series_global_begin); series_global_wait() / synchronize() completes it."""
        self._ck(self._lib.arianna_series_global_begin(self._h, int(n_stores), C.c_void_p(int(records_pinned_ptr))))

    def series_global_wait(self):
        self._ck(self._lib.arianna_series_global_wait(self._h))

    def sweep_replay(self, u_cat, z, u_acc, want_decisions: bool = False):
        z = np.ascontiguousarray(z, dtype=np.float64)
        u_acc = np.ascontiguousarray(u_acc, dtype=np.float64)
        K = z.shape[0]
        if z.shape != (K, self.n_chains) or u_acc.shape != z.shape:
            raise ValueError("draw arrays must be step-major [K][n_chains]")
        if u_cat is not None:
            u_cat = np.ascontiguousarray(u_cat, dtype=np.float64)
            if u_cat.shape != z.shape:
                raise ValueError("u_cat must be [K][n_chains]")
        dec = np.empty((K, self.n_chains), dtype=np.uint8) if want_decisions else None
        self._ck(self._lib.arianna_sweep_replay(self._h, K, _ptr(u_cat), _ptr(z), _ptr(u_acc), _ptr(dec), 0))
        return dec

    def sweep_replay_device(self, K: int, u_cat_ptr: int, z_ptr: int, u_acc_ptr: int, decisions_ptr: int = 0):
        self._ck(self._lib.arianna_sweep_replay(self._h, int(K), C.c_void_p(u_cat_ptr or None), C.c_void_p(z_ptr),
                                                C.c_void_p(u_acc_ptr), C.c_void_p(decisions_ptr or None), 1))

    # -- XOSHIRO mode -------------------------------------------------------------------------------------
    def set_rng_state(self, states):
        s = np.ascontiguousarray(states, dtype=np.uint64)
        if s.shape != (self.n_chains, 4):
            raise ValueError("states must be [n_chains][4] uint64")
        self._ck(self._lib.arianna_set_rng_state(self._h, _ptr(s)))

    def get_rng_state(self):
        s = np.empty((self.n_chains, 4), dtype=np.uint64)
        self._ck(self._lib.arianna_get_rng_state(self._h, _ptr(s)))
        return s

    def set_ziggurat_tables(self, ki, wi, fi):
        ki = np.ascontiguousarray(ki, dtype=np.uint64)
        wi = np.ascontiguousarray(wi, dtype=np.float64)
        fi = np.ascontiguousarray(fi, dtype=np.float64)
        assert ki.shape == wi.shape == fi.shape == (256,)
        self._ck(self._lib.arianna_set_ziggurat_tables(self._h, _ptr(ki), _ptr(wi), _ptr(fi)))

    # -- callbacks ----------------------------------------------------------------------------------------
    def callbacks(self):
        """(mean energy, per-move mean acceptance) over the LOCAL shard."""
        me = C.c_double()
        acc = (C.c_double * self.n_moves)()
        self._ck(self._lib.arianna_callbacks(self._h, C.byref(me), acc))
        return me.value, np.array(acc[:], dtype=np.float64)

    def callback_sums(self):
        s = (C.c_double * (2 + self.n_moves))()
        self._ck(self._lib.arianna_callback_sums(self._h, s))
        return np.array(s[:], dtype=np.float64)

    def callback_sums_device(self):
        """(device pointer, n) of [Σe, Σ acc/tot per move, count] -- valid until the next sweep."""
        p = C.c_void_p()
        n = C.c_int32()
        self._ck(self._lib.arianna_callback_sums_device(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def callback_sums_tensor(self):
        """torch view (no copy) of the device sums, for an in-place dist.all_reduce."""
        import torch
        p, n = self.callback_sums_device()
        return torch.as_tensor(_DeviceBuffer(p, n, self.stream_ptr), device="cuda")

    def counters(self):
        acc = (C.c_int64 * self.n_moves)()
        tot = (C.c_int64 * self.n_moves)()
        self._ck(self._lib.arianna_get_counters(self._h, acc, tot))
        return np.array(acc[:], dtype=np.int64), np.array(tot[:], dtype=np.int64)

    def chain_counters(self):
        acc = np.empty((self.n_moves, self.n_chains), dtype=np.uint32)
        tot = np.empty((self.n_moves, self.n_chains), dtype=np.uint32)
        self._ck(self._lib.arianna_get_chain_counters(self._h, _ptr(acc), _ptr(tot)))
        return acc, tot

    # -- PGMC ---------------------------------------------------------------------------------------------
    def pgmc_estimate(self, q_batch: int, learn_ids: Sequence[int]):
        ids = (C.c_int32 * len(learn_ids))(*[int(i) for i in learn_ids])
        self._ck(self._lib.arianna_pgmc_estimate(self._h, int(q_batch), ids, len(learn_ids)))

    def pgmc_estimate_replay(self, q_batch: int, learn_ids: Sequence[int], z):
        z = np.ascontiguousarray(z, dtype=np.float64)
        if z.shape != (len(learn_ids), q_batch, self.n_chains):
            raise ValueError("z must be [n_learn][q_batch][n_chains]")
        ids = (C.c_int32 * len(learn_ids))(*[int(i) for i in learn_ids])
        self._ck(self._lib.arianna_pgmc_estimate_replay(self._h, int(q_batch), ids, len(learn_ids), _ptr(z), 0))

    def pgmc_read(self, n_learn: int):
        """Accumulated SUMS [n_learn][5] = (j, ∇j, ∇logq_forward, g, n) of the local shard."""
        out = (L.GradientData * n_learn)()
        self._ck(self._lib.arianna_pgmc_read(self._h, out, n_learn))
        return np.array([[r.j, r.dj, r.dlogq_forward, r.g, r.n] for r in out], dtype=np.float64).reshape(n_learn, 5)

    def pgmc_reset(self):
        self._ck(self._lib.arianna_pgmc_reset(self._h))

    def pgmc_update_device(self, learn_ids: Sequence[int], optimisers):
        """PolicyGradientUpdate on the device (arianna_pgmc_update_device): `optimisers` = one (kind, p1, p2) per
        learnable move, kind a name of learning.jl ("VPG", "BLPG", "BLAPG", "NPG", "ANPG", "BLANPG", "Static").
        Asynchronous; get_params / params_sync refresh the host copy."""
        n = len(learn_ids)
        ids = (C.c_int32 * n)(*[int(i) for i in learn_ids])
        opts = (L.Optimiser * n)()
        for o, (kind, p1, p2) in zip(opts, optimisers):
            o.kind, o.p1, o.p2 = L.OPT_KINDS[kind], float(p1), float(p2)
        self._ck(self._lib.arianna_pgmc_update_device(self._h, ids, opts, n))

    def params_sync(self):
        self._ck(self._lib.arianna_params_sync(self._h))

    def pgmc_sums_tensor(self):
        import torch
        p = C.c_void_p()
        n = C.c_int32()
        self._ck(self._lib.arianna_pgmc_sums_device(self._h, C.byref(p), C.byref(n)))
        return torch.as_tensor(_DeviceBuffer(p.value, n.value, self.stream_ptr), device="cuda")

    # -- NCCL inside the library (hosts without torch.distributed) -------------------------------------------
    @staticmethod
    def nccl_unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        L.check(None, L.load().arianna_nccl_unique_id(buf))
        return buf.raw

    def comm_init(self, unique_id: bytes, rank: int, n_ranks: int):
        buf = C.create_string_buffer(unique_id, 128)
        self._ck(self._lib.arianna_comm_init(self._h, buf, int(rank), int(n_ranks)))

    def callbacks_global(self):
        me = C.c_double()
        acc = (C.c_double * self.n_moves)()
        self._ck(self._lib.arianna_callbacks_global(self._h, C.byref(me), acc))
        return me.value, np.array(acc[:], dtype=np.float64)

    def pgmc_read_global(self, n_learn: int):
        out = (L.GradientData * n_learn)()
        self._ck(self._lib.arianna_pgmc_read_global(self._h, out, n_learn))
        return np.array([[r.j, r.dj, r.dlogq_forward, r.g, r.n] for r in out], dtype=np.float64).reshape(n_learn, 5)

    # -- plumbing -----------------------------------------------------------------------------------------
    @property
    def stream_ptr(self) -> int:
        s = C.c_void_p()
        self._ck(self._lib.arianna_get_stream(self._h, C.byref(s)))
        return s.value or 0

    def torch_stream(self):
        """The engine's stream as a torch.cuda.ExternalStream (events / NCCL ordering on the launching stream)."""
        import torch
        return torch.cuda.ExternalStream(self.stream_ptr)

    def synchronize(self):
        self._ck(self._lib.arianna_synchronize(self._h))

    def timing(self):
        """(sweep_ms, pgmc_ms): device time of the last sweep / series / host job and of the last estimator pass
        (arianna_timing; NaN when there was none)."""
        a, b = C.c_double(), C.c_double()
        self._ck(self._lib.arianna_timing(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    @property
    def launch_count(self) -> int:
        n = C.c_int64()
        self._ck(self._lib.arianna_launch_count(self._h, C.byref(n)))
        return n.value

    @property
    def steps_done(self) -> int:
        n = C.c_int64()
        self._ck(self._lib.arianna_steps_done(self._h, C.byref(n)))
        return n.value

    def device_info(self):
        sm, ma, mi, hb = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
        self._ck(self._lib.arianna_device_info(self._h, C.byref(sm), C.byref(ma), C.byref(mi), C.byref(hb)))
        return {"sm_count": sm.value, "cc": (ma.value, mi.value), "hbm_bytes": hb.value}

    def debug_math(self, kind: int, a=None, b=None, c=None):
        """Evaluate the device math layer on arrays (arianna_debug_math)."""
        arrs = [None if v is None else np.ascontiguousarray(v, dtype=t)
                for v, t in ((a, np.float64), (b, np.uint64), (c, np.uint64))]
        n = next(v.size for v in arrs if v is not None)
        out = np.empty(4 * n if kind in (6, 7) else n if (kind == 9 or kind < 3) else 2 * n, dtype=np.float64)
        self._ck(self._lib.arianna_debug_math(self._h, int(kind), _ptr(arrs[0]), _ptr(arrs[1]), _ptr(arrs[2]),
                                              _ptr(out), n))
        return out

    def measure_fp64_peak(self) -> float:
        v = C.c_double()
        self._ck(self._lib.arianna_measure_fp64_peak(self._h, C.byref(v)))
        return v.value
