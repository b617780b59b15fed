"""ctypes binding of libarianna_cuda.so (include/arianna_cuda.h).  Loading fails loudly when the library is
missing -- there is no CPU path in this package."""
from __future__ import annotations

import ctypes as C
import os

from ._build import LIB_PATH

MAX_MOVES = 16
MAX_LADDER = 256
MAX_HISTOGRAM_CELLS = 16384

OK, ERR_INVALID, ERR_CUDA, ERR_NOMEM, ERR_UNSUPPORTED, ERR_NO_DEVICE, ERR_NCCL = range(7)
POT_HARMONIC, POT_QUARTIC, POT_DOUBLE_WELL = 0, 1, 2
RNG_PHILOX, RNG_XOSHIRO = 0, 1
ARITH_EXACT, ARITH_FAST = 0, 1
SWEEP_REDUCE = 1
OBS_X, OBS_E = 0, 1

POTENTIALS = {"harmonic": POT_HARMONIC, "quartic": POT_QUARTIC, "double_well": POT_DOUBLE_WELL}
RNG_MODES = {"philox": RNG_PHILOX, "xoshiro": RNG_XOSHIRO}
ARITH_MODES = {"exact": ARITH_EXACT, "fast": ARITH_FAST}
DTYPES = {"f64": 0, "f32": 1}
OBSERVABLES = {"x": OBS_X, "e": OBS_E}


class Config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("device", C.c_int32),
        ("n_chains", C.c_int64),
        ("chain_offset", C.c_int64),
        ("n_chains_total", C.c_int64),
        ("seed", C.c_int64),
        ("beta", C.c_double),
        ("potential", C.c_int32),
        ("n_moves", C.c_int32),
        ("sigma", C.c_double * MAX_MOVES),
        ("weight", C.c_double * MAX_MOVES),
        ("rng_mode", C.c_int32),
        ("arith_mode", C.c_int32),
        ("stream", C.c_void_p),
        ("dtype", C.c_int32),
        ("reserved", C.c_int32),
    ]


class GradientData(C.Structure):
    _fields_ = [("j", C.c_double), ("dj", C.c_double), ("dlogq_forward", C.c_double), ("g", C.c_double),
                ("n", C.c_double)]


class Optimiser(C.Structure):
    _fields_ = [("kind", C.c_int32), ("reserved", C.c_int32), ("p1", C.c_double), ("p2", C.c_double)]


OPT_KINDS = {"Static": 0, "VPG": 1, "BLPG": 2, "BLAPG": 3, "NPG": 4, "ANPG": 5, "BLANPG": 6}


class AriannaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libarianna_cuda error {code}: {msg}")
        self.code = code


# every symbol include/arianna_cuda.h declares: (restype, argtypes)
_H = C.c_void_p
_D = C.POINTER(C.c_double)
SYMBOLS = {
    "arianna_abi_version": (C.c_uint32, []),
    "arianna_last_error": (C.c_char_p, [_H]),
    "arianna_create": (C.c_int32, [C.POINTER(Config), C.POINTER(_H)]),
    "arianna_destroy": (C.c_int32, [_H]),
    "arianna_set_state": (C.c_int32, [_H, C.c_void_p]),
    "arianna_init_synthetic": (C.c_int32, [_H, C.c_int64]),
    "arianna_get_state": (C.c_int32, [_H, C.c_void_p, C.c_void_p]),
    "arianna_set_state_f32": (C.c_int32, [_H, C.c_void_p]),
    "arianna_get_state_f32": (C.c_int32, [_H, C.c_void_p, C.c_void_p]),
    "arianna_get_state_async": (C.c_int32, [_H, C.c_void_p]),
    "arianna_copy_wait": (C.c_int32, [_H]),
    "arianna_host_alloc": (C.c_int32, [C.c_int64, C.c_int32, C.POINTER(C.c_void_p)]),
    "arianna_host_free": (C.c_int32, [C.c_void_p]),
    "arianna_set_beta": (C.c_int32, [_H, C.c_double]),
    "arianna_set_betas": (C.c_int32, [_H, C.c_void_p]),
    "arianna_set_ladder": (C.c_int32, [_H, C.c_int32, _D]),
    "arianna_replica_exchange": (C.c_int32, [_H]),
    "arianna_exchange_counters": (C.c_int32, [_H, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "arianna_ladder_sums": (C.c_int32, [_H, _D]),
    "arianna_set_histogram": (C.c_int32, [_H, C.c_int32, C.c_double, C.c_double, C.c_int32, C.c_int32]),
    "arianna_histogram_accumulate": (C.c_int32, [_H]),
    "arianna_histogram_read": (C.c_int32, [_H, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]),
    "arianna_histogram_reset": (C.c_int32, [_H]),
    "arianna_set_params": (C.c_int32, [_H, C.c_int32, _D, C.c_int32, _D]),
    "arianna_get_params": (C.c_int32, [_H, C.c_int32, _D, C.c_int32]),
    "arianna_sweep": (C.c_int32, [_H, C.c_int64, C.c_uint32]),
    "arianna_sweep_series": (C.c_int32, [_H, C.c_int32, C.POINTER(C.c_int64), C.c_void_p]),
    "arianna_series_device": (C.c_int32, [_H, C.POINTER(C.c_void_p), C.POINTER(C.c_int32)]),
    "arianna_series_global": (C.c_int32, [_H, C.c_int32, C.c_void_p]),
    "arianna_series_per_launch": (C.c_int32, [_H, C.POINTER(C.c_int32)]),
    "arianna_run_host_job": (C.c_int32, [_H, C.c_void_p, C.c_int32, C.POINTER(C.c_int64), C.c_void_p, C.c_void_p,
                                         C.c_int32]),
    "arianna_job_timing": (C.c_int32, [_H, _D, _D, _D, _D]),
    "arianna_sweep_replay": (C.c_int32, [_H, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]),
    "arianna_set_rng_state": (C.c_int32, [_H, C.c_void_p]),
    "arianna_get_rng_state": (C.c_int32, [_H, C.c_void_p]),
    "arianna_set_ziggurat_tables": (C.c_int32, [_H, C.c_void_p, C.c_void_p, C.c_void_p]),
    "arianna_callbacks": (C.c_int32, [_H, _D, _D]),
    "arianna_callback_sums": (C.c_int32, [_H, _D]),
    "arianna_callback_sums_device": (C.c_int32, [_H, C.POINTER(C.c_void_p), C.POINTER(C.c_int32)]),
    "arianna_get_counters": (C.c_int32, [_H, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "arianna_get_chain_counters": (C.c_int32, [_H, C.c_void_p, C.c_void_p]),
    "arianna_pgmc_estimate": (C.c_int32, [_H, C.c_int32, C.POINTER(C.c_int32), C.c_int32]),
    "arianna_pgmc_estimate_replay": (C.c_int32, [_H, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.c_void_p, C.c_int32]),
    "arianna_pgmc_read": (C.c_int32, [_H, C.POINTER(GradientData), C.c_int32]),
    "arianna_pgmc_reset": (C.c_int32, [_H]),
    "arianna_pgmc_update_device": (C.c_int32, [_H, C.POINTER(C.c_int32), C.POINTER(Optimiser), C.c_int32]),
    "arianna_params_sync": (C.c_int32, [_H]),
    "arianna_pgmc_sums_device": (C.c_int32, [_H, C.POINTER(C.c_void_p), C.POINTER(C.c_int32)]),
    "arianna_get_stream": (C.c_int32, [_H, C.POINTER(C.c_void_p)]),
    "arianna_synchronize": (C.c_int32, [_H]),
    "arianna_timing": (C.c_int32, [_H, _D, _D]),
    "arianna_launch_count": (C.c_int32, [_H, C.POINTER(C.c_int64)]),
    "arianna_steps_done": (C.c_int32, [_H, C.POINTER(C.c_int64)]),
    "arianna_device_info": (C.c_int32, [_H, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                        C.POINTER(C.c_int64)]),
    "arianna_measure_fp64_peak": (C.c_int32, [_H, _D]),
    "arianna_nccl_unique_id": (C.c_int32, [C.c_void_p]),
    "arianna_comm_init": (C.c_int32, [_H, C.c_void_p, C.c_int32, C.c_int32]),
    "arianna_callbacks_global": (C.c_int32, [_H, _D, _D]),
    "arianna_series_global_begin": (C.c_int32, [_H, C.c_int32, C.c_void_p]),
    "arianna_series_global_wait": (C.c_int32, [_H]),
    "arianna_pgmc_read_global": (C.c_int32, [_H, C.POINTER(GradientData), C.c_int32]),
    "arianna_debug_math": (C.c_int32, [_H, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
}

_lib = None


def load() -> C.CDLL:
    """dlopen the in-tree library and bind every declared symbol.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(needs nvcc).  montecarlo_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library ever disagree
        fn.restype = res
        fn.argtypes = args
    if lib.arianna_abi_version() != 2:
        raise ImportError("libarianna_cuda.so ABI version mismatch")
    _lib = lib
    return lib


def check(handle, code):
    if code != OK:
        msg = load().arianna_last_error(handle)
        raise AriannaError(code, msg.decode() if msg else "?")
