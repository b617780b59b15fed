"""CPU references of the engine's replica exchange, for the tests: `exchange_oracle.c` (libm exp, compiled here with
gcc into a per-user temporary directory, so the repository tree stays untouched) and an independent numpy restatement
of the same round.  Both act on an `oracle.oracle.Ensemble` (its x, e and Move counters)."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle_np as N

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "exchange_oracle.c")
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        tag = hashlib.sha256(src).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"exchange_oracle_{os.getuid()}_{tag}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-fvisibility=hidden",
                                   "-std=c11", "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, so)                 # atomic: concurrent test processes may build it at the same time
        _lib = C.CDLL(so)
        _lib.xo_exchange_uniform.restype = C.c_double
        _lib.xo_exchange_uniform.argtypes = [C.c_uint64, C.c_uint64]
    return _lib


def _p(a, ty):
    return a.ctypes.data_as(C.POINTER(ty))


def exchange(ens, L, seed, R, offset=0, betas=None):
    """Round R of ladders of L chains on `ens` (x and e in place); `offset` is the global index of its chain 0, β the
    per-chain `betas` (default: ens.beta everywhere).  Returns the swaps per rung pair."""
    b = np.ascontiguousarray(np.full(ens.M, ens.beta) if betas is None else betas, dtype=np.float64)
    assert b.shape == (ens.M,) and ens.M % L == 0 and offset % L == 0
    acc = np.zeros(L - 1, dtype=np.int64)
    lib().xo_exchange_round(C.c_int64(ens.M), C.c_int(L), C.c_int64(seed), C.c_int64(offset), C.c_int64(R),
                            C.c_int(ens.pot), _p(ens.x, C.c_double), _p(ens.e, C.c_double), _p(b, C.c_double),
                            _p(acc, C.c_int64))
    return acc


def ladder_sums(ens, L):
    """Per-rung callback records [L][2 + n_moves] = (Σ e, Σ acc/tot per move, count)."""
    out = np.empty((L, 2 + ens.n_moves), dtype=np.float64)
    lib().xo_ladder_sums(C.c_int64(ens.M), C.c_int(L), C.c_int(ens.n_moves), _p(ens.e, C.c_double),
                         _p(ens.acc, C.c_int64), _p(ens.tot, C.c_int64), _p(out, C.c_double))
    return out


def exchange_uniform(sid, R):
    return lib().xo_exchange_uniform(int(sid), int(R))


def _potential(pot, x):
    if pot == 0:
        return x * x
    if pot == 1:
        x2 = x * x
        return x2 * x2
    w = x * x - 1.0
    return w * w


def exchange_round_np(x, betas, L, seed, offset, R, pot):
    """The same round in numpy (Philox from oracle_np, np.exp): x in place; returns swaps per rung pair."""
    M = x.size
    r = np.arange(R & 1, L - 1, 2)
    g = (np.arange(0, M, L)[:, None] + r[None, :]).ravel()
    sid = np.uint64(seed + offset) + g.astype(np.uint64)
    c0, c1, _, _ = N.philox4x32_10(sid & np.uint64(0xFFFFFFFF), np.full(g.size, R & 0xFFFFFFFF),
                                   sid >> np.uint64(32), np.full(g.size, (R >> 32) << 8), 4, 0x41524941)
    A = c0 | (c1 << np.uint64(32))
    u = (A >> np.uint64(11)).astype(np.float64) * 2.0 ** -53
    with np.errstate(over="ignore", invalid="ignore"):
        e0, e1 = _potential(pot, x[g]), _potential(pot, x[g + 1])
        ex = np.exp((betas[g] - betas[g + 1]) * (e0 - e1))
        a = np.where(ex > 1.0, 1.0, ex)
    sw = a > u
    gs = g[sw]
    x[gs], x[gs + 1] = x[gs + 1].copy(), x[gs].copy()
    acc = np.zeros(L - 1, dtype=np.int64)
    np.add.at(acc, np.tile(r, M // L)[sw], 1)
    return acc
