"""TEST INFRASTRUCTURE ONLY - ctypes front-end of ``oracle/spgg_oracle.c``.

Used by ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline
legs as the *checker*; never imported by the product package.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libspgg_oracle.so")
NSTAT = 40

# column indices of a stat row (mirror of spgg_oracle.h / include/spgg.h)
ST = dict(NC_OLD=0, N_CD=1, N_DC=2, NC_NEW=3, SUM_P=4, SUM_P_C=5, SUM_P_D=6, SUM_WP_P=7,
          SUM_REW_C=8, SUM_REW_D=9, SUM_RATIO=10, GROUP0=11, SUM_R=17, SUM_Q=18,
          SUM_Q_C=22, SUM_Q_D=26, SUM_NI=30, N_BEST_POS=31, N_BEST_2ND=32, GMAX=33)
# TD rule codes (include/spgg.h: SPGG_ALGO_*) and the draw pairs each consumes per iteration
ALGOS = {"qlearning": 0, "sarsa": 1, "expected_sarsa": 2, "double_qlearning": 3}
PAIRS = {0: 1, 1: 3, 2: 1, 3: 2}


class OracleParams(C.Structure):
    _fields_ = [("L", C.c_int32), ("M", C.c_int32), ("state_mode", C.c_int32),
                ("algorithm", C.c_int32),
                ("r", C.c_double), ("c", C.c_double), ("cost", C.c_double),
                ("alpha", C.c_double), ("gamma", C.c_double), ("kappa", C.c_double),
                ("lambda_eps", C.c_double), ("rep_gain_C", C.c_double),
                ("delta_R_D", C.c_double), ("R_min", C.c_double), ("R_max", C.c_double),
                ("wP", C.c_double)]


def build(force: bool = False) -> str:
    srcs = [os.path.join(_HERE, f) for f in ("spgg_oracle.c", "spgg_oracle.h")]
    if force or not os.path.exists(_LIB_PATH) or any(
            os.path.exists(s) and os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in srcs):
        subprocess.check_call(["make", "-C", _HERE, "-s", "libspgg_oracle.so"])
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB_PATH)
        dp = C.POINTER(C.c_double)
        for name, qt in (("oracle_step_f64", C.c_double), ("oracle_step_f32", C.c_float)):
            fn = getattr(_lib, name)
            fn.restype = C.c_int
            fn.argtypes = [C.POINTER(OracleParams), C.c_void_p, C.c_void_p, C.c_void_p,
                           C.c_double, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32,
                           C.c_uint32, dp]
        _lib.oracle_philox4x32_10.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.oracle_site_word.restype = C.c_uint32
        _lib.oracle_site_word.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_int]
        _lib.oracle_thr24.restype = C.c_uint32
        _lib.oracle_thr24.argtypes = [C.c_double]
        _lib.oracle_reward_table.argtypes = [C.POINTER(OracleParams), C.c_void_p]
        _lib.oracle_num_threads.restype = C.c_int
        i32, vp = C.c_int, C.c_void_p
        _lib.oracle_state_digest.argtypes = [i32, i32, i32, i32, i32, vp, vp, vp, vp, vp]
        _lib.oracle_digest_weights.argtypes = [i32, i32, i32, i32, i32, vp]
        _lib.oracle_init_random.argtypes = [i32, i32, i32, i32, i32, C.c_uint64, vp, vp, vp]
        _lib.oracle_init_random.restype = None
        _lib.oracle_init_random_digest.argtypes = [i32, i32, i32, i32, i32, C.c_uint64, vp]
        _lib.oracle_explore_actions.argtypes = [i32, i32, i32, C.c_uint64, C.c_uint32, vp]
        _lib.oracle_explore_actions.restype = None
    return _lib


def params_from_dict(p: dict) -> OracleParams:
    """``p`` uses the reference ctor's argument names (spgg.py:50-56)."""
    return OracleParams(
        L=int(p["L"]), M=2 if p.get("use_second_order", True) else 1,
        state_mode=1 if p.get("state_representation", "reputation") == "action" else 0,
        algorithm=ALGOS[str(p.get("algorithm", "qlearning")).lower()],
        r=float(p["r"]), c=float(p.get("c", 1)), cost=float(p.get("cost", 0.5)),
        alpha=float(p.get("alpha", 0.1)), gamma=float(p.get("gamma", 0.9)),
        kappa=float(p.get("influence_factor", 1.0)),
        lambda_eps=float(p.get("lambda_epsilon", 0.01)),
        rep_gain_C=float(p.get("rep_gain_C", 0.5)), delta_R_D=float(p.get("delta_R_D", 1)),
        R_min=float(p.get("R_min", -10)), R_max=float(p.get("R_max", 10)),
        wP=float(p.get("reward_weight_payoff", 1.0)))


def philox(ctr, key):
    c = np.asarray(ctr, np.uint32)
    k = np.asarray(key, np.uint32)
    out = np.zeros(4, np.uint32)
    lib().oracle_philox4x32_10(c.ctypes.data, k.ctypes.data, out.ctypes.data)
    return out


def site_word(seed: int, step: int, stream: int, i: int, j: int) -> int:
    """The Philox word the step functions draw for site (i, j) (spgg_oracle.h)."""
    return int(lib().oracle_site_word(int(seed), int(step), int(stream), int(i), int(j)))


def thr24(eps: float) -> int:
    return int(lib().oracle_thr24(float(eps)))


def reward_table(p: dict) -> np.ndarray:
    tab = np.zeros(128, np.float32)
    op = params_from_dict(p)
    lib().oracle_reward_table(C.byref(op), tab.ctypes.data)
    return tab


def _digest_shape(L, rows, period):
    return (period, period) if period else (rows, L)


def digest_weights(L: int, nq: int, period: int | None = None, row0: int = 0, rows: int | None = None):
    """The multipliers ``state_digest`` applies, one set per value slot: (P, P, 2 + nq) uint64 for a
    lattice of period P, else (rows, L, 2 + nq).  Computing them is the costly part of a digest;
    pass them back to ``state_digest`` to digest many states of the same geometry."""
    rows = L if rows is None else int(rows)
    w = np.empty(_digest_shape(L, rows, period) + (2 + nq,), np.uint64)
    if lib().oracle_digest_weights(int(L), int(row0), rows, int(period or 0), int(nq), w.ctypes.data):
        raise ValueError(f"period {period} does not divide L = {L}")
    return w


def state_digest(S, R, Q=None, L: int | None = None, row0: int = 0, period: int | None = None,
                 weights=None):
    """``Engine.digest`` of a host state (include/spgg.h: spgg_state_digest): S (rows, L) 0/1, R (rows, L)
    and Q (rows, L, 2, 2[, 2]) as ``Engine.get_state`` returns them, the rows starting at global row
    ``row0``.  With ``period`` = P the arrays hold a P x P state and the digest is that of the L x L
    lattice tiled with it.  Q = None digests S and R only (the Q word is 0)."""
    S = np.ascontiguousarray(S, np.uint8)
    R = np.ascontiguousarray(R, np.float64)
    rows, width = S.shape
    L = width if L is None else int(L)
    if R.shape != S.shape or _digest_shape(L, rows, period) != S.shape:
        raise ValueError(f"S {S.shape} and R {R.shape} do not describe the geometry (L={L}, period={period})")
    nq = 4
    if Q is not None:
        Q = np.ascontiguousarray(Q, np.float64)
        nq = Q.size // S.size
        if nq not in (4, 8) or Q.size != nq * S.size:
            raise ValueError(f"Q must hold 4 or 8 values per site, got shape {Q.shape}")
    if weights is not None and weights.shape != S.shape + (2 + nq,):
        raise ValueError(f"weights {weights.shape} do not match the state")
    out = np.zeros(3, np.uint64)
    rc = lib().oracle_state_digest(int(L), int(row0), rows, int(period or 0), nq,
                                   S.ctypes.data, R.ctypes.data, None if Q is None else Q.ctypes.data,
                                   None if weights is None else np.ascontiguousarray(weights).ctypes.data,
                                   out.ctypes.data)
    if rc:
        raise ValueError(f"period {period} does not divide L = {L}")
    return tuple(int(x) for x in out)


def init_random(L: int, seed: int, nq: int = 4, precision: str = "fp32", row0: int = 0, rows: int | None = None):
    """``Engine.init_random(seed)`` restated on the host: (S, R, Q) of rows [row0, row0 + rows) in the
    layout of ``Engine.get_state``."""
    rows = L if rows is None else int(rows)
    S = np.empty((rows, L), np.uint8)
    R = np.empty((rows, L), np.float64)
    Q = np.empty((rows, L, 2, 2) if nq == 4 else (rows, L, 2, 2, 2), np.float64)
    lib().oracle_init_random(int(L), int(row0), rows, int(nq), int(precision == "fp32"), int(seed) & (2 ** 64 - 1),
                             S.ctypes.data, R.ctypes.data, Q.ctypes.data)
    return S, R, Q


def init_random_digest(L: int, seed: int, nq: int = 4, precision: str = "fp32", row0: int = 0,
                       rows: int | None = None):
    """``state_digest(*init_random(...))`` without holding the state: for lattices beyond host memory."""
    rows = L if rows is None else int(rows)
    out = np.zeros(3, np.uint64)
    if lib().oracle_init_random_digest(int(L), int(row0), rows, int(nq), int(precision == "fp32"),
                                       int(seed) & (2 ** 64 - 1), out.ctypes.data):
        raise ValueError(f"nq must be 4 or 8, got {nq}")
    return tuple(int(x) for x in out)


def explore_actions(L: int, seed: int, step: int, i0: int, i1: int):
    """Actions (0 = C, 1 = D) of rows [i0, i1) at iteration ``step`` when epsilon = 1: every site explores
    and takes bit 0 of its stream-0 Philox word (``site_word``)."""
    a = np.empty((i1 - i0, L), np.uint8)
    lib().oracle_explore_actions(int(L), int(i0), int(i1), int(seed) & (2 ** 64 - 1), int(step), a.ctypes.data)
    return a


class Sim:
    """Stateful driver: holds S (uint8), R, Q and steps them with either
    arithmetic.  ``precision`` = 'fp64' (reference order) or 'fp32'
    (throughput-mode arithmetic).  ``p['algorithm']`` picks the TD rule; Double
    Q-learning holds both tables, ``Q`` of shape (L, L, 2, 2, 2) laid out
    [site][table][s][a] like ``Engine.get_state``."""

    def __init__(self, p: dict, S0, R0, Q0, precision="fp64", seed=0):
        self.p = dict(p)
        self.op = params_from_dict(p)
        self.L = int(p["L"])
        self.precision = precision
        self.pairs = PAIRS[self.op.algorithm]
        ft = np.float64 if precision == "fp64" else np.float32
        self.S = np.ascontiguousarray(np.asarray(S0) != 0, dtype=np.uint8)
        self.R = np.array(R0, dtype=ft, order="C")          # copies: the caller's arrays stay as they are
        qshape = (self.L, self.L, 2, 2, 2) if self.op.algorithm == 3 else (self.L, self.L, 2, 2)
        if np.asarray(Q0).size != np.prod(qshape):
            raise ValueError(f"Q0 must hold {qshape} values for this TD rule")
        self.Q = np.array(np.asarray(Q0).reshape(qshape), dtype=ft, order="C")
        self.eps = float(p.get("epsilon", 0.5))
        self.decay = float(p.get("epsilon_decay", 0.995))
        self.eps_min = float(p.get("epsilon_min", 0.01))
        self.seed = int(seed)
        self.t = 0
        self.fn = lib().oracle_step_f64 if precision == "fp64" else lib().oracle_step_f32

    @property
    def q_combined(self):
        """The table the policy acts on: Q itself, or the mean of Double Q's two tables."""
        if self.Q.ndim == 5:
            return (self.Q[:, :, 0] + self.Q[:, :, 1]) / self.Q.dtype.type(2)
        return self.Q

    def step(self, u=None, b=None):
        """One iteration; returns the stat row (NSTAT doubles).  Replayed draws: ``u``, ``b`` of
        shape (L, L), or (pairs, L, L) with the pairs the TD rule consumes (SARSA 3, Double Q 2:
        u of pair 1 chooses the table, spgg_oracle.h)."""
        self.t += 1
        st = np.zeros(NSTAT)
        if u is not None:
            u = np.ascontiguousarray(u, np.float64)
            b = np.ascontiguousarray(b, np.uint8)
            if u.size != self.pairs * self.L * self.L or b.size != u.size:
                raise ValueError(f"this TD rule consumes {self.pairs} draw pair(s) per iteration")
            up, bp = u.ctypes.data, b.ctypes.data
        else:
            up = bp = None
        rc = self.fn(C.byref(self.op), self.S.ctypes.data, self.R.ctypes.data,
                     self.Q.ctypes.data, self.eps, up, bp, self.seed, self.t,
                     thr24(self.eps), st.ctypes.data_as(C.POINTER(C.c_double)))
        assert rc == 0
        self.eps = max(self.eps * self.decay, self.eps_min)  # algorithms.py:42
        return st

    def run(self, n, draws=None):
        """``draws(t, L) -> (u, b)`` (shapes as ``step``) or None for Philox.  Stops like spgg.py:405
        when the lattice is uniform.  Returns the stat rows of completed steps."""
        rows = []
        for _ in range(n):
            nC = int((self.S == 0).sum())
            if nC == 0 or nC == self.L * self.L:
                break
            if draws is not None:
                u, b = draws(self.t + 1, self.L)
                rows.append(self.step(u, b))
            else:
                rows.append(self.step())
        return np.array(rows).reshape(-1, NSTAT)
