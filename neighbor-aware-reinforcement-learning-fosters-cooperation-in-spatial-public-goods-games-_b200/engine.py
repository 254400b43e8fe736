"""Thin object wrapper over the C ABI (``include/spgg.h``): one ``Engine`` = one
``spgg_t`` handle = ``n_replicas`` lattices resident on one GPU.

Argument names follow the reference ctor (``src/model/spgg.py:50-56``).
"""
from __future__ import annotations

import ctypes as C
from typing import Iterable, Sequence

import numpy as np

from . import _lib as L_

_ALGOS = {"qlearning": L_.ALGO_QLEARNING, "q-learning": L_.ALGO_QLEARNING,
          "sarsa": L_.ALGO_SARSA,
          "expected_sarsa": L_.ALGO_EXPECTED_SARSA, "expected-sarsa": L_.ALGO_EXPECTED_SARSA,
          "double_qlearning": L_.ALGO_DOUBLE_QLEARNING, "double-q-learning": L_.ALGO_DOUBLE_QLEARNING}


def params_struct(p: dict, seed: int = 0, precision: str = "fp32", rows=None, row0: int = 0,
                  r_storage: str = "auto") -> L_.Params:
    """Reference keyword arguments -> ``spgg_params_t``.  Defaults are the
    reference ctor defaults (spgg.py:50-56)."""
    state = p.get("state_representation", "reputation")
    if state not in ("reputation", "action"):
        # same message as spgg.py:309-310
        raise ValueError(f"Unknown state_representation: {state}. "
                         f"Must be 'reputation' or 'action'")
    algo = str(p.get("algorithm", "qlearning")).lower()
    if algo not in _ALGOS:
        # same message as algorithms.py:382-383
        raise ValueError(f"Unknown algorithm: {algo}. "
                         f"Supported: 'qlearning', 'sarsa', 'expected_sarsa', 'double_qlearning'")
    if precision not in ("fp32", "fp64"):
        raise ValueError(f"precision must be 'fp32' or 'fp64', got {precision!r}")
    Lsz = int(p.get("L", 50))
    return L_.Params(
        L=Lsz, rows=int(Lsz if rows is None else rows), row0=int(row0),
        M=2 if p.get("use_second_order", True) else 1,
        state_mode=L_.STATE_ACTION if state == "action" else L_.STATE_REPUTATION,
        precision=L_.PREC_FP64 if precision == "fp64" else L_.PREC_FP32,
        algorithm=_ALGOS[algo],
        r_storage={"auto": L_.RSTORE_AUTO, "int8": L_.RSTORE_INT8, "fp32": L_.RSTORE_FP32}[r_storage],
        r=float(p.get("r", 2)), c=float(p.get("c", 1)), cost=float(p.get("cost", 0.5)),
        alpha=float(p.get("alpha", 0.1)), gamma=float(p.get("gamma", 0.9)),
        epsilon=float(p.get("epsilon", 0.5)), epsilon_decay=float(p.get("epsilon_decay", 0.995)),
        epsilon_min=float(p.get("epsilon_min", 0.01)),
        kappa=float(p.get("influence_factor", 1.0)),
        lambda_eps=float(p.get("lambda_epsilon", 0.01)),
        rep_gain_C=float(p.get("rep_gain_C", 0.5)), delta_R_D=float(p.get("delta_R_D", 1)),
        R_min=float(p.get("R_min", -10)), R_max=float(p.get("R_max", 10)),
        wP=float(p.get("reward_weight_payoff", 1.0)), seed=int(seed) & (2 ** 64 - 1))


def cluster_which(of) -> int:
    """``of`` of the cluster methods -> the ``which`` of the C ABI (0 cooperators, 1 defectors)."""
    which = {"C": 0, "D": 1, 0: 0, 1: 1}.get(of if isinstance(of, (str, int)) and not isinstance(of, bool) else None)
    if which is None:
        raise ValueError(f"of must be 'C' or 'D' (or 0 / 1), got {of!r}")
    return which


def pair_correlation(counts, n_sites: int) -> np.ndarray:
    """Two-point correlation of the strategies from ``pair_counts`` (shape (2, max_d+1, 2)) of a lattice of
    ``n_sites`` sites: C(ax, d) = (n_CC/N - f^2) / (f - f^2) with f = n_C/N, float64 of shape (2, max_d+1);
    C(ax, 0) = 1, and NaN everywhere when f is 0 or 1 (no fluctuation to correlate).  The counts themselves
    carry the other bond statistics: ``counts[:, 1, 1] / N`` is the interface density along each axis (the
    fraction of nearest-neighbour bonds joining a cooperator and a defector)."""
    c = np.asarray(counts, dtype=np.float64)
    if c.ndim != 3 or c.shape[0] != 2 or c.shape[2] != 2 or c.shape[1] < 1:
        raise ValueError(f"counts must have shape (2, max_d+1, 2), got {c.shape}")
    N = float(n_sites)
    f = c[0, 0, 0] / N
    if f <= 0.0 or f >= 1.0:
        return np.full(c.shape[:2], np.nan)
    return (c[:, :, 0] / N - f * f) / (f - f * f)


_BLOCK_FIELDS = {"R": L_.BLOCK_R, "Q": L_.BLOCK_Q}


def block_flags(fields) -> int:
    """``fields`` of the block-field methods (a name or a sequence of "R" and "Q") -> the flags of the C ABI."""
    names = (fields,) if isinstance(fields, str) else tuple(fields)
    flags = 0
    for f in names:
        if not isinstance(f, str) or f not in _BLOCK_FIELDS:
            raise ValueError(f"fields must name 'R' and/or 'Q', got {fields!r}")
        flags |= _BLOCK_FIELDS[f]
    return flags


def block_rows(L: int, b: int, row0: int = 0, rows: int | None = None) -> tuple[int, int]:
    """(I0, nI): the block rows of side ``b`` that hold rows [row0, row0 + rows) of an L x L lattice."""
    rows = L if rows is None else rows
    I0 = row0 // b
    return I0, (row0 + rows - 1) // b - I0 + 1


def block_result(counts, sums, flags: int, q_shape) -> dict:
    """The flat arrays of ``spgg_block_fields`` (counts (nI, B, 2) int64, sums (nI, B, 2, m) float64) -> the dict
    of ``Engine.block_fields``."""
    out = {"n": counts[:, :, 0], "n_C": counts[:, :, 1]}
    ch = 0
    if flags & L_.BLOCK_R:
        out["R"] = sums[:, :, :, 0]
        ch = 1
    if flags & L_.BLOCK_Q:
        out["Q"] = sums[:, :, :, ch:].reshape(sums.shape[:3] + tuple(q_shape))
    return out


def block_means(fields: dict) -> dict:
    """Means per block from ``block_fields``: ``coop`` = n_C / n, and for each of "R" and "Q" that is present
    the mean over all sites (``R``), over the cooperators (``R_C``) and over the defectors (``R_D``) of the
    block, shapes (B, B) for R and (B, B) + the Q shape of ``get_state`` for Q.  NaN where a class is empty."""
    n = np.asarray(fields["n"], np.float64)
    nC = np.asarray(fields["n_C"], np.float64)
    nD = n - nC
    out = {"coop": nC / n}
    with np.errstate(invalid="ignore", divide="ignore"):
        for key in ("R", "Q"):
            if key not in fields:
                continue
            s = np.asarray(fields[key], np.float64)
            tail = (1,) * (s.ndim - 3)
            sA, sC = s[:, :, 0], s[:, :, 1]
            for suffix, tot, cnt in (("", sA, n), ("_C", sC, nC), ("_D", sA - sC, nD)):
                c = cnt.reshape(cnt.shape + tail)
                out[key + suffix] = np.where(c > 0, tot / np.where(c > 0, c, 1.0), np.nan)
    return out


class Engine:
    """``n`` independent lattices on one device.  ``param_list`` is one dict (or a
    sequence of dicts, one per replica) with the reference ctor's argument names."""

    def __init__(self, param_list, seeds: Sequence[int] | int = 0, precision: str = "fp32",
                 device: int = 0, rows=None, row0: int = 0, r_storage: str = "auto"):
        if isinstance(param_list, dict):
            param_list = [param_list]
        param_list = list(param_list)
        n = len(param_list)
        if isinstance(seeds, int):
            seeds = [seeds + i for i in range(n)]
        self.lib = L_.load()
        arr = (L_.Params * n)(*[params_struct(p, s, precision, rows, row0, r_storage)
                                for p, s in zip(param_list, seeds)])
        self.n_replicas = n
        self.L = int(arr[0].L)
        self.rows = int(arr[0].rows)
        self.row0 = int(arr[0].row0)
        self.precision = precision
        # Q values per site: 4, or the two tables of Double Q-learning ([site][table][s][a])
        self.nq = 8 if int(arr[0].algorithm) == L_.ALGO_DOUBLE_QLEARNING else 4
        self._h = C.c_void_p()
        L_.check(self.lib.spgg_create(arr, n, int(device), C.byref(self._h)))
        self.device = int(device)
        self._last_n = 0

    # -- lifetime
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.spgg_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- state
    def set_state(self, S, R, Q, replica: int = 0):
        n = self.rows * self.L
        S8 = np.ascontiguousarray(np.asarray(S).reshape(-1) != 0, dtype=np.uint8)
        Rd = np.ascontiguousarray(np.asarray(R, dtype=np.float64).reshape(-1))
        Qd = np.ascontiguousarray(np.asarray(Q, dtype=np.float64).reshape(-1))
        if S8.size != n or Rd.size != n or Qd.size != self.nq * n:
            raise ValueError(f"state arrays must describe {self.rows}x{self.L} sites "
                             f"({self.nq} Q values per site)")
        L_.check(self.lib.spgg_set_state(self._h, replica, S8.ctypes.data, Rd.ctypes.data,
                                         Qd.ctypes.data))

    def init_random(self, seed: int, replica: int = 0):
        L_.check(self.lib.spgg_init_random(self._h, replica, int(seed) & (2 ** 64 - 1)))

    def get_state(self, replica: int = 0, want_q: bool = True):
        n = self.rows * self.L
        S = np.empty(n, np.uint8)
        R = np.empty(n, np.float64)
        Q = np.empty(self.nq * n, np.float64) if want_q else None
        L_.check(self.lib.spgg_get_state(self._h, replica, S.ctypes.data, R.ctypes.data,
                                         Q.ctypes.data if want_q else None))
        S = S.reshape(self.rows, self.L)
        R = R.reshape(self.rows, self.L)
        if want_q:
            Q = Q.reshape((self.rows, self.L, 2, 2) if self.nq == 4 else (self.rows, self.L, 2, 2, 2))
        return S, R, Q

    # -- checkpoint / resume (include/spgg.h: spgg_set_progress)
    def set_progress(self, iteration: int, epsilons):
        """Continue a run: the states just uploaded are those after ``iteration`` completed
        iterations with exploration rates ``epsilons`` (one per replica)."""
        eps = np.ascontiguousarray(np.atleast_1d(np.asarray(epsilons, dtype=np.float64)))
        if eps.size != self.n_replicas:
            raise ValueError(f"need one epsilon per replica ({self.n_replicas}), got {eps.size}")
        L_.check(self.lib.spgg_set_progress(self._h, int(iteration), eps.ctypes.data))

    def checkpoint(self) -> dict:
        """Everything a later process needs to continue this run bit for bit: S, R, Q of every
        replica, the iteration counter and the exploration rates."""
        st = [self.status(r) for r in range(self.n_replicas)]
        states = [self.get_state(r) for r in range(self.n_replicas)]
        return {"iteration": int(max(s.iteration for s in st)), "epsilon": [float(s.epsilon) for s in st],
                "S": [s[0] for s in states], "R": [s[1] for s in states], "Q": [s[2] for s in states]}

    def restore(self, ck: dict):
        """Upload a ``checkpoint()`` into this (fresh) handle and continue from its iteration."""
        for r in range(self.n_replicas):
            self.set_state(ck["S"][r], ck["R"][r], ck["Q"][r], replica=r)
        self.set_progress(ck["iteration"], ck["epsilon"])

    def digest(self, replica: int = 0) -> tuple[int, int, int]:
        """Position-keyed 64-bit digests (S, R, Q) of the owned rows; strips of one lattice add up
        (mod 2^64) to the digest of the whole lattice (include/spgg.h: spgg_state_digest)."""
        out = (C.c_uint64 * 3)()
        L_.check(self.lib.spgg_state_digest(self._h, replica, out))
        return int(out[0]), int(out[1]), int(out[2])

    def get_q(self, replica: int = 0):
        """The Q table alone, as float64 in the reference's layout (the strategies and reputations stay)."""
        n = self.rows * self.L
        Q = np.empty(self.nq * n, np.float64)
        L_.check(self.lib.spgg_get_state(self._h, replica, None, None, Q.ctypes.data))
        return Q.reshape((self.rows, self.L, 2, 2) if self.nq == 4 else (self.rows, self.L, 2, 2, 2))

    def r_histogram(self, bins: int, lo: float, hi: float, replica: int = 0):
        """``np.histogram(R, bins=bins, range=(lo, hi))`` computed on the device: (counts int64, edges)."""
        edges = np.linspace(lo, hi, bins + 1, dtype=np.float64)
        counts = np.zeros(bins, np.int64)
        L_.check(self.lib.spgg_r_histogram(self._h, replica, int(bins), edges.ctypes.data, counts.ctypes.data))
        return counts, edges

    # -- clusters (include/spgg.h: spgg_clusters)
    def _clusters(self, replica, of, periodic) -> int:
        which = cluster_which(of)
        n = C.c_int64()
        L_.check(self.lib.spgg_clusters(self._h, int(replica), which, L_.CLUSTER_PERIODIC if periodic else 0,
                                        C.byref(n)))
        return int(n.value)

    def cluster_sizes(self, replica: int = 0, of="C", periodic: bool = False) -> np.ndarray:
        """Sizes (int64) of the 4-connected clusters of cooperators (``of="C"``) or defectors (``"D"``),
        computed on the device: ``np.bincount(label(S == of)[0].ravel())[1:]`` with scipy's labelling
        (spgg.py:631-633), in the order of each cluster's first site in raster order.  ``periodic=True``
        also joins clusters across the edges of the torus."""
        n = self._clusters(replica, of, periodic)
        sizes = np.empty(n, np.int64)
        L_.check(self.lib.spgg_cluster_sizes(self._h, sizes.ctypes.data, n))
        return sizes

    def cluster_labels(self, replica: int = 0, of="C", periodic: bool = False):
        """``scipy.ndimage.label(S == of)`` computed on the device: (labels int32 (rows, L), n); labels
        1..n numbered by each cluster's first site in raster order, 0 where the site is not selected."""
        n = self._clusters(replica, of, periodic)
        labels = np.empty((self.rows, self.L), np.int32)
        L_.check(self.lib.spgg_cluster_labels(self._h, labels.ctypes.data))
        return labels, n

    # -- strategy pair counts (include/spgg.h: spgg_pair_counts)
    def pair_counts(self, max_d: int, replica: int = 0) -> np.ndarray:
        """Exact strategy pair counts over the torus, computed on the device: int64 of shape (2, max_d+1, 2)
        with ``[ax, d, 0]`` the sites x that cooperate together with x + d along numpy axis ``ax`` and
        ``[ax, d, 1]`` those whose partner holds the other strategy (``[ax, 0]`` = (n_C, 0));
        1 <= max_d <= L/2.  ``pair_correlation`` turns them into C(d)."""
        out = np.zeros((2, max(int(max_d), 0) + 1, 2), np.int64)
        L_.check(self.lib.spgg_pair_counts(self._h, int(replica), int(max_d), out.ctypes.data))
        return out

    # -- block fields (include/spgg.h: spgg_block_fields)
    def block_fields(self, b: int, replica: int = 0, fields=("R", "Q")) -> dict:
        """Counts and sums over the b x b blocks of the lattice (B = ceil(L/b) per side, anchored at site
        (0, 0), the last block row and column ragged when b does not divide L), computed on the device:
        ``"n"`` and ``"n_C"`` int64 (B, B), the sites and the cooperators of each block; for each field asked
        for, ``"R"`` float64 (B, B, 2) and ``"Q"`` float64 (B, B, 2) + the Q shape of ``get_state``, the sums
        over all sites ([..., 0, ...]) and over the cooperators ([..., 1, ...]).  ``fields=()`` reads only the
        strategy bits.  Counts and int8-stored R are exact; fp32 / fp64 values are summed in fp64 in a fixed
        order.  On a strip handle the leading axis runs over the block rows holding its rows, with the strip's
        own contribution.  ``block_means`` turns the result into means."""
        flags = block_flags(fields)
        b, L = int(b), self.L
        counts, sums = np.zeros(2, np.int64), np.zeros(1)
        B = -(-L // b) if 1 <= b <= L else 0
        if B and B * B <= 1 << 24:   # else the library rejects b before writing
            I0, nI = block_rows(L, b, self.row0, self.rows)
            m = (1 if flags & L_.BLOCK_R else 0) + (self.nq if flags & L_.BLOCK_Q else 0)
            counts, sums = np.zeros((nI, B, 2), np.int64), np.zeros((nI, B, 2, m))
        L_.check(self.lib.spgg_block_fields(self._h, int(replica), b, flags, counts.ctypes.data,
                                            sums.ctypes.data if flags else None))
        return block_result(counts, sums, flags, (2, 2) if self.nq == 4 else (2, 2, 2))

    def set_replay(self, u, b):
        """``u`` (n,rows,L) float64 and ``b`` (n,rows,L) 0/1: the reference's draw
        arrays for the next n iterations (algorithms.py:105,108)."""
        u = np.ascontiguousarray(u, dtype=np.float64)
        b = np.ascontiguousarray(b, dtype=np.uint8)
        if u.ndim == 4:   # (n, pairs, rows, L): SARSA draws three pairs per iteration
            L_.check(self.lib.spgg_set_replay_pairs(self._h, u.shape[0], u.shape[1], u.ctypes.data,
                                                    b.ctypes.data))
            return
        n = u.shape[0] if u.ndim == 3 else 0
        L_.check(self.lib.spgg_set_replay(self._h, n, u.ctypes.data if n else None,
                                          b.ctypes.data if n else None))

    # -- stepping
    def step(self, n: int, stream: int | None = None):
        L_.check(self.lib.spgg_step(self._h, int(n), C.c_void_p(stream or 0)))
        self._last_n = int(n)

    def sync(self):
        L_.check(self.lib.spgg_sync(self._h))

    def stats(self, replica: int = 0, first: int = 0, n: int | None = None) -> np.ndarray:
        """Rows of the last ``step`` call (row 0 = starting state, row k = k-th iteration)."""
        if n is None:
            n = self._last_n + 1 - first
        out = np.empty((n, L_.NSTAT), np.float64)
        L_.check(self.lib.spgg_get_stats(self._h, replica, first, n, out.ctypes.data))
        return out

    def describe(self) -> str:
        """Which kernels serve this handle (resident cluster / cooperative grid, TMA fast path, general)."""
        buf = C.create_string_buffer(256)
        self.lib.spgg_describe(self._h, buf, 256)
        return buf.value.decode()

    def status(self, replica: int = 0) -> L_.Status:
        st = L_.Status()
        L_.check(self.lib.spgg_query(self._h, replica, C.byref(st)))
        return st
