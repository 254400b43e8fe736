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


HIST_MAX_BINS = 1024


def hist_edges(lo, hi, bins: int) -> np.ndarray:
    """The edges of ``np.histogram(x, bins=bins, range=(lo, hi))``: (lo, hi) checked as NumPy checks a range,
    widened by 0.5 each way when lo == hi, then ``np.linspace``."""
    lo, hi = float(lo), float(hi)
    if not (np.isfinite(lo) and np.isfinite(hi)):
        raise ValueError(f"histogram range ({lo}, {hi}) is not finite")
    if lo > hi:
        raise ValueError(f"histogram range ({lo}, {hi}): max must be larger than min")
    if lo == hi:
        lo, hi = lo - 0.5, hi + 0.5
    return np.linspace(lo, hi, bins + 1, endpoint=True, dtype=np.float64)


def hist_replicas(replica, n_replicas: int) -> tuple[int, int]:
    """``replica`` of the histogram methods (an int, or a ``range`` of consecutive replicas) -> (rep0, n)."""
    if isinstance(replica, range):
        if replica.step != 1 or len(replica) == 0:
            raise ValueError(f"replica must be a non-empty range of consecutive replicas, got {replica!r}")
        rep0, n = replica.start, len(replica)
    elif isinstance(replica, (int, np.integer)) and not isinstance(replica, bool):
        rep0, n = int(replica), 1
    else:
        raise ValueError(f"replica must be an int or a range, got {replica!r}")
    if rep0 < 0 or rep0 + n > n_replicas:
        raise ValueError(f"replicas {rep0} .. {rep0 + n - 1} outside [0, {n_replicas})")
    return rep0, n


def hist_channels(flags: int, nq: int) -> list[str]:
    """The channels of ``spgg_histograms`` for ``flags``, by field: "R" once, then "Q" nq times."""
    return (["R"] if flags & L_.HIST_R else []) + (["Q"] * nq if flags & L_.HIST_Q else [])


def hist_edge_rows(bins: int, chans: Sequence[str], minmax, ranges) -> np.ndarray:
    """Edges (n, m, bins + 1) of the channels ``chans``: from ``ranges[field]`` where given, else NumPy's default
    range per replica and channel from ``minmax`` (n, m, 2), the (min, max) over all sites of
    ``spgg_value_ranges`` (not read for a field with a range)."""
    ranges = {} if ranges is None else ranges
    n = minmax.shape[0]
    edges = np.empty((n, len(chans), bins + 1))
    for ch, f in enumerate(chans):
        for r in range(n):
            lo, hi = ranges[f] if f in ranges else minmax[r, ch]
            edges[r, ch] = hist_edges(lo, hi, bins)
    return edges


def hist_result(counts, policy, edges, chans, q_shape, batched: bool, replica) -> dict:
    """The flat arrays of ``spgg_histograms`` (counts (n, m, 2, bins), policy (n, 2, 2) or None, edges
    (n, m, bins + 1)) -> the dict of ``Engine.histograms``."""
    n, bins = counts.shape[0], counts.shape[-1]
    out = {"replica": replica}
    ch = 0
    if "R" in chans:
        out["R"], out["R_edges"] = counts[:, 0], edges[:, 0]
        ch = 1
    if "Q" in chans:
        out["Q"] = np.moveaxis(counts[:, ch:], 2, 1).reshape((n, 2) + tuple(q_shape) + (bins,))
        out["Q_edges"] = edges[:, ch:].reshape((n,) + tuple(q_shape) + (bins + 1,))
    if policy is not None:
        out["policy"] = policy
    if not batched:
        out = {k: (v[0] if isinstance(v, np.ndarray) else v) for k, v in out.items()}
    return out


def class_histograms(h: dict) -> dict:
    """The result of ``histograms`` with the defectors added: for "R", "Q" and "policy" where present the class
    axis holds [all, cooperators, defectors] (defectors = all - cooperators), and "R_density" / "Q_density" are
    ``np.histogram(..., density=True)`` of each class (NaN where a class has no count in range)."""
    batched = isinstance(h["replica"], range)
    ax = 1 if batched else 0
    out = dict(h)
    for key in ("R", "Q", "policy"):
        if key not in h:
            continue
        c = np.asarray(h[key])
        a, cc = np.take(c, 0, axis=ax), np.take(c, 1, axis=ax)
        out[key] = np.stack([a, cc, a - cc], axis=ax)
        if key == "policy":
            continue
        widths = np.diff(h[key + "_edges"], axis=-1)
        widths = np.expand_dims(widths, ax)
        tot = out[key].sum(axis=-1, keepdims=True)
        with np.errstate(invalid="ignore", divide="ignore"):
            out[key + "_density"] = np.where(tot > 0, out[key] / np.where(tot > 0, tot, 1) / widths, np.nan)
    return out


def snapshot_slot(slot) -> int:
    """``slot`` of the snapshot methods -> the slot index of the C ABI, in [0, ``SPGG_MAX_SNAPSHOTS``)."""
    if not isinstance(slot, (int, np.integer)) or isinstance(slot, bool) or not 0 <= slot < L_.MAX_SNAPSHOTS:
        raise ValueError(f"slot must be an int in [0, {L_.MAX_SNAPSHOTS}), got {slot!r}")
    return int(slot)


def overlap_result(counts, changed, diffs, flags: int, q_shape, batched: bool, t0: int, t: int) -> dict:
    """The flat arrays of ``spgg_overlap`` (counts (n, 2, 2) int64, changed (n, m) int64, diffs (n, m, 3)) -> the
    dict of ``Engine.overlap``."""
    n = counts.shape[0]
    out = {"S": counts}
    ch = 0
    if flags & L_.SNAP_R:
        out["R_changed"], out["R_diff"] = changed[:, 0], diffs[:, 0]
        ch = 1
    if flags & L_.SNAP_Q:
        out["Q_changed"] = changed[:, ch:].reshape((n,) + tuple(q_shape))
        out["Q_diff"] = diffs[:, ch:].reshape((n,) + tuple(q_shape) + (3,))
    if not batched:
        out = {k: v[0] for k, v in out.items()}
    out["t0"], out["t"] = int(t0), int(t)
    return out


def overlap_measures(o: dict, n_sites: int) -> dict:
    """Summary measures of an ``overlap`` result over a lattice of ``n_sites`` sites (a leading replica axis
    carries through): ``hamming`` = (n_CD + n_DC) / N, the fraction of sites whose strategy differs;
    ``autocorrelation`` = (n_CC/N - f0 f) / sqrt(f0 (1 - f0) f (1 - f)) with f0, f the cooperator fractions then
    and now (NaN when either state is uniform); ``persistence_C`` = n_CC / n_C(t0) and ``persistence_D`` =
    n_DD / n_D(t0) (NaN when that class was empty at t0); and for each field present ``R_rms`` / ``Q_rms`` =
    sqrt(sum d^2 / N) and ``R_mean_abs`` / ``Q_mean_abs`` = sum |d| / N (per Q entry)."""
    S = np.asarray(o["S"], np.float64)
    if S.shape[-2:] != (2, 2):
        raise ValueError(f"o['S'] must end in (2, 2), got {S.shape}")
    N = float(n_sites)
    nCC, nCD, nDC, nDD = S[..., 0, 0], S[..., 0, 1], S[..., 1, 0], S[..., 1, 1]
    f0, f = (nCC + nCD) / N, (nCC + nDC) / N
    nC0, nD0 = nCC + nCD, nDC + nDD
    den = np.sqrt(f0 * (1.0 - f0) * f * (1.0 - f))
    with np.errstate(invalid="ignore", divide="ignore"):
        out = {"hamming": (nCD + nDC) / N,
               "autocorrelation": np.where(den > 0, (nCC / N - f0 * f) / np.where(den > 0, den, 1.0), np.nan),
               "persistence_C": np.where(nC0 > 0, nCC / np.where(nC0 > 0, nC0, 1.0), np.nan),
               "persistence_D": np.where(nD0 > 0, nDD / np.where(nD0 > 0, nD0, 1.0), np.nan)}
    for key in ("R", "Q"):
        if key + "_diff" in o:
            d = np.asarray(o[key + "_diff"], np.float64)
            out[key + "_rms"] = np.sqrt(d[..., 2] / N)
            out[key + "_mean_abs"] = d[..., 1] / N
    return {k: np.asarray(v)[()] for k, v in out.items()}


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

    # -- value distributions (include/spgg.h: spgg_value_ranges / spgg_histograms)
    def _value_ranges(self, rep0: int, n: int, flags: int) -> np.ndarray:
        m = len(hist_channels(flags, self.nq))
        mm = np.zeros((n, m, 2, 2))
        L_.check(self.lib.spgg_value_ranges(self._h, rep0, n, flags, mm.ctypes.data))
        return mm

    def value_ranges(self, replica=0, fields=("R", "Q")) -> dict:
        """Exact (min, max) of every field over all sites and over the cooperators, computed on the device:
        ``"R"`` float64 (2, 2) [class, min/max] and ``"Q"`` float64 (2,) + the Q shape of ``get_state`` + (2,),
        class 0 all sites and 1 the cooperators (+inf / -inf for an empty class).  ``replica`` is an int or a
        ``range`` of consecutive replicas, which adds a leading replica axis."""
        flags = block_flags(fields)   # SPGG_HIST_R / SPGG_HIST_Q are the bits of SPGG_BLOCK_R / SPGG_BLOCK_Q
        rep0, n = hist_replicas(replica, self.n_replicas)
        mm = self._value_ranges(rep0, n, flags)
        out, ch = {}, 0
        if flags & L_.HIST_R:
            out["R"] = mm[:, 0]
            ch = 1
        if flags & L_.HIST_Q:
            qs = (2, 2) if self.nq == 4 else (2, 2, 2)
            out["Q"] = np.moveaxis(mm[:, ch:], 2, 1).reshape((n, 2) + qs + (2,))
        return out if isinstance(replica, range) else {k: v[0] for k, v in out.items()}

    def _histograms(self, rep0: int, n: int, flags: int, bins: int, edges, policy: bool):
        """``spgg_histograms`` of replicas rep0 .. rep0+n-1 with edges (n, m, bins + 1) -> (counts (n, m, 2,
        bins) int64, policy (n, 2, 2) int64 or None)."""
        m = len(hist_channels(flags, self.nq))
        edges = np.ascontiguousarray(edges, np.float64)
        counts = np.zeros((n, m, 2, bins), np.int64)
        pol = np.zeros((n, 2, 2), np.int64) if policy else None
        L_.check(self.lib.spgg_histograms(self._h, rep0, n, flags, bins, edges.ctypes.data if m else None,
                                          counts.ctypes.data if m else None,
                                          pol.ctypes.data if policy else None))
        return counts, pol

    def histograms(self, bins: int, replica=0, fields=("R", "Q"), ranges=None, policy: bool = True) -> dict:
        """``np.histogram(x, bins=bins, range=...)`` of R and of every Q entry, over all sites and over the
        cooperators, and the greedy-policy counts, computed on the device with exact integer counts.
        ``replica``: an int, or a ``range`` of consecutive replicas (a leading replica axis on every array).
        ``ranges``: {"R": (lo, hi), "Q": (lo, hi)}; a field without one gets NumPy's default range, (min, max)
        over all sites of its replica and channel (``value_ranges``).  Returns ``"R"`` int64 (2, bins)
        [all, C] and ``"R_edges"`` (bins + 1,); ``"Q"`` int64 (2,) + the Q shape of ``get_state`` + (bins,)
        and ``"Q_edges"`` (Q shape + (bins + 1,)); with ``policy``, ``"policy"`` int64 (2, 2) [class, state],
        the sites whose greedy action in state s is C (argmax of Q, or of (QA + QB) / 2 for Double
        Q-learning); and ``"replica"``.  ``class_histograms`` adds the defectors and the densities."""
        bins = int(bins)
        if not 1 <= bins <= HIST_MAX_BINS:
            raise ValueError(f"bins must be in [1, {HIST_MAX_BINS}], got {bins}")
        flags = block_flags(fields)
        rep0, n = hist_replicas(replica, self.n_replicas)
        chans = hist_channels(flags, self.nq)
        ranges = {} if ranges is None else dict(ranges)
        for f in ranges:
            if f not in ("R", "Q"):
                raise ValueError(f"ranges may name 'R' and 'Q', got {f!r}")
        need = any(f not in ranges for f in chans)
        mm = self._value_ranges(rep0, n, flags)[:, :, :1] if need else np.zeros((n, len(chans), 1, 2))
        edges = hist_edge_rows(bins, chans, mm[:, :, 0], ranges)
        counts, pol = self._histograms(rep0, n, flags, bins, edges, policy)
        return hist_result(counts, pol, edges, chans, (2, 2) if self.nq == 4 else (2, 2, 2),
                           isinstance(replica, range), replica)

    # -- state overlaps (include/spgg.h: spgg_snapshot / spgg_overlap)
    def snapshot(self, slot: int = 0, replica=0, fields=("R", "Q")) -> int:
        """Keep a copy of the current state of ``replica`` (an int, or a ``range`` of consecutive replicas) in
        ``slot`` on the device: the strategies always, R and Q as ``fields`` asks.  Replaces what the slot held;
        the copy survives stepping and state uploads until ``drop_snapshot`` or ``close``.  Returns the
        iteration counter stored with it."""
        flags = block_flags(fields)   # SPGG_SNAP_R / SPGG_SNAP_Q are the bits of SPGG_BLOCK_R / SPGG_BLOCK_Q
        slot = snapshot_slot(slot)
        rep0, n = hist_replicas(replica, self.n_replicas)
        L_.check(self.lib.spgg_snapshot(self._h, slot, rep0, n, flags))
        return self.snapshot_info(slot)["iteration"]

    def snapshot_info(self, slot: int = 0) -> dict:
        """``{"iteration", "replica", "fields"}`` of the snapshot in ``slot`` (``replica`` an int, or a range
        for several replicas)."""
        slot = snapshot_slot(slot)
        it, rep0, n, flags = C.c_int64(), C.c_int(), C.c_int(), C.c_int()
        L_.check(self.lib.spgg_snapshot_info(self._h, slot, C.byref(it), C.byref(rep0), C.byref(n), C.byref(flags)))
        rep = rep0.value if n.value == 1 else range(rep0.value, rep0.value + n.value)
        fields = tuple(f for f, bit in (("R", L_.SNAP_R), ("Q", L_.SNAP_Q)) if flags.value & bit)
        return {"iteration": int(it.value), "replica": rep, "fields": fields}

    def drop_snapshot(self, slot: int = 0):
        """Free the snapshot in ``slot`` (nothing happens if it is empty)."""
        L_.check(self.lib.spgg_snapshot_free(self._h, snapshot_slot(slot)))

    def _overlap(self, slot: int, rep0: int, n: int, flags: int):
        """``spgg_overlap`` -> (counts (n, 2, 2) int64, changed (n, m) int64, diffs (n, m, 3) float64)."""
        m = len(hist_channels(flags, self.nq))
        counts, changed, diffs = np.zeros((n, 2, 2), np.int64), np.zeros((n, m), np.int64), np.zeros((n, m, 3))
        L_.check(self.lib.spgg_overlap(self._h, slot, rep0, n, flags, counts.ctypes.data,
                                       changed.ctypes.data if m else None, diffs.ctypes.data if m else None))
        return counts, changed, diffs

    def overlap(self, slot: int = 0, replica=0, fields=("R", "Q")) -> dict:
        """What changed between the snapshot in ``slot`` and the current state, computed on the device.  Replica
        ``replica`` + i is compared with replica i of the snapshot, so a slot taken of replica a compared at
        replica b measures how far two replicas are apart.  Returns ``"S"`` int64 (2, 2) [then, now] (0 = C,
        1 = D); for R ``"R_changed"`` (the number of sites whose value differs) and ``"R_diff"`` (3,) [max |d|,
        sum |d|, sum d^2], d = now - then; for Q ``"Q_changed"`` and ``"Q_diff"`` with the Q shape of
        ``get_state`` (+ (3,)); ``"t0"`` the snapshot's iteration and ``"t"`` the current one.  Counts and maxima
        are exact; the sums are fp64 in an order fixed by the lattice shape.  A ``range`` of replicas adds a
        leading replica axis.  ``overlap_measures`` turns the result into Hamming distance, autocorrelation,
        persistence and RMS change."""
        flags = block_flags(fields)
        slot = snapshot_slot(slot)
        rep0, n = hist_replicas(replica, self.n_replicas)
        counts, changed, diffs = self._overlap(slot, rep0, n, flags)
        t0 = self.snapshot_info(slot)["iteration"]
        return overlap_result(counts, changed, diffs, flags, (2, 2) if self.nq == 4 else (2, 2, 2),
                              isinstance(replica, range), t0, self.status(rep0).iteration)

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
