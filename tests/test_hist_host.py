"""Value distributions (include/spgg.h: spgg_value_ranges / spgg_histograms, Engine.histograms,
StripEngine.histograms) without a GPU: the NumPy restatement the device tests compare with, checked against plain
np.histogram on masked arrays on values placed on the edges; NumPy's default range; the greedy policy with ties;
strip sums; class_histograms; and the argument checks."""
import ctypes as C

import numpy as np
import pytest

BINS = (1, 7, 20, 64, 1024)


def _channels(R, Q, flags):
    chans = []
    if flags & 1:
        chans.append(np.asarray(R, np.float64).reshape(-1))
    if flags & 2:
        q = np.asarray(Q, np.float64)
        q = q.reshape(q.shape[0] * q.shape[1], -1)
        chans += [q[:, z] for z in range(q.shape[1])]
    return chans


def _bins_of(x, e):
    """The uniform-bin rule of spgg_histograms (NumPy's): -1 outside [e[0], e[-1]], else the float index corrected
    by one against the edges, the last bin closed."""
    nb = len(e) - 1
    lo, hi = e[0], e[nb]
    keep = (x >= lo) & (x <= hi)
    idx = np.clip(((x - lo) * (nb / (hi - lo))).astype(np.int64), 0, nb - 1)
    idx = np.where(x < e[idx], idx - 1, idx)
    idx = np.where((x >= e[np.minimum(idx + 1, nb)]) & (idx != nb - 1), idx + 1, idx)
    return np.where(keep, idx, -1)


def numpy_policy(S, Q, algo):
    """policy[k, s]: the sites of class k (0 all, 1 cooperators) whose greedy action in state s is C."""
    Q = np.asarray(Q, np.float64)
    if algo == "double_qlearning":
        Q = (Q[..., 0, :, :] + Q[..., 1, :, :]) / 2
    greedy_c = np.argmax(Q, axis=-1) == 0                # (rows, L, 2)
    coop = np.asarray(S) == 0
    return np.stack([greedy_c.sum(axis=(0, 1)), greedy_c[coop].sum(axis=0)]).astype(np.int64)


def numpy_histograms(S, R, Q, edges, algo, flags=3):
    """Host restatement of spgg_histograms for one replica (S, R of shape (rows, L), Q as get_state returns it):
    edges (m, bins + 1) per channel -> counts int64 (m, 2, bins) [channel, class, bin] and policy int64 (2, 2)."""
    coop = (np.asarray(S) == 0).reshape(-1)
    edges = np.asarray(edges, np.float64)
    nb = edges.shape[1] - 1
    chans = _channels(R, Q, flags)
    counts = np.zeros((len(chans), 2, nb), np.int64)
    for ch, x in enumerate(chans):
        b = _bins_of(x, edges[ch])
        counts[ch, 0] = np.bincount(b[b >= 0], minlength=nb)
        counts[ch, 1] = np.bincount(b[(b >= 0) & coop], minlength=nb)
    return counts, numpy_policy(S, Q, algo)


def numpy_value_ranges(S, R, Q, flags=3):
    """Host restatement of spgg_value_ranges for one replica: (m, 2, 2) [channel, class, min / max]."""
    coop = (np.asarray(S) == 0).reshape(-1)
    out = []
    for x in _channels(R, Q, flags):
        row = []
        for sel in (x, x[coop]):
            row.append([sel.min(), sel.max()] if sel.size else [np.inf, -np.inf])
        out.append(row)
    return np.array(out, np.float64).reshape(-1, 2, 2)


def default_edges(S, R, Q, bins, flags=3):
    """NumPy's default edges of every channel: hist_edges over (min, max) of all sites."""
    from spgg_b200.engine import hist_edges
    return np.stack([hist_edges(x.min(), x.max(), bins) for x in _channels(R, Q, flags)])


def _plain(S, R, Q, edges, flags=3):
    """np.histogram itself on the masked arrays"""
    coop = (np.asarray(S) == 0).reshape(-1)
    out = []
    for ch, x in enumerate(_channels(R, Q, flags)):
        e = edges[ch]
        a, ea = np.histogram(x, bins=len(e) - 1, range=(e[0], e[-1]))
        c, _ = np.histogram(x[coop], bins=len(e) - 1, range=(e[0], e[-1]))
        assert np.array_equal(ea, e)
        out.append([a, c])
    return np.array(out, np.int64)


def _edge_state(rs, L, lo, hi, bins, nq=4):
    """A lattice whose values sit on every edge, on hi, just outside the range, on +-0.0 and in between."""
    e = np.linspace(lo, hi, bins + 1)
    pool = np.concatenate([e, np.nextafter(e, -np.inf), np.nextafter(e, np.inf), [lo - 1e-300, hi + 1e-300, 0.0,
                           -0.0, np.nextafter(lo, -np.inf), np.nextafter(hi, np.inf)], rs.uniform(lo, hi, 64)])
    S = rs.randint(0, 2, (L, L)).astype(np.uint8)
    R = rs.choice(pool, (L, L))
    Q = rs.choice(pool, (L, L) + ((2, 2) if nq == 4 else (2, 2, 2)))
    return S, R, Q, e


@pytest.mark.parametrize("bins", BINS)
@pytest.mark.parametrize("lo,hi", [(-10.0, 10.0), (-1.0, 0.0), (0.0, 1.0), (-0.3, 0.7), (-0.01, 0.0123), (1e-3, 1e5)])
def test_restatement_equals_np_histogram_on_the_edges(bins, lo, hi):
    rs = np.random.RandomState(bins * 7 + int(abs(lo) * 13))
    S, R, Q, e = _edge_state(rs, 24, lo, hi, bins)
    edges = np.stack([e] * 5)
    counts, _ = numpy_histograms(S, R, Q, edges, "qlearning")
    assert np.array_equal(counts, _plain(S, R, Q, edges))
    # every value in range is counted, in both classes
    for ch, x in enumerate(_channels(R, Q, 3)):
        assert counts[ch, 0].sum() == ((x >= lo) & (x <= hi)).sum()


@pytest.mark.parametrize("bins", BINS)
def test_default_ranges_and_equal_extremes(bins):
    from spgg_b200.engine import hist_edges
    rs = np.random.RandomState(bins)
    for v in (0.0, -0.0, 3.0, -2.5, 1e-300):
        x = np.full(50, v)
        assert np.array_equal(hist_edges(x.min(), x.max(), bins), np.histogram_bin_edges(x, bins))
        S = np.zeros((5, 10), np.uint8)
        R = x.reshape(5, 10)
        edges = default_edges(S, R, None, bins, flags=1)
        counts, _ = numpy_histograms(S, R, np.zeros((5, 10, 2, 2)), edges, "qlearning", flags=1)
        assert np.array_equal(counts[0, 0], np.histogram(x, bins)[0])
    S, R, Q, _ = _edge_state(rs, 16, -3.0, 5.0, bins)
    edges = default_edges(S, R, Q, bins)
    for ch, x in enumerate(_channels(R, Q, 3)):
        assert np.array_equal(edges[ch], np.histogram_bin_edges(x, bins))
    assert np.array_equal(numpy_histograms(S, R, Q, edges, "qlearning")[0], _plain(S, R, Q, edges))


def test_value_ranges_restatement():
    rs = np.random.RandomState(3)
    S, R, Q, _ = _edge_state(rs, 12, -1.0, 1.0, 7)
    mm = numpy_value_ranges(S, R, Q)
    coop = S.reshape(-1) == 0
    for ch, x in enumerate(_channels(R, Q, 3)):
        assert mm[ch, 0, 0] == x.min() and mm[ch, 0, 1] == x.max()
        assert mm[ch, 1, 0] == x[coop].min() and mm[ch, 1, 1] == x[coop].max()
    mm = numpy_value_ranges(np.ones_like(S), R, Q)   # no cooperators
    assert (mm[:, 1, 0] == np.inf).all() and (mm[:, 1, 1] == -np.inf).all()


@pytest.mark.parametrize("algo", ["qlearning", "double_qlearning"])
def test_policy_with_ties(algo):
    rs = np.random.RandomState(11)
    L = 32
    shape = (L, L, 2, 2) if algo == "qlearning" else (L, L, 2, 2, 2)
    vals = np.array([0.0, -0.0, 0.1, 0.2, 0.3, 1e-300, 5e-324, -5e-324, 1.0, np.nextafter(1.0, 2.0)])
    Q = rs.choice(vals, shape)
    # ties: both actions equal (or, for Double Q, equal means from different tables)
    Q[: L // 2, :, ..., 1] = Q[: L // 2, :, ..., 0]
    if algo == "double_qlearning":
        Q[L // 2:, :, 0, :, 0], Q[L // 2:, :, 1, :, 0] = 0.1, 0.2
        Q[L // 2:, :, 0, :, 1], Q[L // 2:, :, 1, :, 1] = 0.2, 0.1
    S = rs.randint(0, 2, (L, L)).astype(np.uint8)
    pol = numpy_policy(S, Q, algo)
    Qb = Q if algo == "qlearning" else (Q[..., 0, :, :] + Q[..., 1, :, :]) / 2
    for k, mask in enumerate((np.ones((L, L), bool), S == 0)):
        for s in range(2):
            assert pol[k, s] == (Qb[mask][:, s, 0] >= Qb[mask][:, s, 1]).sum()
            assert pol[k, s] == (np.argmax(Qb[mask][:, s, :], axis=-1) == 0).sum()


@pytest.mark.parametrize("world", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("L", [40, 100])
def test_strip_results_add_up(world, L):
    from spgg_b200.engine import hist_edges
    from spgg_b200.strips import strip_rows
    rs = np.random.RandomState(world * 100 + L)
    S, R, Q, _ = _edge_state(rs, L, -2.0, 3.0, 20, nq=8)
    bins = 20
    parts = []
    for k in range(world):
        r0, n = strip_rows(L, world, k)
        parts.append((S[r0:r0 + n], R[r0:r0 + n], Q[r0:r0 + n]))
    # min / max of the strips' ranges = the lattice's; the same edges on every rank
    mms = np.stack([numpy_value_ranges(*p) for p in parts])
    mm = numpy_value_ranges(S, R, Q)
    assert np.array_equal(mms[..., 0].min(0), mm[..., 0]) and np.array_equal(mms[..., 1].max(0), mm[..., 1])
    edges = np.stack([hist_edges(a, b, bins) for a, b in mm[:, 0]])
    tot_c, tot_p = 0, 0
    for p in parts:
        c, pol = numpy_histograms(*p, edges, "double_qlearning")
        tot_c, tot_p = tot_c + c, tot_p + pol
    c, pol = numpy_histograms(S, R, Q, edges, "double_qlearning")
    assert np.array_equal(tot_c, c) and np.array_equal(tot_p, pol)
    assert np.array_equal(c, _plain(S, R, Q, edges))


def test_class_histograms():
    from spgg_b200.engine import class_histograms, hist_result
    rs = np.random.RandomState(5)
    S, R, Q, _ = _edge_state(rs, 20, -1.0, 1.0, 9)
    edges = default_edges(S, R, Q, 9)
    counts, pol = numpy_histograms(S, R, Q, edges, "qlearning")
    h = hist_result(counts[None], pol[None], edges[None], ["R"] + ["Q"] * 4, (2, 2), False, 0)
    assert h["R"].shape == (2, 9) and h["Q"].shape == (2, 2, 2, 9) and h["Q_edges"].shape == (2, 2, 10)
    ch = class_histograms(h)
    coop = S.reshape(-1) == 0
    x = R.reshape(-1)
    for k, sel in enumerate((x, x[coop], x[~coop])):
        want, _ = np.histogram(sel, bins=edges[0])
        dens, _ = np.histogram(sel, bins=edges[0], density=True)
        assert np.array_equal(ch["R"][k], want)
        assert np.allclose(ch["R_density"][k], dens, rtol=1e-12, atol=0)
    q = Q.reshape(-1, 2, 2)
    want, _ = np.histogram(q[~coop][:, 1, 0], bins=edges[1 + 2])
    assert np.array_equal(ch["Q"][2, 1, 0], want)
    assert np.array_equal(ch["policy"][2], pol[0] - pol[1])
    # a batch: the class axis follows the replica axis
    hb = hist_result(np.stack([counts] * 2), np.stack([pol] * 2), np.stack([edges] * 2), ["R"] + ["Q"] * 4, (2, 2),
                     True, range(3, 5))
    cb = class_histograms(hb)
    assert cb["R"].shape == (2, 3, 9) and np.array_equal(cb["R"][1], ch["R"])
    assert np.array_equal(cb["Q_density"][0], ch["Q_density"], equal_nan=True)


def test_null_handle_is_rejected_without_a_gpu():
    import spgg_b200
    from spgg_b200 import _lib
    lib = spgg_b200.load()
    e = np.linspace(0.0, 1.0, 5)
    cnt = np.full(64, -7, np.int64)
    mm = np.full(16, -7.0)
    for flags in (0, 1, 3):
        assert lib.spgg_histograms(None, 0, 1, flags, 4, e.ctypes.data, cnt.ctypes.data, cnt.ctypes.data) == _lib.E_INVALID
        assert lib.spgg_value_ranges(None, 0, 1, flags, mm.ctypes.data) == _lib.E_INVALID
    assert (cnt == -7).all() and (mm == -7.0).all()


def _null_engine(n_replicas=1, nq=4):
    import spgg_b200
    eng = spgg_b200.Engine.__new__(spgg_b200.Engine)
    eng.lib, eng._h, eng.L, eng.rows, eng.row0, eng.nq = spgg_b200.load(), C.c_void_p(), 16, 16, 0, nq
    eng.n_replicas = n_replicas
    return eng


def test_engine_histograms_checks_its_arguments():
    eng = _null_engine(n_replicas=3)
    for bins in (0, -1, 1025):
        with pytest.raises(ValueError, match="bins"):
            eng.histograms(bins)
    for bad in (("R", "X"), "RQ", ("q",), (1,)):
        with pytest.raises(ValueError, match="fields"):
            eng.histograms(4, fields=bad)
        with pytest.raises(ValueError, match="fields"):
            eng.value_ranges(fields=bad)
    for rep in (3, -1, range(2, 4), range(0, 3, 2), range(1, 1), True, 1.0, "0"):
        with pytest.raises(ValueError, match="replica"):
            eng.histograms(4, replica=rep)
        with pytest.raises(ValueError, match="replica"):
            eng.value_ranges(replica=rep)
    with pytest.raises(ValueError, match="ranges"):
        eng.histograms(4, ranges={"S": (0, 1)})
    for lo, hi in ((1.0, 0.0), (0.0, np.inf), (np.nan, 1.0)):
        with pytest.raises(ValueError, match="range"):
            eng.histograms(4, fields=("R",), ranges={"R": (lo, hi)})
    # valid arguments reach the library, which rejects the null handle
    with pytest.raises(ValueError, match="null"):
        eng.histograms(4, replica=range(0, 3), ranges={"R": (0, 1), "Q": (-1, 1)})
    with pytest.raises(ValueError, match="null"):
        eng.value_ranges(replica=range(1, 3))
    with pytest.raises(ValueError, match="null"):
        eng.histograms(4, fields=())   # policy only


def test_strip_engine_histograms_checks_its_arguments_first():
    import torch
    from spgg_b200 import strips
    se = strips.StripEngine.__new__(strips.StripEngine)
    se.torch, se.L, se.world, se.rank = torch, 64, 1, 0
    with pytest.raises(ValueError, match="fields"):
        se.histograms(4, fields=("S",))
    with pytest.raises(ValueError, match="bins"):
        se.histograms(2000)
