"""State overlaps (include/spgg.h: spgg_snapshot / spgg_overlap, Engine.overlap, StripEngine.overlap) without a GPU:
the NumPy restatement the device tests compare with, checked on hand-made pairs of states (identical, all flipped,
+-0.0, int8-quantum values, Double-Q shapes); overlap_measures; the strip assembly; and the argument checks."""
import ctypes as C

import numpy as np
import pytest

U = 2.0 ** -53


def numpy_overlap(then, now, fields=("R", "Q"), nq=4):
    """What spgg_overlap computes, from two (S, R, Q) triples as get_state returns them: counts int64 (2, 2)
    [then, now] (0 = C, 1 = D), and per channel (R if asked, then the nq Q entries) changed int64 (m,) =
    count_nonzero(now != then) and diffs float64 (m, 3) = [max |d|, sum |d|, sum d^2], d = now - then in fp64
    (the sums by np.sum)."""
    S0, R0, Q0 = then
    S1, R1, Q1 = now
    S0, S1 = np.asarray(S0).reshape(-1), np.asarray(S1).reshape(-1)
    counts = np.array([[np.count_nonzero((S0 == a) & (S1 == b)) for b in (0, 1)] for a in (0, 1)], np.int64)
    chans = []
    if "R" in fields:
        chans.append((np.asarray(R1, np.float64).reshape(-1), np.asarray(R0, np.float64).reshape(-1)))
    if "Q" in fields:
        qn = np.asarray(Q1, np.float64).reshape(-1, nq)
        qt = np.asarray(Q0, np.float64).reshape(-1, nq)
        chans += [(qn[:, z], qt[:, z]) for z in range(nq)]
    changed = np.array([np.count_nonzero(a != b) for a, b in chans], np.int64)
    diffs = np.zeros((len(chans), 3))
    for ch, (a, b) in enumerate(chans):
        d = a - b
        ad = np.abs(d)
        diffs[ch] = ad.max(), ad.sum(), (d * d).sum()
    return counts, changed, diffs


def sum_bound(n_sites, diffs):
    """The largest difference two fp64 sums of the same n non-negative terms, each within (n-1) 2^-53 sum of the
    exact sum (spgg_overlap and np.sum), can show: per channel, for k = 1, 2."""
    return 2.0 * max(n_sites - 1, 0) * U * np.asarray(diffs)[..., 1:]


def _state(rs, L, nq=4, p_coop=0.5, rq=None):
    S = (rs.rand(L, L) >= p_coop).astype(np.uint8)
    R = rs.uniform(-10, 10, (L, L)) if rq is None else rs.randint(int(-10 / rq), int(10 / rq) + 1, (L, L)) * rq
    Q = rs.uniform(-0.5, 0.5, (L, L) + (2,) * (2 if nq == 4 else 3))
    return S, R, Q


def test_identical_states():
    rs = np.random.RandomState(1)
    st = _state(rs, 9)
    c, ch, d = numpy_overlap(st, st)
    assert np.array_equal(c, [[np.count_nonzero(st[0] == 0), 0], [0, np.count_nonzero(st[0] == 1)]])
    assert not ch.any() and not d.any() and ch.shape == (5,) and d.shape == (5, 3)


def test_all_sites_flipped():
    rs = np.random.RandomState(2)
    S, R, Q = _state(rs, 7, p_coop=0.3)
    c, ch, d = numpy_overlap((S, R, Q), (1 - S, R + 1.0, -Q), fields=("R", "Q"))
    nC = np.count_nonzero(S == 0)
    assert np.array_equal(c, [[0, nC], [49 - nC, 0]])
    assert ch[0] == 49 and d[0, 0] == 1.0 and d[0, 1] == 49.0 and d[0, 2] == 49.0
    q = Q.reshape(-1, 4)
    assert np.array_equal(ch[1:], np.count_nonzero(q, axis=0))
    assert np.array_equal(d[1:, 0], 2 * np.abs(q).max(0))


def test_signed_zeros_are_unchanged():
    L = 4
    S = np.zeros((L, L), np.uint8)
    R0, R1 = np.zeros((L, L)), np.full((L, L), -0.0)
    Q0, Q1 = np.full((L, L, 2, 2), -0.0), np.zeros((L, L, 2, 2))
    c, ch, d = numpy_overlap((S, R0, Q0), (S, R1, Q1))
    assert np.array_equal(c, [[16, 0], [0, 0]]) and not ch.any() and not d.any()


def test_int8_quantum_values_are_exact():
    """values on a quantum grid of 2^-k: every difference, square and partial sum is exact"""
    L = 6
    S = np.ones((L, L), np.uint8)
    R0 = np.arange(L * L).reshape(L, L) % 7 * 0.5 - 1.5
    R1 = R0.copy()
    R1[::2] += 0.25
    R1[1::3, 2] -= 3.0
    Q = np.zeros((L, L, 2, 2))
    c, ch, d = numpy_overlap((S, R0, Q), (S, R1, Q), fields=("R",))
    dd = (R1 - R0).reshape(-1)
    assert ch[0] == np.count_nonzero(dd) and d[0, 0] == np.abs(dd).max()
    assert d[0, 1] == sum(abs(x) for x in dd.tolist()) and d[0, 2] == sum(x * x for x in dd.tolist())
    assert np.array_equal(c, [[0, 0], [0, 36]])


def test_double_q_shapes():
    rs = np.random.RandomState(3)
    then, now = _state(rs, 5, nq=8), _state(rs, 5, nq=8)
    c, ch, d = numpy_overlap(then, now, nq=8)
    assert c.sum() == 25 and ch.shape == (9,) and d.shape == (9, 3)
    qa, qb = np.asarray(now[2]).reshape(25, 8), np.asarray(then[2]).reshape(25, 8)
    for z in range(8):
        assert d[1 + z, 0] == np.abs(qa[:, z] - qb[:, z]).max()
    c2, ch2, d2 = numpy_overlap(then, now, fields=("Q",), nq=8)
    assert np.array_equal(c2, c) and np.array_equal(ch2, ch[1:]) and np.array_equal(d2, d[1:])
    c3, ch3, d3 = numpy_overlap(then, now, fields=(), nq=8)
    assert np.array_equal(c3, c) and ch3.shape == (0,) and d3.shape == (0, 3)


def _result(counts, changed=None, diffs=None, batched=False, nq=4):
    from spgg_b200.engine import overlap_result
    counts = np.asarray(counts, np.int64).reshape(-1, 2, 2)
    n = counts.shape[0]
    m = 0 if changed is None else np.asarray(changed).shape[-1]
    changed = np.zeros((n, m), np.int64) if changed is None else np.asarray(changed).reshape(n, m)
    diffs = np.zeros((n, m, 3)) if diffs is None else np.asarray(diffs).reshape(n, m, 3)
    flags = (1 if m in (1, 1 + nq) else 0) | (2 if m >= nq else 0)
    return overlap_result(counts, changed, diffs, flags, (2, 2) if nq == 4 else (2, 2, 2), batched, 3, 10)


def test_overlap_result_layout():
    rs = np.random.RandomState(4)
    then, now = _state(rs, 8), _state(rs, 8)
    c, ch, d = numpy_overlap(then, now)
    o = _result(c, ch, d)
    assert o["t0"] == 3 and o["t"] == 10 and np.array_equal(o["S"], c)
    assert o["R_changed"] == ch[0] and np.array_equal(o["R_diff"], d[0])
    assert o["Q_changed"].shape == (2, 2) and o["Q_diff"].shape == (2, 2, 3)
    assert np.array_equal(o["Q_changed"].reshape(-1), ch[1:]) and np.array_equal(o["Q_diff"].reshape(4, 3), d[1:])
    ob = _result(np.stack([c, c]), np.stack([ch, ch]), np.stack([d, d]), batched=True)
    assert ob["S"].shape == (2, 2, 2) and ob["R_changed"].shape == (2,) and ob["Q_diff"].shape == (2, 2, 2, 3)
    o8 = _result(c, np.zeros(9, np.int64), np.zeros((9, 3)), nq=8)
    assert o8["Q_changed"].shape == (2, 2, 2) and o8["Q_diff"].shape == (2, 2, 2, 3)
    assert set(_result(c)) == {"S", "t0", "t"}


def test_overlap_measures():
    from spgg_b200.engine import overlap_measures
    N = 100
    # identity, mixed state: autocorrelation 1, Hamming 0, persistence 1
    m = overlap_measures({"S": [[30, 0], [0, 70]], "R_diff": [0.0, 0.0, 0.0]}, N)
    assert m["hamming"] == 0.0 and m["autocorrelation"] == pytest.approx(1.0)
    assert m["persistence_C"] == 1.0 and m["persistence_D"] == 1.0 and m["R_rms"] == 0.0 and m["R_mean_abs"] == 0.0
    # a hand count: f0 = 0.4, f = 0.5
    m = overlap_measures({"S": [[30, 10], [20, 40]], "Q_diff": np.tile([1.0, 8.0, 25.0], (2, 2, 1))}, N)
    assert m["hamming"] == 0.3
    assert m["autocorrelation"] == pytest.approx((0.3 - 0.2) / np.sqrt(0.4 * 0.6 * 0.5 * 0.5))
    assert m["persistence_C"] == 0.75 and m["persistence_D"] == pytest.approx(40 / 60)
    assert m["Q_rms"].shape == (2, 2) and np.allclose(m["Q_rms"], 0.5) and np.allclose(m["Q_mean_abs"], 0.08)
    # every site flipped: autocorrelation -1
    assert overlap_measures({"S": [[0, 40], [60, 0]]}, N)["autocorrelation"] == pytest.approx(-1.0)
    # uniform states: no fluctuation to correlate, and an empty class
    for S in ([[100, 0], [0, 0]], [[0, 0], [0, 100]], [[0, 0], [40, 60]], [[60, 40], [0, 0]]):
        m = overlap_measures({"S": S}, N)
        assert np.isnan(m["autocorrelation"]), S
    m = overlap_measures({"S": [[0, 0], [40, 60]]}, N)
    assert np.isnan(m["persistence_C"]) and m["persistence_D"] == 0.6 and m["hamming"] == 0.4
    m = overlap_measures({"S": [[60, 40], [0, 0]]}, N)
    assert np.isnan(m["persistence_D"]) and m["persistence_C"] == 0.6
    # a replica axis carries through
    m = overlap_measures({"S": [[[30, 0], [0, 70]], [[0, 0], [0, 100]]], "R_diff": [[0, 4.0, 4.0], [0, 1.0, 1.0]]}, N)
    assert m["hamming"].shape == (2,) and m["autocorrelation"][0] == pytest.approx(1.0)
    assert np.isnan(m["autocorrelation"][1]) and np.allclose(m["R_rms"], [0.2, 0.1])
    with pytest.raises(ValueError):
        overlap_measures({"S": np.zeros(3)}, N)


@pytest.mark.parametrize("world", [1, 2, 3, 4, 5])
def test_strip_assembly(world):
    """the strips' restatements assembled in rank order == the whole lattice's: counts, changed and max exactly,
    sums within the bound; the same parts always give the same bits"""
    from spgg_b200.strips import assemble_overlap, strip_rows
    L = 40
    rs = np.random.RandomState(world)
    then, now = _state(rs, L), _state(rs, L)
    now[1][::3] = then[1][::3]
    want = numpy_overlap(then, now)
    parts = []
    for k in range(world):
        row0, rows = strip_rows(L, world, k)
        sl = slice(row0, row0 + rows)
        c, ch, d = numpy_overlap(tuple(a[sl] for a in then), tuple(a[sl] for a in now))
        parts.append((c[None], ch[None], d[None]))
    c, ch, d = assemble_overlap(parts)
    assert c.shape == (1, 2, 2) and np.array_equal(c[0], want[0]) and np.array_equal(ch[0], want[1])
    assert np.array_equal(d[0, :, 0], want[2][:, 0])
    assert (np.abs(d[0, :, 1:] - want[2][:, 1:]) <= sum_bound(L * L, want[2])).all()
    again = assemble_overlap([tuple(x.copy() for x in p) for p in parts])
    assert all(a.tobytes() == b.tobytes() for a, b in zip((c, ch, d), again))
    s = np.zeros_like(d[..., 1:])
    for p in parts:
        s = s + p[2][..., 1:]
    assert s.tobytes() == d[..., 1:].copy().tobytes()       # rank order


def test_null_handle_is_rejected_without_a_gpu():
    import spgg_b200
    from spgg_b200 import _lib
    lib = spgg_b200.load()
    cnt = np.full(8, -7, np.int64)
    chg = np.full(16, -7, np.int64)
    dif = np.full(48, -7.0)
    it = C.c_int64(-7)
    for flags in (0, 1, 3):
        assert lib.spgg_snapshot(None, 0, 0, 1, flags) == _lib.E_INVALID
        assert lib.spgg_overlap(None, 0, 0, 1, flags, cnt.ctypes.data, chg.ctypes.data, dif.ctypes.data) == _lib.E_INVALID
    assert lib.spgg_snapshot_info(None, 0, C.byref(it), None, None, None) == _lib.E_INVALID
    assert lib.spgg_snapshot_free(None, 0) == _lib.E_INVALID
    assert (cnt == -7).all() and (chg == -7).all() and (dif == -7.0).all() and it.value == -7


def _null_engine(n_replicas=1, nq=4):
    import spgg_b200
    eng = spgg_b200.Engine.__new__(spgg_b200.Engine)
    eng.lib, eng._h, eng.L, eng.rows, eng.row0, eng.nq = spgg_b200.load(), C.c_void_p(), 16, 16, 0, nq
    eng.n_replicas = n_replicas
    return eng


def test_engine_overlap_checks_its_arguments():
    eng = _null_engine(n_replicas=3)
    for bad in (("R", "X"), "RQ", ("q",), (1,), ("S",)):
        with pytest.raises(ValueError, match="fields"):
            eng.snapshot(fields=bad)
        with pytest.raises(ValueError, match="fields"):
            eng.overlap(fields=bad)
    for rep in (3, -1, range(2, 4), range(0, 3, 2), range(1, 1), True, 1.0, "0"):
        with pytest.raises(ValueError, match="replica"):
            eng.snapshot(replica=rep)
        with pytest.raises(ValueError, match="replica"):
            eng.overlap(replica=rep)
    for slot in (-1, 8, 1.0, True, "0", None):
        for call in (lambda: eng.snapshot(slot=slot), lambda: eng.overlap(slot=slot),
                     lambda: eng.snapshot_info(slot), lambda: eng.drop_snapshot(slot)):
            with pytest.raises(ValueError, match="slot"):
                call()
    # valid arguments reach the library, which rejects the null handle
    for call in (lambda: eng.snapshot(7, replica=range(0, 3)), lambda: eng.overlap(0, replica=range(1, 3), fields=()),
                 lambda: eng.snapshot_info(3), lambda: eng.drop_snapshot(0)):
        with pytest.raises(ValueError, match="null"):
            call()


def test_strip_engine_overlap_checks_its_arguments_first():
    import torch
    from spgg_b200 import strips
    se = strips.StripEngine.__new__(strips.StripEngine)
    se.torch, se.L, se.world, se.rank = torch, 64, 1, 0
    with pytest.raises(ValueError, match="fields"):
        se.snapshot(fields=("S",))
    with pytest.raises(ValueError, match="fields"):
        se.overlap(fields=("S",))
    with pytest.raises(ValueError, match="slot"):
        se.snapshot(slot=8)
    with pytest.raises(ValueError, match="slot"):
        se.overlap(slot=-1)
