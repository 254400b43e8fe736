"""Block fields (include/spgg.h: spgg_block_fields, Engine.block_fields, StripEngine.block_fields) without a GPU:
the NumPy restatement the device tests compare with, checked against a loop over sites; the assembly of strip
partials into the whole lattice's; block_means; and the argument checks."""
import ctypes as C

import numpy as np
import pytest

U = 2.0 ** -53


def numpy_block_fields(S, R, Q, b, flags, row0=0, L=None):
    """Host restatement of spgg_block_fields on the rows [row0, row0 + rows) of an L x L lattice (S, R of shape
    (rows, L), Q of shape (rows, L, ...) as get_state returns them; R / Q may be None when not asked for).
    Returns counts int64 (nI, B, 2) {n, n_C}, sums float64 (nI, B, 2, m) [all, cooperators] and abs_sums
    (the same sums of |x|), over the block rows I0 .. I0 + nI - 1 that hold the rows."""
    S = np.asarray(S)
    rows, Lc = S.shape
    L = Lc if L is None else L
    B = -(-L // b)
    I0 = row0 // b
    nI = (row0 + rows - 1) // b - I0 + 1
    idx = (((np.arange(rows) + row0) // b - I0)[:, None] * B + (np.arange(L) // b)[None, :]).ravel()
    coop = (S == 0).ravel()
    nb = nI * B
    counts = np.stack([np.bincount(idx, minlength=nb), np.bincount(idx[coop], minlength=nb)], -1).astype(np.int64)
    chans = []
    if flags & 1:
        chans.append(np.asarray(R, np.float64).reshape(-1))
    if flags & 2:
        q = np.asarray(Q, np.float64).reshape(rows * L, -1)
        chans += [q[:, z] for z in range(q.shape[1])]
    m = len(chans)
    sums = np.zeros((nb, 2, m))
    abs_sums = np.zeros((nb, 2, m))
    for ch, x in enumerate(chans):
        sums[:, 0, ch] = np.bincount(idx, weights=x, minlength=nb)
        sums[:, 1, ch] = np.bincount(idx[coop], weights=x[coop], minlength=nb)
        abs_sums[:, 0, ch] = np.bincount(idx, weights=np.abs(x), minlength=nb)
        abs_sums[:, 1, ch] = np.bincount(idx[coop], weights=np.abs(x[coop]), minlength=nb)
    return counts.reshape(nI, B, 2), sums.reshape(nI, B, 2, m), abs_sums.reshape(nI, B, 2, m)


def sum_bound(counts, abs_sums):
    """The largest difference two fp64 sums of the same n values x_i, each within (n-1) 2^-53 sum |x_i| of the
    exact sum (spgg_block_fields and np.bincount), can show: per block, class and channel."""
    n = counts[..., :, None].astype(np.float64)     # (.., 2, 1): all sites, cooperators
    return 2.0 * np.maximum(n - 1.0, 0.0) * U * abs_sums


def _brute(S, R, Q, b, row0, L):
    rows = S.shape[0]
    B = -(-L // b)
    I0 = row0 // b
    nI = (row0 + rows - 1) // b - I0 + 1
    nq = Q.shape[-1]
    counts = np.zeros((nI, B, 2), np.int64)
    sums = np.zeros((nI, B, 2, 1 + nq))
    for i in range(rows):
        for j in range(L):
            I, J = (row0 + i) // b - I0, j // b
            vals = [R[i, j]] + list(Q[i, j])
            counts[I, J, 0] += 1
            for k in (0, 1) if S[i, j] == 0 else (0,):
                counts[I, J, 1] += k
                sums[I, J, k] += vals
    return counts, sums


def _dyadic(rs, shape, scale=1024):
    """Values whose sums are exact in any order, so the restatement must equal the loop bit for bit."""
    return rs.randint(-2048, 2048, shape) / scale


@pytest.mark.parametrize("L", range(4, 14))
def test_numpy_restatement_equals_the_loop(L):
    rs = np.random.RandomState(L)
    S = (rs.rand(L, L) < 0.6).astype(np.uint8)
    R = _dyadic(rs, (L, L), 2)
    for nq in (4, 8):
        Q = _dyadic(rs, (L, L, nq))
        for b in range(1, L + 1):
            for row0, rows in ((0, L), (1, L - 1), (L // 2, L - L // 2), (L // 3, 2), (L - 1, 1)):
                sl = slice(row0, row0 + rows)
                want_c, want_s = _brute(S[sl], R[sl], Q[sl], b, row0, L)
                c, s, a = numpy_block_fields(S[sl], R[sl], Q[sl].reshape(rows, L, *(2,) * (nq.bit_length() - 1)), b, 3,
                                             row0, L)
                assert np.array_equal(c, want_c), (b, row0, rows)
                assert np.array_equal(s, want_s), (b, row0, rows)
                assert (a >= np.abs(s)).all()
                # the flag sets select channels of the same sums
                assert np.array_equal(numpy_block_fields(S[sl], R[sl], None, b, 1, row0, L)[1], s[..., :1])
                assert np.array_equal(numpy_block_fields(S[sl], None, Q[sl], b, 2, row0, L)[1], s[..., 1:])
                assert numpy_block_fields(S[sl], None, None, b, 0, row0, L)[1].shape[-1] == 0


def _strip_parts(S, R, Q, b, world, pad_value):
    from spgg_b200 import strips
    from spgg_b200.engine import block_rows
    L = S.shape[0]
    nIs = [block_rows(L, b, *strips.strip_rows(L, world, k))[1] for k in range(world)]
    parts = []
    for k in range(world):
        row0, rows = strips.strip_rows(L, world, k)
        sl = slice(row0, row0 + rows)
        c, s, _ = numpy_block_fields(S[sl], R[sl], Q[sl], b, 3, row0, L)
        # padded to the largest block-row count, as the all-gather pads; the padding must not be read
        cp = np.full((max(nIs),) + c.shape[1:], pad_value, np.int64)
        sp = np.full((max(nIs),) + s.shape[1:], float(pad_value))
        cp[:len(c)], sp[:len(s)] = c, s
        parts.append((cp, sp))
    return parts


@pytest.mark.parametrize("world", range(1, 6))
@pytest.mark.parametrize("L", (20, 37, 64, 100))
def test_strip_partials_assemble_into_the_lattice(world, L):
    from spgg_b200 import strips
    rs = np.random.RandomState(world * 1000 + L)
    S = (rs.rand(L, L) < 0.5).astype(np.uint8)
    R = rs.randint(-20, 21, (L, L)) * 0.5
    Q = rs.uniform(-0.01, 0.01, (L, L, 4))
    for b in sorted({1, 3, 7, 16, 17, L // 2 + 1, L}):
        if -(-L // b) ** 2 > 1 << 24:
            continue
        want_c, want_s, want_a = numpy_block_fields(S, R, Q, b, 3)
        counts, sums = strips.assemble_block_fields(L, b, world, _strip_parts(S, R, Q, b, world, -999))
        assert counts.shape == want_c.shape and sums.shape == want_s.shape
        assert np.array_equal(counts, want_c), b
        assert np.array_equal(sums[..., 0], want_s[..., 0]), b    # half-integer R: exact in any order
        assert (np.abs(sums - want_s) <= sum_bound(want_c, want_a)).all(), b


def _means(S, R=None, Q=None, b=2):
    from spgg_b200.engine import block_means, block_result
    flags = (1 if R is not None else 0) | (2 if Q is not None else 0)
    c, s, _ = numpy_block_fields(S, R, Q, b, flags)
    return block_means(block_result(c[:, :, :], s, flags, (2, 2)))


def test_block_means_all_cooperators():
    L = 6
    R = np.arange(L * L, dtype=np.float64).reshape(L, L)
    Q = np.ones((L, L, 2, 2))
    m = _means(np.zeros((L, L), np.uint8), R, Q, b=3)
    assert (m["coop"] == 1.0).all()
    want = R.reshape(2, 3, 2, 3).mean(axis=(1, 3))
    assert np.allclose(m["R"], want) and np.allclose(m["R_C"], want)
    assert np.isnan(m["R_D"]).all() and np.isnan(m["Q_D"]).all()
    assert m["Q"].shape == (2, 2, 2, 2) and (m["Q_C"] == 1.0).all()


def test_block_means_all_defectors():
    L = 5
    R = np.full((L, L), -2.5)
    m = _means(np.ones((L, L), np.uint8), R, None, b=2)
    assert (m["coop"] == 0.0).all()
    assert (m["R"] == -2.5).all() and (m["R_D"] == -2.5).all()
    assert np.isnan(m["R_C"]).all()
    assert "Q" not in m


def test_block_means_checkerboard():
    L = 8
    S = (np.add.outer(np.arange(L), np.arange(L)) % 2).astype(np.uint8)
    R = np.where(S == 0, 3.0, -1.0)
    Q = np.stack([np.where(S == 0, 1.0, 0.0)] * 4, -1).reshape(L, L, 2, 2)
    m = _means(S, R, Q, b=2)
    assert m["coop"].shape == (4, 4) and (m["coop"] == 0.5).all()
    assert (m["R"] == 1.0).all() and (m["R_C"] == 3.0).all() and (m["R_D"] == -1.0).all()
    assert (m["Q_C"] == 1.0).all() and (m["Q_D"] == 0.0).all() and (m["Q"] == 0.5).all()


def test_block_means_ragged_last_block():
    L, b = 7, 3                      # blocks of 3, 3 and 1 rows / columns
    S = np.zeros((L, L), np.uint8)
    S[6, :] = 1                      # the last block row holds one row, all defectors
    S[:, 6] = 1
    R = np.ones((L, L))
    m = _means(S, R, None, b=b)
    c, _, _ = numpy_block_fields(S, R, None, b, 1)
    assert c[2, 2, 0] == 1 and c[0, 2, 0] == 3 and c[2, 0, 0] == 3 and c[0, 0, 0] == 9
    assert m["coop"][0, 0] == 1.0 and m["coop"][2, 2] == 0.0 and m["coop"][0, 2] == 0.0
    assert np.isnan(m["R_C"][2, :]).all() and np.isnan(m["R_D"][:2, :2]).all()
    assert (m["R"] == 1.0).all()


def test_null_handle_is_rejected_without_a_gpu():
    import spgg_b200
    from spgg_b200 import _lib
    lib = spgg_b200.load()
    cnt = np.full(8, -7, np.int64)
    sums = np.full(8, -7.0)
    for flags in (0, 1, 3):
        rc = lib.spgg_block_fields(None, 0, 1, flags, cnt.ctypes.data, sums.ctypes.data)
        assert rc == _lib.E_INVALID
        with pytest.raises(ValueError):
            _lib.check(rc)
    assert (cnt == -7).all() and (sums == -7.0).all()


def test_engine_block_fields_checks_fields_and_reaches_the_library_check():
    import spgg_b200
    eng = spgg_b200.Engine.__new__(spgg_b200.Engine)
    eng.lib, eng._h, eng.L, eng.rows, eng.row0, eng.nq = spgg_b200.load(), C.c_void_p(), 16, 16, 0, 4
    for bad in (("R", "X"), "RQ", ("q",), (1,), ("R", None)):
        with pytest.raises(ValueError, match="fields"):
            eng.block_fields(4, fields=bad)
    for b in (4, 0, 17):
        with pytest.raises(ValueError, match="null"):
            eng.block_fields(b, fields=())


def test_strip_engine_block_fields_checks_fields_first():
    import torch
    from spgg_b200 import strips
    se = strips.StripEngine.__new__(strips.StripEngine)
    se.torch, se.L, se.world, se.rank = torch, 64, 1, 0
    with pytest.raises(ValueError, match="fields"):
        se.block_fields(4, fields=("S",))
