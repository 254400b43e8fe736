"""Strategy pair counts (include/spgg.h: spgg_pair_counts, Engine.pair_counts) without a GPU: the NumPy
restatement the device tests compare with, checked against the definition by brute force; pair_correlation
on lattices whose correlations are known; and the argument checks of the new entry points."""
import ctypes as C

import numpy as np
import pytest


def numpy_pair_counts(S, max_d, ds=None):
    """Host restatement of spgg_pair_counts: int64 (2, max_d+1, 2), [ax, d] = (#x with C(x) and C(x + d e_ax),
    #x whose partner holds the other strategy) over the torus, [ax, 0] = (n_C, 0).  S == 0 cooperates.  With
    ``ds`` only those offsets (and d = 0) are filled in; the rest stays -1."""
    c = np.asarray(S) == 0
    out = np.full((2, max_d + 1, 2), -1, np.int64)
    for ax in (0, 1):
        out[ax, 0] = (np.count_nonzero(c), 0)
        for d in (range(1, max_d + 1) if ds is None else ds):
            p = np.roll(c, -d, axis=ax)        # p[x] = c[x + d e_ax]
            out[ax, d] = (np.count_nonzero(c & p), np.count_nonzero(c != p))
    return out


def _brute(S, max_d):
    L = S.shape[0]
    out = np.zeros((2, max_d + 1, 2), np.int64)
    for ax in (0, 1):
        for d in range(max_d + 1):
            for i in range(L):
                for j in range(L):
                    a = S[i, j]
                    b = S[(i + d) % L, j] if ax == 0 else S[i, (j + d) % L]
                    out[ax, d, 0] += a == 0 and b == 0
                    out[ax, d, 1] += a != b
    return out


@pytest.mark.parametrize("L", range(4, 13))
def test_numpy_restatement_equals_the_definition(L):
    rs = np.random.RandomState(L)
    for p in (0.1, 0.5, 0.9):
        S = (rs.rand(L, L) >= p).astype(np.uint8)
        want = _brute(S, L // 2)
        got = numpy_pair_counts(S, L // 2)
        assert np.array_equal(got, want), (L, p)
        N, nC = L * L, int((S == 0).sum())
        assert np.array_equal(2 * (nC - got[:, :, 0]), got[:, :, 1])     # n_CD = n_DC on the torus
        sub = numpy_pair_counts(S, L // 2, ds=[1, L // 2])
        assert np.array_equal(sub[:, [0, 1, L // 2]], want[:, [0, 1, L // 2]])
        assert (got[:, :, 0] + got[:, :, 1] <= N).all()


def _corr(S, max_d):
    from spgg_b200.engine import pair_correlation
    return pair_correlation(numpy_pair_counts(S, max_d), S.size)


@pytest.mark.parametrize("L", [4, 8, 10, 64])
def test_pair_correlation_of_a_checkerboard_alternates(L):
    ii, jj = np.indices((L, L))
    C_ = _corr(((ii + jj) % 2).astype(np.uint8), L // 2)
    assert C_.shape == (2, L // 2 + 1)
    assert np.array_equal(C_, np.tile((-1.0) ** np.arange(L // 2 + 1), (2, 1)))


def test_pair_correlation_of_stripes_and_the_interface_density():
    from spgg_b200.engine import pair_correlation
    L = 12
    ii, jj = np.indices((L, L))
    S = (jj % 4 < 2).astype(np.uint8)       # vertical stripes of width 2: constant down a column
    counts = numpy_pair_counts(S, L // 2)
    C_ = pair_correlation(counts, S.size)
    assert np.array_equal(C_[0], np.ones(L // 2 + 1))
    assert np.allclose(C_[1], [1, 0, -1, 0, 1, 0, -1])
    # interface density: no C-D bond along the columns, every second bond across them
    assert counts[0, 1, 1] == 0 and counts[1, 1, 1] / S.size == 0.5


def test_pair_correlation_is_nan_without_both_strategies():
    from spgg_b200.engine import pair_correlation
    for S in (np.zeros((6, 6), np.uint8), np.ones((6, 6), np.uint8)):
        assert np.isnan(_corr(S, 3)).all()
    with pytest.raises(ValueError):
        pair_correlation(np.zeros((3, 2, 2)), 36)


def test_pair_entry_points_reject_a_null_handle_without_a_gpu():
    import spgg_b200
    from spgg_b200 import _lib
    lib = spgg_b200.load()
    buf = np.full(64, -7, np.int64)
    for rc in (lib.spgg_pair_counts(None, 0, 1, buf.ctypes.data),
               lib.spgg_strip_pair_record_bytes(None, 1, 1),
               lib.spgg_strip_pair_record(None, 1, 1, buf.ctypes.data),
               lib.spgg_strip_pair_counts(None, 1, 0, buf.ctypes.data, 1, 1, buf.ctypes.data)):
        assert rc == _lib.E_INVALID
        with pytest.raises(ValueError):
            _lib.check(rc)
    assert (buf == -7).all()


def test_strip_engine_pair_counts_reaches_the_library_check():
    import torch
    import spgg_b200
    from spgg_b200 import strips
    se = strips.StripEngine.__new__(strips.StripEngine)
    se.lib, se.h, se._open, se.torch = spgg_b200.load(), C.c_void_p(), 0, torch
    se.L, se.world, se.rank = 64, 1, 0
    with pytest.raises(ValueError, match="null handle"):
        se.pair_counts(4)
