"""Host side of the cluster labelling (include/spgg.h: spgg_clusters): the periodic oracle the GPU
tests compare with, checked against a plain breadth-first search on the torus, and the argument
checks that need no GPU."""
import ctypes as C
from collections import deque

import numpy as np
import pytest
from scipy.ndimage import label


def periodic_label(mask):
    """``scipy.ndimage.label(mask)`` on the torus: clusters also join across row L-1 | 0 and column
    L-1 | 0; labels 1..n in increasing order of each cluster's smallest linear index."""
    mask = np.asarray(mask, bool)
    lab, n = label(mask)
    parent = np.arange(n + 1)

    def find(x):
        while parent[x] != x:
            parent[x] = parent[parent[x]]
            x = parent[x]
        return x

    for a, b in ((lab[-1, :], lab[0, :]), (lab[:, -1], lab[:, 0])):
        for x, y in zip(a[(a > 0) & (b > 0)], b[(a > 0) & (b > 0)]):
            rx, ry = find(x), find(y)
            if rx != ry:
                parent[max(rx, ry)] = min(rx, ry)
    root = np.array([find(x) for x in range(n + 1)])
    merged = root[lab]
    # scipy numbers in raster order of first sites, so a merged set's smallest scipy label is its first site
    roots = np.unique(root[1:])
    rank = np.zeros(n + 1, np.int64)
    rank[roots] = np.arange(1, len(roots) + 1)
    return rank[merged].astype(np.int32), len(roots)


def bfs_torus_label(mask):
    mask = np.asarray(mask, bool)
    H, W = mask.shape
    out = np.zeros((H, W), np.int32)
    n = 0
    for i in range(H):
        for j in range(W):
            if mask[i, j] and not out[i, j]:
                n += 1
                out[i, j] = n
                q = deque([(i, j)])
                while q:
                    a, b = q.popleft()
                    for da, db in ((1, 0), (-1, 0), (0, 1), (0, -1)):
                        x, y = (a + da) % H, (b + db) % W
                        if mask[x, y] and not out[x, y]:
                            out[x, y] = n
                            q.append((x, y))
    return out, n


def _patterns(L):
    yield np.ones((L, L), bool)
    yield np.zeros((L, L), bool)
    ii, jj = np.indices((L, L))
    yield (ii + jj) % 2 == 0
    yield jj % 3 == 0
    yield ii % 2 == 1
    yield (jj == 0) | (jj == L - 1)
    yield (ii == 0) | (ii == L - 1)
    comb = np.zeros((L, L), bool)
    comb[0, :] = True
    comb[:, ::2] = True
    yield comb


@pytest.mark.parametrize("L", list(range(1, 41)))
def test_periodic_oracle_equals_bfs_on_the_torus(L):
    rs = np.random.RandomState(L)
    masks = [rs.rand(L, L) < p for p in (0.3, 0.5, 0.593, 0.7)] + list(_patterns(L))
    for m in masks:
        got, n = periodic_label(m)
        want, nw = bfs_torus_label(m)
        assert n == nw
        assert np.array_equal(got, want)


def test_periodic_oracle_without_seams_is_scipy():
    m = np.zeros((9, 9), bool)
    m[2:4, 2:7] = True
    m[6, 1] = True
    got, n = periodic_label(m)
    want, nw = label(m)
    assert n == nw and np.array_equal(got, want)


def test_cluster_entry_points_reject_a_null_handle_without_a_gpu():
    import spgg_b200
    from spgg_b200 import _lib
    lib = spgg_b200.load()
    n = C.c_int64(-7)
    sizes = np.zeros(4, np.int64)
    labels = np.zeros(16, np.int32)
    for rc in (lib.spgg_clusters(None, 0, 0, 0, C.byref(n)),
               lib.spgg_cluster_sizes(None, sizes.ctypes.data, 4),
               lib.spgg_cluster_labels(None, labels.ctypes.data)):
        assert rc == _lib.E_INVALID
        with pytest.raises(ValueError):
            _lib.check(rc)
    assert n.value == -7
    # the Engine methods check `of` before they reach the library
    eng = spgg_b200.Engine.__new__(spgg_b200.Engine)
    eng.lib, eng._h, eng.rows, eng.L = lib, C.c_void_p(), 4, 4
    for of in ("X", 2, None, True):
        with pytest.raises(ValueError, match="of must be"):
            eng.cluster_sizes(of=of)
    with pytest.raises(ValueError):
        eng.cluster_sizes()
    with pytest.raises(ValueError):
        eng.cluster_labels(of="D", periodic=True)
