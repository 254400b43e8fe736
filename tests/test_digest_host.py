"""The host restatements the large-lattice GPU tests rest on, against plain NumPy and Python.

``c_oracle.state_digest`` restates ``spgg_state_digest`` (csrc/spgg_kernels.cuh: k_state_digest),
``c_oracle.init_random`` / ``init_random_digest`` restate ``spgg_init_random`` (k_init_random) and
``c_oracle.explore_actions`` gives the actions of an iteration at epsilon = 1.  Each is checked
here against an independent restatement: NumPy uint64 arithmetic for the digest, ``c_oracle.philox``
plus exact rationals for the start state (the device forms -0.01 + 0.02 u as one fused multiply-add)."""
from fractions import Fraction

import numpy as np
import pytest

from oracle import c_oracle

U64 = np.uint64


def _mix(x):
    with np.errstate(over="ignore"):
        x = x ^ (x >> U64(33))
        x = x * U64(0xff51afd7ed558ccd)
        x = x ^ (x >> U64(33))
        x = x * U64(0xc4ceb9fe1a85ec53)
        return x ^ (x >> U64(33))


def _np_digest(S, R, Q, row0=0):
    """k_state_digest in NumPy: sum over sites of (hash | 1) * (bits + 1) mod 2^64 per word."""
    rows, L = S.shape
    i, j = np.meshgrid(np.arange(row0, row0 + rows, dtype=U64), np.arange(L, dtype=U64), indexing="ij")
    key = (i << U64(32)) | j
    nq = Q.size // S.size
    Qf = np.ascontiguousarray(Q, np.float64).reshape(rows, L, nq)
    with np.errstate(over="ignore"):
        k3 = key * U64(3)
        dS = ((_mix(k3 + U64(1)) | U64(1)) * (S.astype(U64) + U64(1))).sum(dtype=U64)
        dR = ((_mix(k3 + U64(2)) | U64(1)) * (np.ascontiguousarray(R, np.float64).view(U64) + U64(1))).sum(dtype=U64)
        dQ = U64(0)
        for z in range(nq):
            h = _mix(k3 + U64(3) + (U64(z + 1) << U64(58))) | U64(1)
            dQ += (h * (np.ascontiguousarray(Qf[..., z]).view(U64) + U64(1))).sum(dtype=U64)
    return int(dS), int(dR), int(dQ)


def _state(rows, L, nq, kind, rs):
    S = rs.randint(0, 2, (rows, L)).astype(np.uint8)
    qshape = (rows, L, 2, 2) if nq == 4 else (rows, L, 2, 2, 2)
    if kind == "int8":                 # int8 units times a quantum of 1/2, as get_state widens them
        R = rs.randint(-20, 21, (rows, L)) * 0.5
        Q = rs.uniform(-1, 1, qshape).astype(np.float32).astype(np.float64)
    elif kind == "fp32":
        R = rs.uniform(-10, 10, (rows, L)).astype(np.float32).astype(np.float64)
        Q = rs.uniform(-1, 1, qshape).astype(np.float32).astype(np.float64)
    else:
        R = rs.uniform(-10, 10, (rows, L))
        Q = rs.uniform(-1, 1, qshape)
    R.flat[::7] = 0.0
    R.flat[3::11] = -0.0
    Q.flat[::13] = -0.0
    return S, R, Q


GEOMS = [(37, 37, 0, 4), (50, 50, 0, 4), (40, 96, 0, 8), (19, 45, 26, 4), (16, 64, 48, 8)]


@pytest.mark.parametrize("kind", ["int8", "fp32", "fp64"])
@pytest.mark.parametrize("rows,L,row0,nq", GEOMS)
def test_digest_equals_numpy(rows, L, row0, nq, kind):
    """Odd L, L % 32 != 0, both Q widths, strips starting at row0 > 0, signed zeros."""
    S, R, Q = _state(rows, L, nq, kind, np.random.RandomState(rows + L + nq))
    want = _np_digest(S, R, Q, row0)
    assert c_oracle.state_digest(S, R, Q, L=L, row0=row0) == want
    w = c_oracle.digest_weights(L, nq, row0=row0, rows=rows)
    assert c_oracle.state_digest(S, R, Q, L=L, row0=row0, weights=w) == want
    assert c_oracle.state_digest(S, R, None, L=L, row0=row0) == want[:2] + (0,)


def test_digests_of_row_blocks_add_up():
    L = 45
    S, R, Q = _state(L, L, 8, "fp32", np.random.RandomState(3))
    whole = c_oracle.state_digest(S, R, Q)
    parts = [c_oracle.state_digest(S[a:b], R[a:b], Q[a:b], L=L, row0=a) for a, b in ((0, 7), (7, 30), (30, 45))]
    assert tuple(sum(p[k] for p in parts) % 2 ** 64 for k in range(3)) == whole


@pytest.mark.parametrize("P,k,nq", [(12, 3, 4), (8, 4, 8), (7, 5, 4)])
def test_periodic_digest_equals_tiled_array(P, k, nq):
    S, R, Q = _state(P, P, nq, "fp32", np.random.RandomState(P * k))
    L = P * k
    reps = (k, k) + (1,) * (Q.ndim - 2)
    want = _np_digest(np.tile(S, (k, k)), np.tile(R, (k, k)), np.tile(Q, reps))
    assert c_oracle.state_digest(S, R, Q, L=L, period=P) == want
    w = c_oracle.digest_weights(L, nq, period=P)
    assert w.shape == (P, P, 2 + nq)
    assert c_oracle.state_digest(S, R, Q, L=L, period=P, weights=w) == want
    with pytest.raises(ValueError):
        c_oracle.state_digest(S, R, Q, L=L + 1, period=P)


def test_every_single_value_change_changes_its_word():
    """Sign flips (including +0.0 -> -0.0) of any one R or Q value, at every site of a small lattice."""
    L = 24
    S, R, Q = _state(L, L, 8, "fp64", np.random.RandomState(9))
    R[R == 0] = 1.5
    d0 = c_oracle.state_digest(S, R, Q)
    w = c_oracle.digest_weights(L, 8)
    Qf = Q.reshape(L, L, 8)
    for i in range(L):
        for j in range(L):
            R[i, j] = -R[i, j]
            d = c_oracle.state_digest(S, R, Q, weights=w)
            R[i, j] = -R[i, j]
            assert d[1] != d0[1] and (d[0], d[2]) == (d0[0], d0[2]), (i, j)
            z = (i + j) % 8
            Qf[i, j, z] = -Qf[i, j, z]
            d = c_oracle.state_digest(S, R, Q, weights=w)
            Qf[i, j, z] = -Qf[i, j, z]
            assert d[2] != d0[2] and d[:2] == d0[:2], (i, j, z)


# ------------------------------------------------------------------ k_init_random
def _fma_q(word, fp32):
    """-0.01 + 0.02 * u with u = (word >> 8) / 2^24, rounded once (exact rational arithmetic)."""
    q = float(Fraction(0.02) * Fraction(int(word) >> 8, 1 << 24) + Fraction(-0.01))
    return float(np.float32(q)) if fp32 else q


def _py_init_random(L, seed, nq, fp32, row0, rows):
    key = [seed & 0xffffffff, seed >> 32]
    S = np.zeros((rows, L), np.uint8)
    Q = np.zeros((rows, L, nq))
    nW = (L + 31) // 32
    for i in range(rows):
        for wi in range(nW):
            word = int(c_oracle.philox([wi >> 2, row0 + i, 0, 2], key)[wi & 3])
            for c in range(wi * 32, min(L, wi * 32 + 32)):
                S[i, c] = (word >> (c & 31)) & 1
        for j in range(L):
            for t in range(nq // 4):
                w = c_oracle.philox([j, row0 + i, t, 1], key)
                for z in range(4):
                    Q[i, j, 4 * t + z] = _fma_q(w[z], fp32)
    return S, np.zeros((rows, L)), Q


@pytest.mark.parametrize("L,row0,rows,nq,precision", [(37, 0, 37, 4, "fp32"), (33, 0, 33, 8, "fp64"),
                                                      (70, 21, 9, 4, "fp64"), (64, 40, 16, 8, "fp32")])
def test_init_random_equals_philox_restatement(L, row0, rows, nq, precision):
    seed = 0x1234_5678_9abc_def0 + L
    S, R, Q = c_oracle.init_random(L, seed, nq, precision, row0=row0, rows=rows)
    Sw, Rw, Qw = _py_init_random(L, seed, nq, precision == "fp32", row0, rows)
    assert np.array_equal(S, Sw)
    assert np.array_equal(R, Rw) and not np.signbit(R).any()
    assert np.array_equal(Q.reshape(rows, L, nq), Qw)
    assert Q.shape == ((rows, L, 2, 2) if nq == 4 else (rows, L, 2, 2, 2))
    assert 0.3 < S.mean() < 0.7 and -0.0101 < Q.min() < -0.009 and 0.009 < Q.max() < 0.01


def test_init_random_fma_differs_from_two_roundings():
    """The restatement is only right with the fused multiply-add: some words round differently."""
    words = np.arange(0, 1 << 24, 4099, dtype=np.uint64) << np.uint64(8)
    fused = np.array([_fma_q(w, False) for w in words])
    unfused = -0.01 + 0.02 * ((words >> np.uint64(8)).astype(np.float64) / 16777216.0)
    assert (fused != unfused).any()


@pytest.mark.parametrize("L,row0,rows,nq,precision", [(37, 0, 37, 4, "fp32"), (96, 32, 48, 8, "fp32"),
                                                      (45, 5, 20, 4, "fp64")])
def test_init_random_digest_equals_digest_of_state(L, row0, rows, nq, precision):
    seed = 987654321 + L
    S, R, Q = c_oracle.init_random(L, seed, nq, precision, row0=row0, rows=rows)
    want = _np_digest(S, R, Q, row0)
    assert c_oracle.init_random_digest(L, seed, nq, precision, row0=row0, rows=rows) == want


def test_explore_actions_are_the_action_words():
    L, seed, step = 37, 2 ** 40 + 17, 3
    a = c_oracle.explore_actions(L, seed, step, 5, 9)
    want = np.array([[c_oracle.site_word(seed, step, 0, i, j) & 1 for j in range(L)] for i in range(5, 9)])
    assert np.array_equal(a, want)
