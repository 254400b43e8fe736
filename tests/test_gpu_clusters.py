"""Cluster labelling on the device (include/spgg.h: spgg_clusters, Engine.cluster_sizes /
cluster_labels): labels and sizes equal scipy.ndimage.label(S == which) exactly, and the periodic
variant equals the torus oracle of test_clusters_host.py, on uploaded lattices, on hand-made
patterns and on the state every kernel path leaves behind; labelling never disturbs a run."""
import os
import subprocess
import sys

import numpy as np
import pytest
from scipy.ndimage import label

from helpers import C1, C2, full_params
from test_clusters_host import periodic_label

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _engine(*a, **k):
    import spgg_b200
    return spgg_b200.Engine(*a, **k)


def _expected(S, of, periodic):
    m = np.asarray(S) == (0 if of in ("C", 0) else 1)
    if periodic:
        return periodic_label(m)
    lab, n = label(m)
    return lab.astype(np.int32), n


def _check(eng, S, replica=0, combos=(("C", False), ("D", False), ("C", True), ("D", True)), labels=True):
    for of, periodic in combos:
        want, n = _expected(S, of, periodic)
        sizes = eng.cluster_sizes(replica, of=of, periodic=periodic)
        assert sizes.dtype == np.int64 and len(sizes) == n, (of, periodic)
        assert np.array_equal(sizes, np.bincount(want.ravel(), minlength=n + 1)[1:]), (of, periodic)
        if labels:
            got, ng = eng.cluster_labels(replica, of=of, periodic=periodic)
            assert ng == n and got.dtype == np.int32 and got.shape == S.shape
            assert np.array_equal(got, want), (of, periodic)


def _set(eng, S, replica=0):
    L = eng.L
    q = np.zeros((L, L) + ((2, 2) if eng.nq == 4 else (2, 2, 2)))
    eng.set_state(S, np.zeros((L, L)), q, replica=replica)


@pytest.mark.parametrize("L", [4, 5, 31, 32, 33, 100, 128, 131, 200, 1000, 1024, 4096])
def test_random_lattices_equal_scipy(L):
    eng = _engine(full_params(dict(C1, L=L)), seeds=1, precision="fp32")
    rs = np.random.RandomState(L)
    for p in (0.3, 0.5, 0.593, 0.7):
        S = (rs.rand(L, L) >= p).astype(np.uint8)      # cooperator (S == 0) with probability p
        _set(eng, S)
        _check(eng, S, labels=L < 4096 or p == 0.593)
    eng.close()


def _serpentine(L):
    """One-site-wide path that snakes through the lattice row by row: about L^2/2 sites in one cluster,
    the deepest union-find there is."""
    S = np.ones((L, L), np.uint8)
    S[::2, :] = 0
    for i in range(1, L, 2):
        S[i, L - 1 if (i // 2) % 2 == 0 else 0] = 0
    return S


def _patterns(L):
    ii, jj = np.indices((L, L))
    yield "all C", np.zeros((L, L), np.uint8)
    yield "all D", np.ones((L, L), np.uint8)
    yield "checkerboard", ((ii + jj) % 2).astype(np.uint8)
    yield "vertical stripes", (jj % 2).astype(np.uint8)
    yield "vertical stripes 3", (jj % 3 != 1).astype(np.uint8)
    yield "horizontal stripes", (ii % 2).astype(np.uint8)
    yield "word-edge stripes", ~((jj % 32 == 31) | (jj % 32 == 0)) & 1
    yield "seam stripes", (~((jj == 0) | (jj == L - 1) | (ii == 0) | (ii == L - 1)) & 1).astype(np.uint8)
    yield "serpentine", _serpentine(L)
    comb = np.ones((L, L), np.uint8)
    comb[0, :] = 0
    comb[:, ::2] = 0
    yield "comb", comb
    yield "last column C", (jj != L - 1).astype(np.uint8)


@pytest.mark.parametrize("L", [4, 33, 100, 256, 257, 1000])
def test_patterns(L):
    eng = _engine(full_params(dict(C1, L=L)), seeds=1, precision="fp32")
    for name, S in _patterns(L):
        S = np.asarray(S, np.uint8)
        _set(eng, S)
        try:
            _check(eng, S)
        except AssertionError as e:
            raise AssertionError(f"{name}: {e}") from e
    # the counts the patterns are built for
    _set(eng, np.zeros((L, L), np.uint8))
    assert list(eng.cluster_sizes()) == [L * L] and list(eng.cluster_sizes(periodic=True)) == [L * L]
    assert len(eng.cluster_sizes(of="D")) == 0
    lab, n = eng.cluster_labels(of="D")
    assert n == 0 and not lab.any()
    ii, jj = np.indices((L, L))
    _set(eng, ((ii + jj) % 2).astype(np.uint8))
    assert len(eng.cluster_sizes()) == (L * L + 1) // 2
    _set(eng, _serpentine(L))
    assert list(eng.cluster_sizes()) == [int((_serpentine(L) == 0).sum())]
    eng.close()


def test_spare_bits_of_the_last_word_are_not_sites():
    """L % 32 != 0: the bits beyond column L-1 of each row's last word are no sites of either kind."""
    for L in (33, 100, 131):
        eng = _engine(full_params(dict(C1, L=L)), seeds=1, precision="fp32")
        for S in (np.ones((L, L), np.uint8), np.zeros((L, L), np.uint8)):
            _set(eng, S)
            _check(eng, S)
        eng.init_random(5)
        _check(eng, eng.get_state(want_q=False)[0])
        eng.close()


def _after_steps(p, L, n, env=None, precision="fp32", monkeypatch=None, want=None):
    if env:
        for k, v in env.items():
            monkeypatch.setenv(k, v)
    try:
        eng = _engine(full_params(dict(p, L=L)), seeds=3, precision=precision)
    finally:
        if env:
            for k in env:
                monkeypatch.delenv(k, raising=False)
    if want:
        assert want in eng.describe(), eng.describe()
    eng.init_random(11)
    eng.step(n)
    S = eng.get_state(want_q=False)[0]
    _check(eng, S, labels=L <= 1000)
    eng.close()


@pytest.mark.parametrize("name,p,L,env,prec,want", [
    ("resident_cluster", C1, 100, None, "fp32", "resident: cluster"),
    ("resident_grid", C2, 1000, None, "fp32", "cooperative grid"),
    ("fast_4096", C1, 4096, None, "fp32", "fast"),
    ("fast_256", C1, 256, {"SPGG_NO_RESIDENT": "1"}, "fp32", "fast"),
    ("lean_fp64", C1, 97, None, "fp64", "k_step_lean"),
    ("sarsa", dict(C1, algorithm="sarsa"), 131, None, "fp32", "k_step"),
    ("double_q", dict(C2, algorithm="double_qlearning"), 131, None, "fp32", "k_step"),
])
def test_after_stepping_on_every_path(monkeypatch, name, p, L, env, prec, want):
    _after_steps(p, L, 37, env, prec, monkeypatch, want)


_POISON_CHILD = r"""
import sys, numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {root!r} + "/tests")
import spgg_b200
from helpers import C1, full_params
from scipy.ndimage import label
L = 256
eng = spgg_b200.Engine(full_params(dict(C1, L=L)), seeds=9, precision="fp32")
assert eng.describe().startswith("fast"), eng.describe()
eng.init_random(4)
eng.step(120)
sizes = eng.cluster_sizes()           # the first synchronising call: it completes the re-run itself
st = eng.status()
assert st.speculation_failures >= 1, st.speculation_failures
assert st.iteration == 120
S = eng.get_state(want_q=False)[0]
lab, n = label(S == 0)
assert np.array_equal(sizes, np.bincount(lab.ravel(), minlength=n + 1)[1:])
print("ok", st.speculation_failures)
"""


def test_fast_path_with_a_pending_rerun():
    env = dict(os.environ, SPGG_NO_RESIDENT="1", SPGG_SPEC_TEST_POISON="5")
    r = subprocess.run([sys.executable, "-c", _POISON_CHILD.format(root=ROOT)], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_batch_replicas_and_a_stopped_replica(monkeypatch):
    """Each replica of a batch, including one that stopped in an earlier chunk (its planes are copied
    forward to the parity the running replicas ended on)."""
    L = 24
    p_stop = full_params(dict(C1, L=L, epsilon=0.0, epsilon_min=0.0))
    Q0 = np.zeros((L, L, 2, 2))
    Q0[..., 1] = 1.0                      # everybody defects after iteration 1
    rs = np.random.RandomState(2)
    for no_res in (False, True):
        if no_res:
            monkeypatch.setenv("SPGG_NO_RESIDENT", "1")
        eng = _engine([p_stop, full_params(dict(C1, L=L)), full_params(dict(C1, L=L, r=4.0))], seeds=[1, 2, 3],
                      precision="fp32")
        monkeypatch.delenv("SPGG_NO_RESIDENT", raising=False)
        eng.set_state(rs.randint(0, 2, (L, L)), np.zeros((L, L)), Q0, replica=0)
        for r in (1, 2):
            eng.set_state(rs.randint(0, 2, (L, L)), np.zeros((L, L)), rs.uniform(-0.01, 0.01, (L, L, 2, 2)), replica=r)
        eng.step(4)
        eng.step(7)                       # replica 0 stopped in the chunk before
        assert eng.status(0).stopped_at == 1 and eng.status(1).iteration == 11
        for r in range(3):
            _check(eng, eng.get_state(r, want_q=False)[0], replica=r)
        eng.close()
    # a larger batch on the general path
    L = 131
    eng = _engine([full_params(dict(C1, L=L, r=3.0 + 0.5 * i)) for i in range(3)], seeds=[5, 6, 7], precision="fp32")
    for r in range(3):
        eng.init_random(20 + r, replica=r)
    eng.step(9)
    for r in range(3):
        _check(eng, eng.get_state(r, want_q=False)[0], replica=r)
    eng.close()


@pytest.mark.parametrize("name,L,env,prec", [
    ("resident", 100, None, "fp32"),
    ("fast", 256, {"SPGG_NO_RESIDENT": "1"}, "fp32"),
    ("lean", 97, None, "fp64"),
])
def test_labelling_does_not_disturb_the_run(monkeypatch, name, L, env, prec):
    p = full_params(dict(C1, L=L))
    outs = []
    for chunks in ((200,), (50, 50, 50, 50)):
        for k, v in (env or {}).items():
            monkeypatch.setenv(k, v)
        eng = _engine(p, seeds=8, precision=prec)
        for k in (env or {}):
            monkeypatch.delenv(k, raising=False)
        eng.init_random(17)
        rows = []
        for c in chunks:
            eng.step(c)
            rows.append(eng.stats()[1:])
            if len(chunks) > 1:
                eng.cluster_sizes(of="D", periodic=True)
                eng.cluster_labels()
        outs.append((eng.digest(),) + eng.get_state() + (np.vstack(rows),))
        eng.close()
    for a, b in zip(*outs):
        assert np.array_equal(np.asarray(a), np.asarray(b))


def test_getters_need_a_current_result():
    import spgg_b200
    from spgg_b200 import _lib
    import ctypes as C
    L = 64
    eng = _engine(full_params(dict(C1, L=L)), seeds=1, precision="fp32")
    lib, h = eng.lib, eng._h
    sizes = np.zeros(L * L, np.int64)
    labels = np.zeros(L * L, np.int32)

    def getters_fail():
        assert lib.spgg_cluster_sizes(h, sizes.ctypes.data, 0) == _lib.E_STATE
        assert lib.spgg_cluster_labels(h, labels.ctypes.data) == _lib.E_STATE

    def label_now():
        n = C.c_int64()
        assert lib.spgg_clusters(h, 0, 0, 0, C.byref(n)) == 0
        assert lib.spgg_cluster_labels(h, labels.ctypes.data) == 0
        assert lib.spgg_cluster_sizes(h, sizes.ctypes.data, n.value + 1) == _lib.E_INVALID
        return n.value

    getters_fail()
    eng.init_random(3)
    label_now()
    eng.step(3)
    getters_fail()
    label_now()
    S, R, Q = eng.get_state()
    eng.set_state(S, R, Q)
    getters_fail()
    label_now()
    eng.init_random(4)
    getters_fail()
    label_now()
    eng.set_progress(0, [eng.status().epsilon])
    getters_fail()
    n = label_now()
    assert lib.spgg_cluster_sizes(h, sizes.ctypes.data, n) == 0
    # bad arguments
    nn = C.c_int64()
    assert lib.spgg_clusters(h, 1, 0, 0, C.byref(nn)) == _lib.E_INVALID
    assert lib.spgg_clusters(h, 0, 2, 0, C.byref(nn)) == _lib.E_INVALID
    assert lib.spgg_clusters(h, 0, 0, 2, C.byref(nn)) == _lib.E_INVALID
    assert lib.spgg_clusters(h, 0, 0, 0, None) == _lib.E_INVALID
    assert lib.spgg_cluster_labels(h, None) == _lib.E_INVALID
    eng.close()
    # a strip of a lattice is not a whole lattice
    strip = spgg_b200.Engine(full_params(dict(C1, L=L)), rows=16, row0=16, precision="fp32")
    with pytest.raises(ValueError, match="strip"):
        strip.cluster_sizes()
    strip.close()


@pytest.mark.parametrize("L", [100, 1024])
def test_dropin_writes_the_device_cluster_sizes(tmp_path, L):
    import spgg_b200
    from spgg_b200 import h5lite
    m = spgg_b200.SPGG(L=L, iterations=30, seed=3, **{k: v for k, v in C1.items() if k != "L"})
    fn = str(tmp_path / "run.h5")
    m.run(fn)
    with h5lite.open_file(fn, "r") as f:
        S = np.asarray(f["Sn_final"][()])
        sizes = np.asarray(f["cluster_sizes"][()])
    lab, n = label(S == 0)
    assert sizes.dtype == np.int64
    assert np.array_equal(sizes, np.bincount(lab.ravel(), minlength=n + 1)[1:].astype(np.int64))
