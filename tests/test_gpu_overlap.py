"""State overlaps on the device (include/spgg.h: spgg_snapshot / spgg_overlap, Engine.snapshot / Engine.overlap)
against the NumPy restatement of test_overlap_host.py on get_state's arrays: joint strategy counts, changed counts
and max |d| exactly, the fp64 sums within the stated bound (exactly for int8-stored R).  Every arithmetic mode and
TD rule, the state every kernel path leaves, adversarial uploaded states, batches and shifted comparisons, the slot
lifecycle, a pending re-run, chunked runs, the error codes, what a call leaves alone, and L = 16384 / 32768."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import C1, C2, full_params
from test_gpu_blocks import MODES, _random_state, _require, _stepped
from test_overlap_host import numpy_overlap, sum_bound

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GiB = 2 ** 30
FIELDS = ((), ("R",), ("Q",), ("R", "Q"))


def _engine(*a, **k):
    import spgg_b200
    return spgg_b200.Engine(*a, **k)


def _packed(o, i=None):
    """the dict of overlap (replica i of a batched one) -> counts (2, 2), changed (m,), diffs (m, 3)"""
    pick = (lambda v: np.asarray(v)) if i is None else (lambda v: np.asarray(v)[i])
    ch, d = [], []
    if "R_changed" in o:
        ch.append(np.atleast_1d(pick(o["R_changed"])))
        d.append(pick(o["R_diff"])[None])
    if "Q_changed" in o:
        ch.append(pick(o["Q_changed"]).reshape(-1))
        d.append(pick(o["Q_diff"]).reshape(-1, 3))
    return (pick(o["S"]), np.concatenate(ch) if ch else np.zeros(0, np.int64),
            np.concatenate(d) if d else np.zeros((0, 3)))


def _compare(got, want, n_sites, exact_r, fields, what=""):
    (gc, gch, gd), (c, ch, d) = got, want
    assert gc.dtype == np.int64 and np.array_equal(gc, c), (what, "S", gc, c)
    assert np.array_equal(gch, ch), (what, "changed", gch, ch)
    assert np.array_equal(gd[:, 0], d[:, 0]), (what, "max", gd[:, 0], d[:, 0])
    assert (np.abs(gd[:, 1:] - d[:, 1:]) <= sum_bound(n_sites, d)).all(), (what, "sums", gd, d)
    if exact_r and "R" in fields:
        assert np.array_equal(gd[0], d[0]), (what, "int8 R sums", gd[0], d[0])


def _check(eng, slot, then, rep=0, exact_r=None, what=""):
    """every field subset of the slot (all fields held) against the restatement of then -> get_state(now)"""
    reps = list(rep) if isinstance(rep, range) else [rep]
    thens = then if isinstance(rep, range) else [then]
    if exact_r is None:
        exact_r = bool(eng.status().r_is_int8)
    nows = [eng.get_state(r) for r in reps]
    for fields in FIELDS:
        o = eng.overlap(slot, replica=rep, fields=fields)
        for i, (t0, t1) in enumerate(zip(thens, nows)):
            got = _packed(o, i if isinstance(rep, range) else None)
            _compare(got, numpy_overlap(t0, t1, fields, eng.nq), eng.rows * eng.L, exact_r, fields, (what, i, fields))
    return o


def _assert_identity(o, nq, what=""):
    c, ch, d = _packed(o)
    assert c[0, 1] == 0 and c[1, 0] == 0, (what, c)
    assert ch.shape == (1 + nq,) and not ch.any() and not d.any(), (what, ch, d)


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("L", [33, 100])
def test_identity_and_uploaded_states(L, mode):
    p, prec, rst, rq = MODES[mode]
    eng = _engine(full_params(dict(p, L=L)), seeds=1, precision=prec, r_storage=rst)
    rs = np.random.RandomState(L)
    a = _random_state(L, eng.nq, rq, prec, 0.3, rs)
    b = _random_state(L, eng.nq, rq, prec, 0.6, rs)
    eng.set_state(*a)
    assert eng.snapshot(2) == 0
    o = eng.overlap(2)
    _assert_identity(o, eng.nq, mode)
    assert o["S"].sum() == L * L and o["S"][0, 0] == np.count_nonzero(a[0] == 0)
    eng.set_state(*b)
    _check(eng, 2, a, what=(mode, L))
    eng.close()


@pytest.mark.parametrize("algo,p,prec", [
    ("sarsa", C1, "fp32"), ("expected_sarsa", C2, "fp32"), ("double_qlearning", C2, "fp32"),
    ("double_qlearning", C1, "fp64"), ("qlearning", C2, "fp64"),
])
def test_identity_for_every_td_rule(algo, p, prec):
    L = 64
    eng = _engine(full_params(dict(p, L=L, algorithm=algo)), seeds=2, precision=prec)
    eng.init_random(3)
    eng.step(4)
    eng.snapshot(0)
    then = eng.get_state()
    _assert_identity(eng.overlap(0), eng.nq, algo)
    eng.step(9)
    _check(eng, 0, then, what=algo)
    eng.close()


@pytest.mark.parametrize("name,path,p,L,prec", [
    ("resident_cluster", "cluster", C1, 100, "fp32"),
    ("resident_grid", "grid", C2, 1000, "fp32"),
    ("fast_4096", "fast", C1, 4096, "fp32"),
    ("fast_partial_tile_column", "fast", C1, 288, "fp32"),
    ("lean_int8", "lean", C1, 97, "fp32"),
    ("lean_fp32_R", "lean", dict(C1, rep_gain_C=0.3, delta_R_D=0.7), 97, "fp32"),
    ("lean_fp64", "lean", C1, 97, "fp64"),
    ("sarsa", "k_step", dict(C1, algorithm="sarsa"), 131, "fp32"),
    ("expected_sarsa", "k_step", dict(C2, algorithm="expected_sarsa"), 131, "fp32"),
    ("double_q", "k_step", dict(C2, algorithm="double_qlearning"), 131, "fp32"),
    ("double_q_fp64", "k_step", dict(C2, algorithm="double_qlearning"), 131, "fp64"),
])
def test_after_stepping_on_every_path(monkeypatch, name, path, p, L, prec):
    eng = _stepped(monkeypatch, path, p, L, prec)
    assert eng.snapshot(1) == 37                      # the call completes the chunk itself
    then = eng.get_state()
    _assert_identity(eng.overlap(1), eng.nq, name)
    eng.step(23)
    o = eng.overlap(1)                                # before get_state: the call completes the chunk itself
    assert o["t0"] == 37 and o["t"] == 60
    _compare(_packed(o), numpy_overlap(then, eng.get_state(), ("R", "Q"), eng.nq), L * L,
             bool(eng.status().r_is_int8), ("R", "Q"), name)
    _check(eng, 1, then, what=name)
    eng.close()


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("L", [20, 97, 288])
def test_adversarial_states(L, mode):
    p, prec, rst, rq = MODES[mode]
    eng = _engine(full_params(dict(p, L=L)), seeds=1, precision=prec, r_storage=rst)
    rs = np.random.RandomState(L + 1)
    nq = eng.nq
    qs = (L, L) + (2,) * (2 if nq == 4 else 3)
    base = _random_state(L, nq, rq, prec, 0.5, rs)
    S0, R0, Q0 = base
    R0 = np.where(rs.rand(L, L) < 0.5, 0.0, R0)
    Q0 = np.where(rs.rand(*qs) < 0.5, 0.0, Q0)
    zeros = (S0, R0, Q0)
    signed = (S0, np.where(R0 == 0, -0.0, R0), np.where(Q0 == 0, -0.0, Q0))
    all_c = (np.zeros((L, L), np.uint8), np.zeros((L, L)), np.zeros(qs))
    all_d = (np.ones((L, L), np.uint8), R0, Q0)
    for a, b, what in ((zeros, signed, "+0 -> -0"), (signed, zeros, "-0 -> +0"), (all_c, all_d, "all C -> all D"),
                       (all_d, all_c, "all D -> all C"), (all_c, base, "all C -> mixed"), (base, all_d, "mixed -> all D")):
        eng.set_state(*a)
        eng.snapshot(0)
        eng.set_state(*b)
        o = _check(eng, 0, eng_state(a, prec), what=(mode, L, what))
        if what.startswith(("+0", "-0")):
            _assert_identity(o, nq, what)
    eng.close()


def eng_state(st, prec):
    """an uploaded state as get_state returns it (fp32 storage rounds; S as 0 / 1 bytes)"""
    S, R, Q = st
    S = (np.asarray(S) != 0).astype(np.uint8)
    if prec == "fp32":
        Q = np.asarray(Q, np.float32).astype(np.float64)
    return S, np.asarray(R, np.float64), np.asarray(Q, np.float64)


def test_batches_shifted_comparisons_and_damage_spreading():
    L = 64
    plist = [full_params(dict(C1, L=L)), full_params(dict(C1, L=L, rep_gain_C=0.5)),
             full_params(dict(C1, L=L, R_min=-3, R_max=3))]
    eng = _engine(plist, seeds=[1, 2, 3], precision="fp32")
    rs = np.random.RandomState(4)
    states = []
    for r, (lo, hi, q) in enumerate(((-10, 10, 1.0), (-2, 7, 0.5), (-3, 3, 1.0))):
        S = rs.randint(0, 2, (L, L)).astype(np.uint8)
        R = rs.randint(int(lo / q), int(hi / q) + 1, (L, L)) * q
        Q = rs.uniform(-0.1 * (r + 1), 0.1, (L, L, 2, 2)).astype(np.float32).astype(np.float64)
        eng.set_state(S, R, Q, replica=r)
        states.append((S, R, Q))
    eng.snapshot(0, replica=range(3))
    for r in range(3):
        eng.snapshot(1 + r, replica=r)
    assert eng.snapshot_info(0)["replica"] == range(3) and eng.snapshot_info(2)["replica"] == 1
    eng.snapshot(4, replica=0)
    # shifted: replica 0's snapshot against replicas 1 and 2 (quanta 1 against 0.5 and 1)
    for r in (1, 2):
        for fields in FIELDS:
            got = _packed(eng.overlap(4, replica=r, fields=fields))
            _compare(got, numpy_overlap(states[0], states[r], fields), L * L, True, fields, ("shifted", r))
    eng.init_random(5, replica=0)
    eng.init_random(6, replica=1)
    eng.init_random(7, replica=2)
    eng.step(25)
    o = _check(eng, 0, states, rep=range(3), what="batch")
    assert o["S"].shape == (3, 2, 2) and o["Q_diff"].shape == (3, 2, 2, 3)
    # a range call equals the single-replica calls, bit for bit
    for sub in (range(0, 3), range(1, 3), range(0, 2)):
        eng.snapshot(5, replica=sub)
        for i, r in enumerate(sub):
            eng.snapshot(1 + i, replica=r)
        eng.step(3)
        got = eng.overlap(5, replica=sub)
        for i, r in enumerate(sub):
            one = eng.overlap(1 + i, replica=r)
            for k in one:
                if k not in ("t0", "t"):
                    assert np.asarray(got[k])[i].tobytes() == np.asarray(one[k]).tobytes(), (sub, r, k)
    eng.close()
    # damage spreading: the same upload in two replicas of different seeds
    eng = _engine([full_params(dict(C1, L=L))] * 2, seeds=[11, 12], precision="fp32")
    st = states[0]
    eng.set_state(*st, replica=0)
    eng.set_state(*st, replica=1)
    eng.snapshot(0, replica=0)
    _assert_identity(eng.overlap(0, replica=1), 4, "t0")
    eng.step(15)
    eng.snapshot(0, replica=0)
    o = eng.overlap(0, replica=1)
    _compare(_packed(o), numpy_overlap(eng.get_state(0), eng.get_state(1)), L * L, True, ("R", "Q"), "damage")
    assert o["S"][0, 1] + o["S"][1, 0] > 0        # the seeds drove the replicas apart
    eng.close()


def test_slot_lifecycle():
    from spgg_b200 import _lib
    L = 48
    eng = _engine(full_params(dict(C1, L=L)), seeds=3, precision="fp32")
    eng.init_random(1)
    eng.step(10)
    assert eng.snapshot(3, fields=("R", "Q")) == 10
    then = eng.get_state()
    assert eng.snapshot_info(3) == {"iteration": 10, "replica": 0, "fields": ("R", "Q")}
    eng.step(5)
    _check(eng, 3, then, what="step")
    rs = np.random.RandomState(2)
    eng.set_state(*_random_state(L, 4, 1.0, "fp32", 0.5, rs))
    _check(eng, 3, then, what="set_state")
    eng.init_random(9)
    _check(eng, 3, then, what="init_random")
    eng.set_progress(500, [0.2])
    o = _check(eng, 3, then, what="set_progress")
    assert o["t0"] == 10 and o["t"] == 500
    assert eng.snapshot_info(3)["iteration"] == 10
    # re-snapshot replaces the slot, with other fields (another size) and the same again (reused memory)
    for fields in (("R",), ("R",), ()):
        assert eng.snapshot(3, fields=fields) == 500
        assert eng.snapshot_info(3)["fields"] == fields
        o = eng.overlap(3, fields=fields)
        assert not _packed(o)[1].any() and not _packed(o)[2].any() and o["S"][0, 1] == o["S"][1, 0] == 0
    with pytest.raises(ValueError, match="flags"):
        eng.overlap(3, fields=("Q",))                # not held by the slot
    eng.drop_snapshot(3)
    eng.drop_snapshot(3)                             # an empty slot: nothing to do
    cnt, chg, dif = np.full(4, -7, np.int64), np.full(5, -7, np.int64), np.full(15, -7.0)
    assert eng.lib.spgg_overlap(eng._h, 3, 0, 1, 0, cnt.ctypes.data, None, None) == _lib.E_STATE
    it = C.c_int64(-7)
    assert eng.lib.spgg_snapshot_info(eng._h, 3, C.byref(it), None, None, None) == _lib.E_STATE
    assert (cnt == -7).all() and it.value == -7
    with pytest.raises(RuntimeError, match="no snapshot"):
        eng.overlap(3)
    # every slot at once, then freed with the handle
    for s in range(8):
        eng.snapshot(s)
    eng.close()


_POISON_CHILD = r"""
import sys, numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {root!r} + "/tests")
import spgg_b200
from helpers import C1, full_params
from test_overlap_host import numpy_overlap, sum_bound
L = 256
eng = spgg_b200.Engine(full_params(dict(C1, L=L)), seeds=9, precision="fp32")
assert eng.describe().startswith("fast"), eng.describe()
eng.init_random(4)
eng.snapshot(0)
then = eng.get_state()
eng.step(120)
o = eng.overlap(0)                    # the first synchronising call: it completes the re-run itself
st = eng.status()
assert st.speculation_failures >= 1, st.speculation_failures
assert st.iteration == 120 and o["t"] == 120
c, ch, d = numpy_overlap(then, eng.get_state())
assert np.array_equal(o["S"], c) and o["R_changed"] == ch[0] and np.array_equal(o["Q_changed"].reshape(-1), ch[1:])
assert np.array_equal(o["R_diff"], d[0]) and np.array_equal(o["Q_diff"].reshape(4, 3)[:, 0], d[1:, 0])
assert (np.abs(o["Q_diff"].reshape(4, 3)[:, 1:] - d[1:, 1:]) <= sum_bound(L * L, d[1:])).all()
eng.step(30)
eng.snapshot(1)                       # a pending chunk again: the snapshot completes it
assert eng.snapshot_info(1)["iteration"] == 150
c, ch, d = numpy_overlap(eng.get_state(), eng.get_state())
o = eng.overlap(1)
assert np.array_equal(o["S"], c) and not o["Q_changed"].any() and not o["Q_diff"].any()
print("ok", st.speculation_failures)
"""


def test_fast_path_with_a_pending_rerun():
    env = dict(os.environ, SPGG_NO_RESIDENT="1", SPGG_SPEC_TEST_POISON="5")
    r = subprocess.run([sys.executable, "-c", _POISON_CHILD.format(root=ROOT)], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.parametrize("name,path,L,prec", [
    ("resident", "cluster", 100, "fp32"),
    ("fast", "fast", 256, "fp32"),
    ("lean", "lean", 97, "fp64"),
])
def test_chunked_runs_are_not_disturbed(monkeypatch, name, path, L, prec):
    from test_gpu_start_states import _engine as _path_engine
    p = full_params(dict(C1, L=L))
    outs, finals = [], []
    for chunks in ((200,), (50, 50, 50, 50)):
        eng = _path_engine(monkeypatch, path, p, seeds=8, precision=prec)
        eng.init_random(17)
        eng.snapshot(0)
        then = eng.get_state()
        rows = []
        for c in chunks:
            eng.step(c)
            if len(chunks) > 1:
                eng.snapshot(1)
                o = eng.overlap(0)
                _compare(_packed(o), numpy_overlap(then, eng.get_state()), L * L, prec == "fp32", ("R", "Q"), c)
                _assert_identity(eng.overlap(1), 4, c)
            rows.append(eng.stats()[1:])
        outs.append((eng.digest(),) + eng.get_state() + (np.vstack(rows),))
        finals.append(eng.overlap(0))
        eng.close()
    for a, b in zip(*outs):
        assert np.array_equal(np.asarray(a), np.asarray(b))
    # the same pair of states, reached in one chunk or in four: bit-identical sums
    for k in finals[0]:
        assert np.asarray(finals[0][k]).tobytes() == np.asarray(finals[1][k]).tobytes(), k


def test_errors_and_what_a_call_leaves_alone():
    from spgg_b200 import _lib
    L = 64
    eng = _engine([full_params(dict(C1, L=L))] * 2, seeds=[1, 2], precision="fp32")
    lib, h = eng.lib, eng._h
    eng.init_random(3, replica=0)
    eng.init_random(4, replica=1)
    eng.snapshot(0, replica=range(2), fields=("R",))
    eng.snapshot(1, replica=1)
    cnt = np.full(8, -7, np.int64)
    chg = np.full(10, -7, np.int64)
    dif = np.full(30, -7.0)
    E = _lib.E_INVALID
    bufs = (cnt.ctypes.data, chg.ctypes.data, dif.ctypes.data)
    for slot, rep0, n, flags in ((-1, 0, 2, 1), (8, 0, 2, 1), (0, 1, 2, 1), (0, -1, 2, 1), (0, 0, 0, 1), (0, 0, 3, 1),
                                 (0, 0, 1, 1), (1, 0, 2, 1), (0, 0, 2, 2), (0, 0, 2, 3), (0, 0, 2, 4), (0, 0, 2, -1)):
        assert lib.spgg_overlap(h, slot, rep0, n, flags, *bufs) == E, (slot, rep0, n, flags)
    for slot, rep0, n, flags in ((-1, 0, 1, 3), (8, 0, 1, 3), (0, 2, 1, 3), (0, -1, 1, 3), (0, 0, 0, 3), (0, 1, 2, 3),
                                 (0, 0, 1, 4), (0, 0, 1, -1)):
        assert lib.spgg_snapshot(h, slot, rep0, n, flags) == E, (slot, rep0, n, flags)
    assert lib.spgg_overlap(h, 0, 0, 2, 1, None, chg.ctypes.data, dif.ctypes.data) == E
    assert lib.spgg_overlap(h, 0, 0, 2, 1, cnt.ctypes.data, None, dif.ctypes.data) == E
    assert lib.spgg_overlap(h, 0, 0, 2, 1, cnt.ctypes.data, chg.ctypes.data, None) == E
    for slot in (-1, 8):
        assert lib.spgg_snapshot_info(h, slot, None, None, None, None) == E
        assert lib.spgg_snapshot_free(h, slot) == E
    assert lib.spgg_overlap(h, 5, 0, 1, 0, *bufs) == _lib.E_STATE
    assert lib.spgg_snapshot_info(h, 5, None, None, None, None) == _lib.E_STATE
    assert (cnt == -7).all() and (chg == -7).all() and (dif == -7.0).all()
    # the earlier slots survived the rejected calls
    assert eng.snapshot_info(0) == {"iteration": 0, "replica": range(2), "fields": ("R",)}
    assert lib.spgg_overlap(h, 0, 0, 2, 0, cnt.ctypes.data, None, None) == 0   # S only: null changed / diffs
    assert cnt.sum() == 2 * L * L and (chg == -7).all()
    with pytest.raises(ValueError, match="replicas"):
        _lib.check(lib.spgg_overlap(h, 1, 1, 2, 3, *bufs))
    # what a call leaves alone: the state, the iteration counter, the statistics rows, a cluster result, pair
    # counts, block fields and histograms
    eng.step(5)
    rows = eng.stats()
    dg = eng.digest()
    pc = eng.pair_counts(L // 2)
    bf = eng.block_fields(5)
    hs = eng.histograms(20, replica=range(2))
    n = C.c_int64()
    assert lib.spgg_clusters(h, 0, 0, 0, C.byref(n)) == 0
    it = eng.status().iteration
    eng.snapshot(2, replica=range(2))
    eng.overlap(2, replica=range(2))
    eng.overlap(0, replica=range(2), fields=("R",))
    eng.overlap(1, replica=0)
    sizes = np.zeros(n.value, np.int64)
    assert lib.spgg_cluster_sizes(h, sizes.ctypes.data, n.value) == 0
    assert eng.status().iteration == it and np.array_equal(eng.stats(), rows) and eng.digest() == dg
    assert np.array_equal(eng.pair_counts(L // 2), pc)
    bf2 = eng.block_fields(5)
    assert all(bf[k].tobytes() == bf2[k].tobytes() for k in bf)
    hs2 = eng.histograms(20, replica=range(2))
    assert all(np.asarray(hs[k]).tobytes() == np.asarray(hs2[k]).tobytes() for k in hs if k != "replica")
    eng.close()


def _f64(st):
    return st[0], np.asarray(st[1], np.float64), np.asarray(st[2], np.float64)


@pytest.mark.parametrize("L", [16384, 32768])
def test_large_lattices(L):
    """init_random(a), snapshot, init_random(b): the overlap against c_oracle.init_random of both seeds, restated
    1024 rows at a time (host memory stays bounded)"""
    from oracle import c_oracle
    _require(6 * GiB, L * L * 40 + 4 * GiB)
    eng = _engine(full_params(dict(C1, L=L)), seeds=1, precision="fp32")
    sa, sb = 7, 8
    eng.init_random(sa)
    eng.snapshot(0)
    eng.init_random(sb)
    got = [_packed(eng.overlap(0, fields=f)) for f in (("R", "Q"), ())]
    eng.close()
    c = np.zeros((2, 2), np.int64)
    ch = np.zeros(5, np.int64)
    d = np.zeros((5, 3))
    step = 1024
    for i0 in range(0, L, step):
        a = c_oracle.init_random(L, sa, 4, "fp32", row0=i0, rows=step)
        b = c_oracle.init_random(L, sb, 4, "fp32", row0=i0, rows=step)
        ci, chi, di = numpy_overlap(_f64(a), _f64(b))
        c += ci
        ch += chi
        d[:, 0] = np.maximum(d[:, 0], di[:, 0])
        d[:, 1:] += di[:, 1:]
    _compare(got[0], (c, ch, d), L * L, True, ("R", "Q"), L)
    assert np.array_equal(got[1][0], c) and c.sum() == L * L
    assert got[0][1][0] == 0 and not got[0][2][0].any()         # R = 0 in both states
