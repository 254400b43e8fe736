"""Strategy pair counts on the device (include/spgg.h: spgg_pair_counts, Engine.pair_counts): exact equality
with the NumPy restatement of test_pairs_host.py, and 2 (n_C - n_CC(d)) == n_diff(d) at every offset, on
uploaded lattices, hand-made patterns and the state every kernel path leaves behind; counting never
disturbs a run."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import C1, C2, full_params
from test_pairs_host import numpy_pair_counts

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _engine(*a, **k):
    import spgg_b200
    return spgg_b200.Engine(*a, **k)


def _set(eng, S, replica=0):
    L = eng.L
    q = np.zeros((L, L) + ((2, 2) if eng.nq == 4 else (2, 2, 2)))
    eng.set_state(S, np.zeros((L, L)), q, replica=replica)


def _offsets(L):
    """max_d values of the random-lattice test: around one word of columns, and L/2"""
    return sorted({d for d in (1, 31, 32, 33, L // 2) if 1 <= d <= L // 2})


def _sampled(L):
    """offsets compared with NumPy on lattices where all of them would take minutes on the host"""
    return sorted({d for d in (1, 2, 31, 32, 33, 1000, L // 2 - 1, L // 2) if 1 <= d <= L // 2})


def _check(got, S, want=None, what=""):
    """got == want wherever want is filled in (want >= 0), and the torus invariant at every offset"""
    max_d = got.shape[1] - 1
    assert got.dtype == np.int64 and got.shape == (2, max_d + 1, 2), what
    nC = int(np.count_nonzero(np.asarray(S) == 0))
    assert (got[:, 0] == [nC, 0]).all(), what
    assert np.array_equal(2 * (nC - got[:, :, 0]), got[:, :, 1]), what
    if want is None:
        want = numpy_pair_counts(S, max_d)
    want = want[:, :max_d + 1]
    sel = want >= 0
    assert np.array_equal(got[sel], want[sel]), (what, np.argwhere((got != want) & sel)[:8])


@pytest.mark.parametrize("L", [4, 5, 31, 32, 33, 64, 100, 127, 128, 200, 1000, 1024, 4000, 4096])
def test_random_lattices_equal_numpy(L):
    eng = _engine(full_params(dict(C1, L=L)), seeds=1, precision="fp32")
    rs = np.random.RandomState(L)
    for p in (0.1, 0.5, 0.9):
        S = (rs.rand(L, L) >= p).astype(np.uint8)      # cooperator (S == 0) with probability p
        _set(eng, S)
        want = numpy_pair_counts(S, L // 2, ds=None if L <= 1024 else _sampled(L))
        for md in _offsets(L):
            _check(eng.pair_counts(md), S, want, what=(L, p, md))
    eng.close()


def _patterns(L):
    ii, jj = np.indices((L, L))
    yield "all C", np.zeros((L, L), np.uint8)
    yield "all D", np.ones((L, L), np.uint8)
    yield "checkerboard", ((ii + jj) % 2).astype(np.uint8)
    for w in (1, 31, 32, 33):
        yield f"vertical stripes {w}", ((jj // w) % 2).astype(np.uint8)
        yield f"horizontal stripes {w}", ((ii // w) % 2).astype(np.uint8)
    yield "last column C", (jj != L - 1).astype(np.uint8)


@pytest.mark.parametrize("L", [4, 33, 64, 100, 257, 1000])
def test_patterns(L):
    eng = _engine(full_params(dict(C1, L=L)), seeds=1, precision="fp32")
    for name, S in _patterns(L):
        _set(eng, S)
        _check(eng.pair_counts(L // 2), S, what=name)
    # the counts the patterns are built for
    N = L * L
    _set(eng, np.zeros((L, L), np.uint8))
    got = eng.pair_counts(L // 2)
    assert (got[:, :, 0] == N).all() and (got[:, :, 1] == 0).all()
    _set(eng, np.ones((L, L), np.uint8))
    assert not eng.pair_counts(L // 2).any()
    if L % 2 == 0:
        ii, jj = np.indices((L, L))
        _set(eng, ((ii + jj) % 2).astype(np.uint8))
        got = eng.pair_counts(L // 2)
        d = np.arange(L // 2 + 1)
        assert (got[:, :, 0] == np.where(d % 2, 0, N // 2)).all() and (got[:, :, 1] == np.where(d % 2, N, 0)).all()
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
        d = eng.describe()
        assert (d.startswith(want[0]) and want[1] in d), d
    eng.init_random(11)
    eng.step(n)
    got = eng.pair_counts(L // 2)                     # before get_state: counting completes the chunk itself
    S = eng.get_state(want_q=False)[0]
    _check(got, S, numpy_pair_counts(S, L // 2, ds=None if L <= 1024 else _sampled(L)))
    eng.close()


@pytest.mark.parametrize("name,p,L,env,prec,want", [
    ("resident_cluster", C1, 100, None, "fp32", ("resident: cluster", "DSMEM")),
    ("resident_grid", C2, 1000, None, "fp32", ("resident: cooperative grid", "L2")),
    ("fast_4096", C1, 4096, None, "fp32", ("fast:", "TMA")),
    ("fast_256", C1, 256, {"SPGG_NO_RESIDENT": "1"}, "fp32", ("fast:", "TMA")),
    ("lean_fp64", C1, 97, None, "fp64", ("general:", "+ k_step_lean)")),
    ("sarsa", dict(C1, algorithm="sarsa"), 131, None, "fp32", ("general:", "+ k_step)")),
    ("double_q", dict(C2, algorithm="double_qlearning"), 131, None, "fp32", ("general:", "+ k_step)")),
])
def test_after_stepping_on_every_path(monkeypatch, name, p, L, env, prec, want):
    _after_steps(p, L, 37, env, prec, monkeypatch, want)


_POISON_CHILD = r"""
import sys, numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {root!r} + "/tests")
import spgg_b200
from helpers import C1, full_params
from test_pairs_host import numpy_pair_counts
L = 256
eng = spgg_b200.Engine(full_params(dict(C1, L=L)), seeds=9, precision="fp32")
assert eng.describe().startswith("fast"), eng.describe()
eng.init_random(4)
eng.step(120)
got = eng.pair_counts(L // 2)         # the first synchronising call: it completes the re-run itself
st = eng.status()
assert st.speculation_failures >= 1, st.speculation_failures
assert st.iteration == 120
S = eng.get_state(want_q=False)[0]
assert np.array_equal(got, numpy_pair_counts(S, L // 2))
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
        got = [eng.pair_counts(L // 2, replica=r) for r in range(3)]
        assert eng.status(0).stopped_at == 1 and eng.status(1).iteration == 11
        assert not got[0][:, 1:, 0].any()   # the stopped replica is all D
        for r in range(3):
            _check(got[r], eng.get_state(r, want_q=False)[0], what=(no_res, r))
        eng.close()
    L = 131
    eng = _engine([full_params(dict(C1, L=L, r=3.0 + 0.5 * i)) for i in range(3)], seeds=[5, 6, 7], precision="fp32")
    for r in range(3):
        eng.init_random(20 + r, replica=r)
    eng.step(9)
    for r in range(3):
        _check(eng.pair_counts(L // 2, replica=r), eng.get_state(r, want_q=False)[0], what=r)
    eng.close()


@pytest.mark.parametrize("name,L,env,prec", [
    ("resident", 100, None, "fp32"),
    ("fast", 256, {"SPGG_NO_RESIDENT": "1"}, "fp32"),
    ("lean", 97, None, "fp64"),
])
def test_counting_does_not_disturb_the_run(monkeypatch, name, L, env, prec):
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
            if len(chunks) > 1:
                eng.pair_counts(L // 2)
                eng.pair_counts(1)
            rows.append(eng.stats()[1:])
        outs.append((eng.digest(),) + eng.get_state() + (np.vstack(rows),))
        eng.close()
    for a, b in zip(*outs):
        assert np.array_equal(np.asarray(a), np.asarray(b))


def test_errors_and_what_counting_leaves_alone():
    import spgg_b200
    from spgg_b200 import _lib
    L = 64
    eng = _engine(full_params(dict(C1, L=L)), seeds=1, precision="fp32")
    lib, h = eng.lib, eng._h
    out = np.full(4 * (L // 2 + 2), -7, np.int64)
    for rep, md in ((1, 1), (-1, 1), (0, 0), (0, -3), (0, L // 2 + 1)):
        assert lib.spgg_pair_counts(h, rep, md, out.ctypes.data) == _lib.E_INVALID, (rep, md)
    assert lib.spgg_pair_counts(h, 0, 1, None) == _lib.E_INVALID
    assert (out == -7).all()
    with pytest.raises(ValueError, match="max_d"):
        eng.pair_counts(L // 2 + 1)
    # a cluster-labelling result, the iteration counter and the statistics rows survive a count
    eng.init_random(3)
    eng.step(5)
    rows = eng.stats()
    n = C.c_int64()
    assert lib.spgg_clusters(h, 0, 0, 0, C.byref(n)) == 0
    it = eng.status().iteration
    assert lib.spgg_pair_counts(h, 0, L // 2, out.ctypes.data) == 0
    sizes = np.zeros(n.value, np.int64)
    assert lib.spgg_cluster_sizes(h, sizes.ctypes.data, n.value) == 0
    assert eng.status().iteration == it and np.array_equal(eng.stats(), rows)
    eng.close()
    # a strip of a lattice is not a whole lattice
    strip = spgg_b200.Engine(full_params(dict(C1, L=L)), rows=16, row0=16, precision="fp32")
    assert strip.lib.spgg_pair_counts(strip._h, 0, 1, out.ctypes.data) == _lib.E_UNSUPPORTED
    with pytest.raises(ValueError, match="strip"):
        strip.pair_counts(1)
    strip.close()
    # strip pair counts serve single-replica handles
    batch = spgg_b200.Engine([full_params(dict(C1, L=L))] * 2, rows=32, row0=0, precision="fp32")
    assert batch.lib.spgg_strip_pair_record_bytes(batch._h, 4, 4) == _lib.E_UNSUPPORTED
    assert batch.lib.spgg_strip_pair_record(batch._h, 4, 4, out.ctypes.data) == _lib.E_UNSUPPORTED
    assert batch.lib.spgg_strip_pair_counts(batch._h, 1, 0, out.ctypes.data, 4, 4, out.ctypes.data) == _lib.E_UNSUPPORTED
    batch.close()


@pytest.mark.parametrize("L", [16384, 32768])
def test_large_lattices_from_init_random(L):
    """S read back alone (no R, no Q: 1 GiB at L = 32768), compared with NumPy at sampled offsets."""
    eng = _engine(full_params(dict(C1, L=L)), seeds=1, precision="fp32")
    eng.init_random(7)
    got = eng.pair_counts(L // 2)
    S = np.empty(L * L, np.uint8)
    assert eng.lib.spgg_get_state(eng._h, 0, S.ctypes.data, None, None) == 0
    eng.close()
    S = S.reshape(L, L)
    _check(got, S, numpy_pair_counts(S, L // 2, ds=[1, 2, 31, 32, 33, 1000, L // 2]), what=L)


def test_strip_records_that_claim_more_rows_than_max_rows_are_refused():
    """Three strip handles of L = 100 (34 / 33 / 33 rows) in one process.  With max_d = 34 the 33-row strips
    pass max_rows = 33; a hand-edited record of the 34-row strip that claims its 34 rows within max_rows = 33
    would make the tail copy read past the record, so the counts refuse it.  Unedited records count."""
    import torch
    import spgg_b200
    from spgg_b200 import _lib
    L, md, mr = 100, 34, 33
    p = full_params(dict(C1, L=L))
    hs = [spgg_b200.Engine(p, rows=r, row0=r0, precision="fp32") for r0, r in ((0, 34), (34, 33), (67, 33))]
    S = (np.random.RandomState(3).rand(L, L) >= 0.5).astype(np.uint8)
    for e, r0 in zip(hs, (0, 34, 67)):
        e.set_state(S[r0:r0 + e.rows], np.zeros((e.rows, L)), np.zeros((e.rows, L, 2, 2)))
    lib = hs[0].lib
    nb = int(lib.spgg_strip_pair_record_bytes(hs[1]._h, md, mr))
    assert lib.spgg_strip_pair_record_bytes(hs[0]._h, md, mr) == _lib.E_INVALID   # 34 rows do not fit in 33
    rec = torch.zeros(3 * nb, dtype=torch.uint8, device="cuda")
    assert lib.spgg_strip_pair_record(hs[0]._h, mr, mr, rec.data_ptr()) == 0       # max_d 33: 33 rows
    for k in (1, 2):
        assert lib.spgg_strip_pair_record(hs[k]._h, md, mr, rec[k * nb:].data_ptr()) == 0
    torch.cuda.synchronize()
    out = np.zeros((2, md + 1, 2), np.int64)
    hdr = rec.view(torch.int32)
    hdr[4], hdr[6] = md, 34                                  # record 0 now claims max_d 34 and its 34 rows
    assert lib.spgg_strip_pair_counts(hs[1]._h, 3, 1, rec.data_ptr(), md, mr, out.ctypes.data) == _lib.E_INVALID
    assert b"max_rows" in lib.spgg_last_error()
    # the same lattice with max_rows = 34 everywhere counts as one handle does
    nb = int(lib.spgg_strip_pair_record_bytes(hs[0]._h, md, 34))
    rec = torch.zeros(3 * nb, dtype=torch.uint8, device="cuda")
    for k in range(3):
        assert lib.spgg_strip_pair_record(hs[k]._h, md, 34, rec[k * nb:].data_ptr()) == 0
    total = np.zeros_like(out)
    for k in range(3):
        assert lib.spgg_strip_pair_counts(hs[k]._h, 3, k, rec.data_ptr(), md, 34, out.ctypes.data) == 0
        total += out
    for e in hs:
        e.close()
    _check(total, S, what="three handles")
