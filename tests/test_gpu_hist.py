"""Value distributions on the device (include/spgg.h: spgg_value_ranges / spgg_histograms, Engine.value_ranges /
Engine.histograms) against np.histogram on get_state's arrays (through the restatement of test_hist_host.py), with
exact equality of every count and extreme: every arithmetic mode and TD rule, the state every kernel path leaves,
adversarial uploaded states, batches, a pending re-run, chunked runs, the error codes, and L = 16384 / 32768."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import C1, C2, full_params
from test_gpu_blocks import MODES, _random_state, _require, _stepped
from test_hist_host import BINS, default_edges, numpy_histograms, numpy_value_ranges

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GiB = 2 ** 30
FIELDS = {1: ("R",), 2: ("Q",), 3: ("R", "Q")}


def _engine(*a, **k):
    import spgg_b200
    return spgg_b200.Engine(*a, **k)


def _algo(nq):
    return "double_qlearning" if nq == 8 else "qlearning"


def _packed(got, nq):
    """the dict of histograms -> counts (m, 2, bins) in the ABI's channel order"""
    parts = []
    if "R" in got:
        parts.append(got["R"][None])
    if "Q" in got:
        q = got["Q"]
        parts.append(np.moveaxis(q.reshape(2, nq, q.shape[-1]), 0, 1))
    return np.concatenate(parts) if parts else np.zeros((0, 2, 0), np.int64)


def _edges_of(got, nq):
    parts = []
    if "R" in got:
        parts.append(got["R_edges"][None])
    if "Q" in got:
        parts.append(got["Q_edges"].reshape(nq, -1))
    return np.concatenate(parts)


def _ranges_packed(got, nq):
    parts = []
    if "R" in got:
        parts.append(got["R"][None])
    if "Q" in got:
        parts.append(np.moveaxis(got["Q"].reshape(2, nq, 2), 0, 1))
    return np.concatenate(parts)


def _check(eng, state, bins, rep=0, ranges=None, what=""):
    """every field set at `bins` (default ranges unless given) and the value ranges, against the restatement"""
    S, R, Q = state
    nq = eng.nq
    mm = numpy_value_ranges(S, R, Q)
    got_mm = _ranges_packed(eng.value_ranges(rep), nq)
    assert (got_mm == mm).all(), (what, "ranges", got_mm, mm)     # == : the sign of a zero extreme is free
    for flags, fields in FIELDS.items():
        got = eng.histograms(bins, replica=rep, fields=fields, ranges=ranges)
        if ranges is None:
            edges = default_edges(S, R, Q, bins, flags)
        else:
            from spgg_b200.engine import hist_edges
            edges = np.stack(([hist_edges(*ranges["R"], bins)] if flags & 1 else [])
                             + ([hist_edges(*ranges["Q"], bins)] * nq if flags & 2 else []))
        assert np.array_equal(_edges_of(got, nq), edges), (what, flags)
        counts, pol = numpy_histograms(S, R, Q, edges, _algo(nq), flags)
        assert np.array_equal(_packed(got, nq), counts), (what, bins, flags)
        assert np.array_equal(got["policy"], pol), (what, "policy")
    got = eng.histograms(bins, replica=rep, fields=())
    assert set(got) == {"replica", "policy"} and np.array_equal(got["policy"], pol), what


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("L", [5, 33, 100, 1000])
def test_uploaded_random_states(L, mode):
    p, prec, rst, rq = MODES[mode]
    eng = _engine(full_params(dict(p, L=L)), seeds=1, precision=prec, r_storage=rst)
    rs = np.random.RandomState(L)
    for p_coop in (0.1, 0.5):
        st = _random_state(L, eng.nq, rq, prec, p_coop, rs)
        eng.set_state(*st)
        for bins in BINS:
            _check(eng, st, bins, what=(mode, L, p_coop))
    eng.close()


def _on_edges(L, nq, rq, prec, rs):
    """R on the integer edges of (-10, 10) / 20 bins (and on the quantum grid), Q on the multiples of 1/8 that are
    the edges of (-0.5, 0.5) / 8 bins, both ends included"""
    S = rs.randint(0, 2, (L, L)).astype(np.uint8)
    step = 1.0 if rq is None else rq
    R = rs.randint(int(-10 / step), int(10 / step) + 1, (L, L)) * step
    Q = rs.randint(-4, 5, (L, L) + (2,) * (2 if nq == 4 else 3)) / 8.0
    Q[0, 0] = -0.0
    return S, R, Q


@pytest.mark.parametrize("mode", list(MODES))
def test_adversarial_states(mode):
    p, prec, rst, rq = MODES[mode]
    L = 100
    eng = _engine(full_params(dict(p, L=L)), seeds=1, precision=prec, r_storage=rst)
    rs = np.random.RandomState(7)
    st = _on_edges(L, eng.nq, rq, prec, rs)
    eng.set_state(*st)
    for bins, ranges in ((20, {"R": (-10, 10), "Q": (-0.5, 0.5)}), (8, {"R": (-10, 10), "Q": (-0.5, 0.5)}),
                         (7, {"R": (-3, 2), "Q": (-0.25, 0.0)}), (1024, None)):
        _check(eng, st, bins, ranges=ranges, what=(mode, "edges", bins))
    qs = st[2].shape
    Q = rs.uniform(-0.01, 0.01, qs)
    if prec == "fp32":
        Q = Q.astype(np.float32).astype(np.float64)
    for name, S in (("all C", np.zeros((L, L), np.uint8)), ("all D", np.ones((L, L), np.uint8)),
                    ("mixed", rs.randint(0, 2, (L, L)).astype(np.uint8))):
        st = (S, np.zeros((L, L)), Q)      # uniform R = 0: every site in one bin, both ends of the range
        eng.set_state(*st)
        for bins in (1, 20, 1024):
            _check(eng, st, bins, what=(mode, name, bins))
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
    got = eng.histograms(20)                          # before get_state: the call completes the chunk itself
    st = eng.get_state()
    counts, pol = numpy_histograms(*st, default_edges(*st, 20), _algo(eng.nq))
    assert np.array_equal(_packed(got, eng.nq), counts) and np.array_equal(got["policy"], pol), name
    for bins in (1, 7, 64, 1024):
        _check(eng, st, bins, what=name)
    eng.close()


def test_batches_and_sub_ranges():
    """Replicas of different R quanta and spreads in one call; every sub-range equals the single-replica calls."""
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
    for sub in (range(0, 3), range(1, 3), range(0, 2), range(2, 3)):
        for bins in (7, 20):
            got = eng.histograms(bins, replica=sub)
            mm = eng.value_ranges(replica=sub)
            assert got["replica"] == sub and got["R"].shape == (len(sub), 2, bins)
            for i, r in enumerate(sub):
                one = eng.histograms(bins, replica=r)
                for k in one:
                    if k != "replica":
                        assert np.array_equal(got[k][i], one[k]), (sub, r, k)
                assert np.array_equal(mm["R"][i], eng.value_ranges(r)["R"])
                st = states[r]
                counts, pol = numpy_histograms(*st, default_edges(*st, bins), "qlearning")
                assert np.array_equal(_packed({k: got[k][i] for k in ("R", "Q")}, 4), counts), (sub, r)
                assert np.array_equal(got["policy"][i], pol)
    # the batch after a run, with different dynamics per replica
    eng.init_random(5, replica=0)
    eng.init_random(6, replica=1)
    eng.init_random(7, replica=2)
    eng.step(25)
    got = eng.histograms(20, replica=range(3))
    for r in range(3):
        st = eng.get_state(r)
        counts, pol = numpy_histograms(*st, default_edges(*st, 20), "qlearning")
        assert np.array_equal(_packed({k: got[k][r] for k in ("R", "Q")}, 4), counts), r
        assert np.array_equal(got["policy"][r], pol)
    eng.close()


_POISON_CHILD = r"""
import sys, numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {root!r} + "/tests")
import spgg_b200
from helpers import C1, full_params
from test_hist_host import default_edges, numpy_histograms
L = 256
eng = spgg_b200.Engine(full_params(dict(C1, L=L)), seeds=9, precision="fp32")
assert eng.describe().startswith("fast"), eng.describe()
eng.init_random(4)
eng.step(120)
got = eng.histograms(20)               # the first synchronising call: it completes the re-run itself
st = eng.status()
assert st.speculation_failures >= 1, st.speculation_failures
assert st.iteration == 120
S, R, Q = eng.get_state()
c, pol = numpy_histograms(S, R, Q, default_edges(S, R, Q, 20), "qlearning")
assert np.array_equal(got["R"], c[0]) and np.array_equal(got["policy"], pol)
assert np.array_equal(np.moveaxis(got["Q"].reshape(2, 4, 20), 0, 1), c[1:])
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
    outs = []
    for chunks in ((200,), (50, 50, 50, 50)):
        eng = _path_engine(monkeypatch, path, p, seeds=8, precision=prec)
        eng.init_random(17)
        rows = []
        for c in chunks:
            eng.step(c)
            if len(chunks) > 1:
                eng.histograms(20)
                eng.value_ranges()
                got = eng.histograms(7, fields=("R",), ranges={"R": (-5, 5)}, policy=False)
                st = eng.get_state()
                want, _ = numpy_histograms(*st, np.linspace(-5.0, 5.0, 8)[None], "qlearning", 1)
                assert np.array_equal(got["R"], want[0])
            rows.append(eng.stats()[1:])
        outs.append((eng.digest(),) + eng.get_state() + (np.vstack(rows),))
        eng.close()
    for a, b in zip(*outs):
        assert np.array_equal(np.asarray(a), np.asarray(b))


def test_errors_and_what_a_call_leaves_alone():
    from spgg_b200 import _lib
    L = 64
    eng = _engine([full_params(dict(C1, L=L))] * 2, seeds=[1, 2], precision="fp32")
    lib, h = eng.lib, eng._h
    nb = 8
    e = np.tile(np.linspace(-1.0, 1.0, nb + 1), 2 * 5)
    cnt = np.full(2 * 5 * 2 * 1024, -7, np.int64)
    pol = np.full(8, -7, np.int64)
    mm = np.full(2 * 5 * 4, -7.0)
    E = _lib.E_INVALID
    for rep0, n, flags in ((2, 1, 3), (-1, 1, 3), (0, 0, 3), (1, 2, 3), (0, 3, 3), (0, 1, 4), (0, 1, -1)):
        assert lib.spgg_histograms(h, rep0, n, flags, nb, e.ctypes.data, cnt.ctypes.data, pol.ctypes.data) == E
        assert lib.spgg_value_ranges(h, rep0, n, flags, mm.ctypes.data) == E
    for bins in (0, -1, 1025):
        big = np.tile(np.linspace(-1.0, 1.0, max(bins, 1) + 1), 10)
        assert lib.spgg_histograms(h, 0, 1, 3, bins, big.ctypes.data, cnt.ctypes.data, None) == E
    assert lib.spgg_histograms(h, 0, 1, 3, nb, None, cnt.ctypes.data, None) == E
    assert lib.spgg_histograms(h, 0, 1, 3, nb, e.ctypes.data, None, None) == E
    assert lib.spgg_value_ranges(h, 0, 1, 3, None) == E
    for bad in ((0, np.nan), (0, np.inf), (3, -np.inf), (nb, 1.0 - 3.0), (4, 2.0)):   # (index, value)
        eb = e.copy()
        eb[9 * (nb + 1) + bad[0]] = bad[1]     # the last edge row: non-finite or decreasing
        assert lib.spgg_histograms(h, 0, 2, 3, nb, eb.ctypes.data, cnt.ctypes.data, None) == E, bad
    flat = np.zeros(nb + 1)
    assert lib.spgg_histograms(h, 0, 1, 1, nb, flat.ctypes.data, cnt.ctypes.data, None) == E   # e[0] == e[nb]
    assert (cnt == -7).all() and (pol == -7).all() and (mm == -7.0).all()
    assert lib.spgg_histograms(h, 0, 1, 0, nb, None, None, None) == 0            # nothing asked for
    assert lib.spgg_histograms(h, 0, 2, 0, nb, None, None, pol.ctypes.data) == 0   # policy only
    assert (pol >= 0).all()
    with pytest.raises(ValueError, match="replicas"):
        _lib.check(lib.spgg_value_ranges(h, 1, 2, 3, mm.ctypes.data))
    # what a call leaves alone: the state, the iteration counter, the statistics rows, a cluster result,
    # pair counts and block fields
    eng.init_random(3, replica=0)
    eng.init_random(4, replica=1)
    eng.step(5)
    rows = eng.stats()
    dg = eng.digest()
    pc = eng.pair_counts(L // 2)
    bf = eng.block_fields(5)
    n = C.c_int64()
    assert lib.spgg_clusters(h, 0, 0, 0, C.byref(n)) == 0
    it = eng.status().iteration
    eng.histograms(1024, replica=range(2))
    eng.value_ranges(range(2))
    sizes = np.zeros(n.value, np.int64)
    assert lib.spgg_cluster_sizes(h, sizes.ctypes.data, n.value) == 0
    assert eng.status().iteration == it and np.array_equal(eng.stats(), rows) and eng.digest() == dg
    assert np.array_equal(eng.pair_counts(L // 2), pc)
    bf2 = eng.block_fields(5)
    assert all(bf[k].tobytes() == bf2[k].tobytes() for k in bf)
    eng.close()


@pytest.mark.parametrize("mode", ["int8_unit1", "int8_unit_half", "fp32_R", "fp64"])
def test_r_channel_equals_r_histogram(mode):
    p, prec, rst, rq = MODES[mode]
    L = 100
    eng = _engine(full_params(dict(p, L=L)), seeds=1, precision=prec, r_storage=rst)
    eng.init_random(2)
    eng.step(30)
    for bins in (1, 7, 20, 64):
        for lo, hi in ((-10.0, 10.0), (-3.5, 2.25), (0.0, 0.5)):
            want, we = eng.r_histogram(bins, lo, hi)
            got = eng.histograms(bins, fields=("R",), ranges={"R": (lo, hi)}, policy=False)
            assert np.array_equal(got["R"][0], want) and np.array_equal(got["R_edges"], we), (mode, bins, lo)
    eng.close()


@pytest.mark.parametrize("L", [16384, 32768])
def test_large_lattices(L):
    """After init_random (R = 0 everywhere: the contended case): counts sum to L^2 in every channel and class,
    and the R and Q histograms equal those of the oracle's init_random, streamed 1024 rows at a time."""
    from oracle import c_oracle
    _require(6 * GiB, L * L * 20 + 2 * GiB)
    eng = _engine(full_params(dict(C1, L=L)), seeds=1, precision="fp32")
    seed = 7
    eng.init_random(seed)
    bins = 64
    got = eng.histograms(bins, ranges={"R": (-10, 10), "Q": (-0.01, 0.01)})
    mm = eng.value_ranges()
    dflt = eng.histograms(20)
    eng.close()
    counts = _packed(got, 4)
    assert (counts[:, 0].sum(-1) == L * L).all()
    n_c = counts[0, 1].sum()
    assert (counts[:, 1].sum(-1) == n_c).all()
    assert got["policy"][0].max() <= L * L
    edges = _edges_of(got, 4)
    want = np.zeros_like(counts)
    pol = np.zeros((2, 2), np.int64)
    lo = np.full((5, 2), np.inf)
    hi = np.full((5, 2), -np.inf)
    for i0 in range(0, L, 1024):
        So, Ro, Qo = c_oracle.init_random(L, seed, 4, "fp32", row0=i0, rows=1024)
        st = (So, np.asarray(Ro, np.float64), np.asarray(Qo, np.float64))
        c, p = numpy_histograms(*st, edges, "qlearning")
        want += c
        pol += p
        m = numpy_value_ranges(*st)
        lo, hi = np.minimum(lo, m[..., 0]), np.maximum(hi, m[..., 1])
    assert np.array_equal(counts, want) and np.array_equal(got["policy"], pol)
    gm = _ranges_packed(mm, 4)
    assert (gm[..., 0] == lo).all() and (gm[..., 1] == hi).all()
    # the default range of R = 0 everywhere is (-0.5, 0.5): one middle bin holds every site
    assert np.array_equal(dflt["R_edges"], np.linspace(-0.5, 0.5, 21))
    assert dflt["R"][0, 10] == L * L and dflt["R"][0].sum() == L * L
