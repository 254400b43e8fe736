"""Block fields on the device (include/spgg.h: spgg_block_fields, Engine.block_fields) against the NumPy
restatement of test_blocks_host.py on get_state: counts and int8-stored R exactly, fp32 / fp64 sums within the
stated bound (n-1) 2^-53 sum |x| per side; on uploaded lattices, the state every kernel path leaves behind,
batches, and the L = 16384 / 32768 lattices.  A call never disturbs a run, and the same state gives the same
bits."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from helpers import C1, C2, full_params
from test_blocks_host import numpy_block_fields, sum_bound
from test_gpu_start_states import FRAC_R, _engine as _path_engine

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GiB = 2 ** 30
FLAGS = {0: (), 1: ("R",), 2: ("Q",), 3: ("R", "Q")}


def _engine(*a, **k):
    import spgg_b200
    return spgg_b200.Engine(*a, **k)


def _b_values(L):
    return sorted({b for b in (1, 2, 3, 7, 32, 33, 100, L // 2 + 1, L) if 1 <= b <= L and (-(-L // b)) ** 2 <= 1 << 24})


def _packed(got, nq):
    """the dict of block_fields -> counts (nI, B, 2) and sums (nI, B, 2, m) in the ABI's channel order"""
    counts = np.stack([got["n"], got["n_C"]], -1)
    parts = []
    if "R" in got:
        parts.append(got["R"][..., None])
    if "Q" in got:
        parts.append(got["Q"].reshape(got["Q"].shape[:3] + (nq,)))
    sums = np.concatenate(parts, -1) if parts else np.zeros(counts.shape + (0,))
    return counts, sums


def _compare(got, want, nq, flags, exact_r, what=""):
    """got: block_fields' dict; want: numpy_block_fields(..., flags=3) of the same state"""
    c, s, a = want
    gc, gs = _packed(got, nq)
    assert gc.dtype == np.int64 and np.array_equal(gc, c), (what, "counts")
    sel = ([0] if flags & 1 else []) + (list(range(1, 1 + nq)) if flags & 2 else [])
    s, a = s[..., sel], a[..., sel]
    assert gs.shape == s.shape, (what, gs.shape, s.shape)
    if flags & 1 and exact_r:
        assert np.array_equal(gs[..., 0], s[..., 0]), (what, "int8 R sums")
    err = np.abs(gs - s)
    bound = sum_bound(c, a)
    assert (err <= bound).all(), (what, float(err.max()), np.argwhere(err > bound)[:4])


def _check_all(eng, b, exact_r, rep=0, what=""):
    """every flag set at block side b against the restatement of get_state"""
    S, R, Q = eng.get_state(rep)
    want = numpy_block_fields(S, R, Q, b, 3, eng.row0, eng.L)
    for flags, fields in FLAGS.items():
        _compare(eng.block_fields(b, replica=rep, fields=fields), want, eng.nq, flags, exact_r, (what, b, flags))


# storage mode -> (params, precision, r_storage, R values in int8 units of rq (None: float R))
MODES = {
    "int8_unit1": (C1, "fp32", "auto", 1.0),
    "int8_unit_half": (dict(C1, rep_gain_C=0.5), "fp32", "auto", 0.5),
    "fp32_R": (C1, "fp32", "fp32", None),
    "fp64": (C1, "fp64", "auto", None),
    "double_q": (dict(C2, algorithm="double_qlearning"), "fp32", "auto", 1.0),
}


def _random_state(L, nq, rq, precision, p_coop, rs):
    S = (rs.rand(L, L) >= p_coop).astype(np.uint8)
    if rq is None:
        R = rs.uniform(-10, 10, (L, L))
    else:
        R = rs.randint(int(-10 / rq), int(10 / rq) + 1, (L, L)) * rq
    Q = rs.uniform(-0.5, 0.5, (L, L) + (2,) * (2 if nq == 4 else 3))
    if precision == "fp32":
        R, Q = R.astype(np.float32).astype(np.float64), Q.astype(np.float32).astype(np.float64)
    return S, R, Q


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("L", [4, 5, 31, 33, 100, 128, 1000, 4000, 4096])
def test_uploaded_random_states(L, mode):
    p, prec, rst, rq = MODES[mode]
    eng = _engine(full_params(dict(p, L=L)), seeds=1, precision=prec, r_storage=rst)
    rs = np.random.RandomState(L)
    # the large lattices take all three densities in one mode, one density in the others
    dens = (0.1, 0.5, 0.9) if L < 4000 or mode == "int8_unit_half" else (0.5,)
    for p_coop in dens:
        S, R, Q = _random_state(L, eng.nq, rq, prec, p_coop, rs)
        eng.set_state(S, R, Q)
        for b in _b_values(L):
            _check_all(eng, b, rq is not None, what=(mode, p_coop))
    eng.close()


def _stepped(monkeypatch, path, p, L, prec="fp32", n=37):
    eng = _path_engine(monkeypatch, path, full_params(dict(p, L=L)), seeds=3, precision=prec)
    eng.init_random(11)
    eng.step(n)
    return eng


@pytest.mark.parametrize("name,path,p,L,prec", [
    ("resident_cluster", "cluster", C1, 100, "fp32"),
    ("resident_grid", "grid", C2, 1000, "fp32"),
    ("fast_4096", "fast", C1, 4096, "fp32"),
    ("fast_partial_tile_column", "fast", C1, 288, "fp32"),
    ("lean_int8", "lean", C1, 97, "fp32"),
    ("lean_fp32_R", "lean", FRAC_R, 97, "fp32"),
    ("lean_fp64", "lean", C1, 97, "fp64"),
    ("sarsa", "k_step", dict(C1, algorithm="sarsa"), 131, "fp32"),
    ("expected_sarsa", "k_step", dict(C2, algorithm="expected_sarsa"), 131, "fp32"),
    ("double_q", "k_step", dict(C2, algorithm="double_qlearning"), 131, "fp32"),
])
def test_after_stepping_on_every_path(monkeypatch, name, path, p, L, prec):
    eng = _stepped(monkeypatch, path, p, L, prec)
    exact_r = bool(eng.status().r_is_int8)
    got = eng.block_fields(7)                         # before get_state: the call completes the chunk itself
    S, R, Q = eng.get_state()
    _compare(got, numpy_block_fields(S, R, Q, 7, 3), eng.nq, 3, exact_r, name)
    for b in (1, 32, 33, L // 2 + 1, L):
        _check_all(eng, b, exact_r, what=name)
    eng.close()


_POISON_CHILD = r"""
import sys, numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {root!r} + "/tests")
import spgg_b200
from helpers import C1, full_params
from test_blocks_host import numpy_block_fields
L = 256
eng = spgg_b200.Engine(full_params(dict(C1, L=L)), seeds=9, precision="fp32")
assert eng.describe().startswith("fast"), eng.describe()
eng.init_random(4)
eng.step(120)
got = eng.block_fields(32)            # the first synchronising call: it completes the re-run itself
st = eng.status()
assert st.speculation_failures >= 1, st.speculation_failures
assert st.iteration == 120
S, R, Q = eng.get_state()
c, s, a = numpy_block_fields(S, R, Q, 32, 3)
assert np.array_equal(got["n"], c[..., 0]) and np.array_equal(got["n_C"], c[..., 1])
assert np.array_equal(got["R"], s[..., 0])
assert (np.abs(got["Q"].reshape(s[..., 1:].shape) - s[..., 1:]) <= 2 * 1024 * 2.0 ** -53 * a[..., 1:]).all()
print("ok", st.speculation_failures)
"""


def test_fast_path_with_a_pending_rerun():
    env = dict(os.environ, SPGG_NO_RESIDENT="1", SPGG_SPEC_TEST_POISON="5")
    r = subprocess.run([sys.executable, "-c", _POISON_CHILD.format(root=ROOT)], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_batch_replicas_and_a_stopped_replica(monkeypatch):
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
        got = [eng.block_fields(5, replica=r) for r in range(3)]
        assert eng.status(0).stopped_at == 1 and eng.status(1).iteration == 11
        assert not got[0]["n_C"].any()    # the stopped replica is all D
        for r in range(3):
            S, R, Q = eng.get_state(r)
            _compare(got[r], numpy_block_fields(S, R, Q, 5, 3), 4, 3, True, (no_res, r))
        eng.close()
    L = 131
    eng = _engine([full_params(dict(C1, L=L, r=3.0 + 0.5 * i)) for i in range(3)], seeds=[5, 6, 7], precision="fp32")
    for r in range(3):
        eng.init_random(20 + r, replica=r)
    eng.step(9)
    for r in range(3):
        _check_all(eng, 10, True, rep=r, what=r)
    eng.close()


@pytest.mark.parametrize("name,path,L,prec", [
    ("resident", "cluster", 100, "fp32"),
    ("fast", "fast", 256, "fp32"),
    ("lean", "lean", 97, "fp64"),
])
def test_calls_do_not_disturb_the_run(monkeypatch, name, path, L, prec):
    p = full_params(dict(C1, L=L))
    outs = []
    for chunks in ((200,), (50, 50, 50, 50)):
        eng = _path_engine(monkeypatch, path, p, seeds=8, precision=prec)
        eng.init_random(17)
        rows = []
        for c in chunks:
            eng.step(c)
            if len(chunks) > 1:
                eng.block_fields(3)
                eng.block_fields(L, fields=())
            rows.append(eng.stats()[1:])
        outs.append((eng.digest(),) + eng.get_state() + (np.vstack(rows),))
        eng.close()
    for a, b in zip(*outs):
        assert np.array_equal(np.asarray(a), np.asarray(b))


def test_same_state_same_bits(monkeypatch):
    """The same call twice, and the same state reached on the fast and on the general path (L = 256 would run
    on the resident kernel by default, so both arms switch it off)."""
    L = 256
    res = []
    for path, env in (("fast", ("SPGG_NO_RESIDENT",)), ("general", ("SPGG_NO_RESIDENT", "SPGG_NO_FAST"))):
        for s in ("SPGG_NO_RESIDENT", "SPGG_NO_FAST"):
            monkeypatch.delenv(s, raising=False)
        for s in env:
            monkeypatch.setenv(s, "1")
        eng = _engine(full_params(dict(C1, L=L)), seeds=5, precision="fp32")
        assert eng.describe().startswith("fast" if path == "fast" else "general"), eng.describe()
        eng.init_random(3)
        eng.step(30)
        a = [eng.block_fields(b) for b in (1, 7, 32, 100, L)]
        bb = [eng.block_fields(b) for b in (1, 7, 32, 100, L)]
        for x, y in zip(a, bb):
            for k in x:
                assert np.array_equal(x[k], y[k]) and x[k].tobytes() == y[k].tobytes(), (path, k)
        res.append((eng.digest(), a))
        eng.close()
    for s in ("SPGG_NO_RESIDENT", "SPGG_NO_FAST"):
        monkeypatch.delenv(s, raising=False)
    assert res[0][0] == res[1][0], "the two paths reached different states"
    for x, y in zip(res[0][1], res[1][1]):
        for k in x:
            assert x[k].tobytes() == y[k].tobytes(), k


def test_errors_and_what_a_call_leaves_alone():
    import spgg_b200
    from spgg_b200 import _lib
    L = 64
    eng = _engine(full_params(dict(C1, L=L)), seeds=1, precision="fp32")
    lib, h = eng.lib, eng._h
    cnt = np.full(2 * L * L, -7, np.int64)
    sums = np.full(2 * 5 * L * L, -7.0)
    for rep, b, flags in ((1, 4, 3), (-1, 4, 3), (0, 0, 3), (0, -2, 0), (0, L + 1, 0), (0, 4, 4), (0, 4, 8), (0, 4, -1)):
        assert lib.spgg_block_fields(h, rep, b, flags, cnt.ctypes.data, sums.ctypes.data) == _lib.E_INVALID, (rep, b, flags)
    assert lib.spgg_block_fields(h, 0, 4, 0, None, sums.ctypes.data) == _lib.E_INVALID
    for flags in (1, 2, 3):
        assert lib.spgg_block_fields(h, 0, 4, flags, cnt.ctypes.data, None) == _lib.E_INVALID
    assert lib.spgg_block_fields(h, 0, 4, 0, cnt.ctypes.data, None) == 0     # counts only: sums may be null
    assert (sums == -7.0).all()
    with pytest.raises(ValueError, match="b = 65"):
        eng.block_fields(L + 1)
    # a cluster-labelling result, the pair counts, the iteration counter and the statistics rows survive a call
    eng.init_random(3)
    eng.step(5)
    rows = eng.stats()
    pc = eng.pair_counts(L // 2)
    n = C.c_int64()
    assert lib.spgg_clusters(h, 0, 0, 0, C.byref(n)) == 0
    it = eng.status().iteration
    eng.block_fields(3)
    sizes = np.zeros(n.value, np.int64)
    assert lib.spgg_cluster_sizes(h, sizes.ctypes.data, n.value) == 0
    assert eng.status().iteration == it and np.array_equal(eng.stats(), rows)
    assert np.array_equal(eng.pair_counts(L // 2), pc)
    eng.close()
    # B * B <= 2^24: L = 4097 needs b >= 2
    big = _engine(full_params(dict(C1, L=4097)), seeds=1, precision="fp32")
    with pytest.raises(ValueError, match="2\\^24"):
        big.block_fields(1, fields=())
    assert big.block_fields(2, fields=())["n"].shape == (2049, 2049)
    big.close()


# ------------------------------------------------------------------ L = 16384 and 32768
def _require(host_bytes, dev_bytes):
    import torch
    with open("/proc/meminfo") as f:
        avail = int(re.search(r"MemAvailable:\s+(\d+) kB", f.read()).group(1)) * 1024
    free, _ = torch.cuda.mem_get_info()
    if avail < host_bytes:
        pytest.skip(f"needs {host_bytes / GiB:.1f} GiB of host memory, {avail / GiB:.1f} GiB available")
    if free < dev_bytes:
        pytest.skip(f"needs {dev_bytes / GiB:.1f} GiB of device memory, {free / GiB:.1f} GiB free")


def _counts(S, b):
    """counts of numpy_block_fields for a whole lattice, one block row at a time (host memory stays bounded)"""
    L = S.shape[0]
    B = -(-L // b)
    out = np.empty((B, B, 2), np.int64)
    starts = np.arange(0, L, b)
    for I in range(B):
        rows = S[I * b:(I + 1) * b]
        out[I, :, 0] = rows.shape[0] * np.diff(np.append(starts, L))
        out[I, :, 1] = np.add.reduceat(np.count_nonzero(rows == 0, axis=0), starts)
    return out


def _aligned(S, R, Q, b):
    """numpy_block_fields of rows that are whole block rows of a lattice b divides, by reshaping: counts, sums,
    abs sums, each (rows/b, L/b, 2[, m])"""
    rows, L = S.shape
    shp = (rows // b, b, L // b, b)
    coop = (S == 0).reshape(shp)
    counts = np.stack([np.full((rows // b, L // b), b * b, np.int64), coop.sum(axis=(1, 3))], -1)
    x = np.concatenate([R.reshape(rows, L, 1), Q.reshape(rows, L, -1)], -1).reshape(shp + (-1,))
    c = coop[..., None]
    sums = np.stack([x.sum(axis=(1, 3)), np.where(c, x, 0.0).sum(axis=(1, 3))], 2)
    ax = np.abs(x)
    abs_sums = np.stack([ax.sum(axis=(1, 3)), np.where(c, ax, 0.0).sum(axis=(1, 3))], 2)
    return counts, sums, abs_sums


@pytest.mark.parametrize("L", [16384, 32768])
def test_large_lattices(L):
    """Counts against S read back alone; all channels after init_random against c_oracle.init_random, restated
    1024 rows at a time (host memory stays bounded)."""
    from oracle import c_oracle
    _require(6 * GiB, L * L * 20 + 2 * GiB)
    eng = _engine(full_params(dict(C1, L=L)), seeds=1, precision="fp32")
    assert eng.describe().startswith("fast"), eng.describe()
    seed = 7
    eng.init_random(seed)
    S = np.empty(L * L, np.uint8)
    assert eng.lib.spgg_get_state(eng._h, 0, S.ctypes.data, None, None) == 0
    S = S.reshape(L, L)
    for b in (8, 32, 1000, L):
        got = eng.block_fields(b, fields=())
        want = _counts(S, b)
        assert np.array_equal(got["n"], want[..., 0]) and np.array_equal(got["n_C"], want[..., 1]), b
    del S
    b, step = 1024, 1024
    got = eng.block_fields(b)
    eng.close()
    gc, gs = _packed(got, 4)
    for i0 in range(0, L, step):
        So, Ro, Qo = c_oracle.init_random(L, seed, 4, "fp32", row0=i0, rows=step)
        c, s, a = _aligned(So, np.asarray(Ro, np.float64), np.asarray(Qo, np.float64), b)
        I = slice(i0 // b, (i0 + step) // b)
        assert np.array_equal(gc[I], c), i0
        assert np.array_equal(gs[I][..., 0], s[..., 0]), i0
        assert (np.abs(gs[I] - s) <= sum_bound(c, a)).all(), i0


def test_tiled_lattice_after_epsilon_0_iterations(monkeypatch):
    """An L = k*P lattice tiled with a P x P state evolves at epsilon = 0 as the P x P torus does, copy for copy
    (test_gpu_large_lattice.py): with b dividing P, the block sums of R and the counts are those of the
    oracle's P x P state, tiled, exactly."""
    from oracle import c_oracle
    P, k = 512, 32
    L = P * k
    _require(L * L * 34 + 2 * GiB, L * L * 44 + 2 * GiB)
    p = full_params(dict(C1, L=L, epsilon=0.0, epsilon_min=0.0))
    rs = np.random.RandomState(1112)
    S0 = rs.randint(0, 2, (P, P)).astype(np.uint8)
    Q0 = rs.uniform(-0.01, 0.01, (P, P, 2, 2)).astype(np.float32).astype(np.float64)
    R0 = np.zeros((P, P))
    eng = _path_engine(monkeypatch, "fast", p, seeds=1112, precision="fp32")

    def tile(a):
        out = np.empty((L, L) + a.shape[2:], a.dtype)
        out.reshape((k, P, k, P) + a.shape[2:])[...] = a[None, :, None]
        return out

    eng.set_state(tile(S0), np.zeros((L, L)), tile(Q0))
    sim = c_oracle.Sim(dict(p, L=P), S0, R0, Q0, "fp32", seed=1112)
    eng.step(12)
    rows_o = sim.run(12)
    assert rows_o.shape[0] == 12 and (rows_o[:, 1] > 0).all()
    for b in (32, 512):
        got = eng.block_fields(b, fields=("R",))
        c, s, _ = numpy_block_fields(sim.S, np.asarray(sim.R, np.float64), None, b, 1)
        reps = L // P
        assert np.array_equal(got["n_C"], np.tile(c[..., 1], (reps, reps))), b
        assert np.array_equal(got["R"], np.tile(s[..., 0], (reps, reps, 1))), b
    eng.close()
