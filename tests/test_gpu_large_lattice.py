"""The digest, the device start state and the L = 32768 lattice against host restatements.

Every other engine-vs-oracle test runs at L <= 4096.  The published one-GPU scaling anchor and the
multi-GPU lines run L = 32768 (2^30 sites, Q offsets beyond 2^34 bytes, 256 tile columns, thousands
of tiles per persistent CTA of k_step_fast), and their only check, ``parity_check`` of
``strips.bench_main``, compares N strips with one handle through ``spgg_state_digest``: a fault both
arms share would pass it.  So here:

1. the device digest equals ``c_oracle.state_digest`` of ``get_state`` on every path and mode, and
   every single sign flip of one R or Q value (+0.0 -> -0.0 included) changes its digest word;
2. ``init_random`` equals its host restatement (whole lattice, strips, and at L = 32768 through the
   digest);
3. at epsilon = 0 the dynamics are deterministic, so an L = k*P lattice tiled with a P x P state
   evolves as the P x P torus does, copy for copy.  The oracle runs at L = P and the engine at L = k*P;
   each chunk compares the digest with the periodic host digest, the integer statistics and the sum
   of R with k^2 times the oracle's, exactly, the global maximum exactly and the float sums to a
   stated tolerance.  (Double Q-learning is left out of this leg: its table choice draws a Philox
   word at every epsilon, keyed by the site's global position, so its copies do not stay equal.)
4. at epsilon = 1 every action is a Philox bit, so S and R after each iteration follow from
   ``c_oracle.explore_actions``, for all 32768 rows and all 1024 words of a row.

The large cases need tens of GB of host memory (an uploaded Q is float64) and of device memory;
each checks ``MemAvailable`` and ``torch.cuda.mem_get_info()`` first and skips, naming what it needs,
when either is short."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from helpers import C1, C2, full_params
from test_gpu_start_states import FRAC_R, INTS, SUM_R, _engine

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GiB = 2 ** 30
M64 = 2 ** 64


def _oracle():
    from oracle import c_oracle
    return c_oracle


def _require(host_bytes, dev_bytes):
    import torch
    with open("/proc/meminfo") as f:
        avail = int(re.search(r"MemAvailable:\s+(\d+) kB", f.read()).group(1)) * 1024
    free, _ = torch.cuda.mem_get_info()
    if avail < host_bytes:
        pytest.skip(f"needs {host_bytes / GiB:.1f} GiB of host memory, {avail / GiB:.1f} GiB available")
    if free < dev_bytes:
        pytest.skip(f"needs {dev_bytes / GiB:.1f} GiB of device memory, {free / GiB:.1f} GiB free")


def _dev_bytes(L, n_rep, nq, precision, r_fp32, fast):
    """Device planes of a handle, with a margin: Q (twice on the fast path), two R and two code planes."""
    eq = 8 if precision == "fp64" else 4
    er = 8 if precision == "fp64" else (4 if r_fp32 else 1)
    return int(n_rep * L * L * (nq * eq * (2 if fast else 1) + 2 * (er + 2) + 1) * 1.05) + GiB


def _tile(a, k):
    """(P, P, ...) -> (k*P, k*P, ...): the lattice whose site (i, j) holds a[i % P, j % P]."""
    P = a.shape[0]
    out = np.empty((k * P, k * P) + a.shape[2:], a.dtype)
    out.reshape((k, P, k, P) + a.shape[2:])[...] = a[None, :, None]
    return out


def _host_digest(eng, rep=0, row0=0):
    S, R, Q = eng.get_state(rep)
    return _oracle().state_digest(S, R, Q, L=eng.L, row0=row0)


def _start(L, nq, precision, seed, zeros=True):
    """A random state; some R and Q values are +0.0 and -0.0."""
    rs = np.random.RandomState(seed)
    S = rs.randint(0, 2, (L, L))
    R = rs.randint(-10, 11, (L, L)).astype(np.float64)
    Q = rs.uniform(-0.01, 0.01, (L, L) + (2,) * (2 if nq == 4 else 3))
    if precision == "fp32":
        Q = Q.astype(np.float32).astype(np.float64)
    if zeros:
        Q.flat[::17] = 0.0
        Q.flat[5::17] = -0.0
        R.flat[::13] = 0.0 if precision != "fp64" else -0.0
    return S, R, Q


# ------------------------------------------------------------------ 1. the digest against the host
DIGEST_CASES = [
    # name, path, params, precision, replicas
    ("cluster_L100", "cluster", dict(C1, L=100), "fp32", 1),
    ("grid_L400", "grid", dict(C1, L=400), "fp32", 1),
    ("fast_L256", "fast", dict(C1, L=256), "fp32", 1),
    ("fast_part_m2_L160", "fast", dict(C1, L=160, use_second_order=True), "fp32", 1),
    ("fast_batch3_L128", "fast", dict(C1, L=128), "fp32", 3),
    ("lean_int8_L100", "lean", dict(C1, L=100), "fp32", 1),
    ("lean_fracR_L300", "lean", dict(FRAC_R, L=300), "fp32", 1),
    ("lean_fp64_L130", "lean", dict(C1, L=130, use_second_order=True), "fp64", 1),
    ("sarsa_k_step_L131", "k_step", dict(C1, L=131, algorithm="sarsa"), "fp32", 1),
    ("double_q_k_step_L131", "k_step", dict(C2, L=131, algorithm="double_qlearning"), "fp32", 1),
    ("double_q_fp64_L70", "k_step", dict(C1, L=70, algorithm="double_qlearning"), "fp64", 1),
]


@pytest.mark.parametrize("name,path,p,precision,n_rep", DIGEST_CASES, ids=[c[0] for c in DIGEST_CASES])
def test_digest_equals_host_restatement(monkeypatch, name, path, p, precision, n_rep):
    """After the upload and after 1, 2 and 5 iterations (both plane parities), every replica."""
    p = full_params(p)
    plist = [dict(p, r=p["r"] + 0.3 * i) for i in range(n_rep)]
    eng = _engine(monkeypatch, path, plist if n_rep > 1 else p, seeds=list(range(7, 7 + n_rep)), precision=precision)
    for rep in range(n_rep):
        eng.set_state(*_start(p["L"], eng.nq, precision, 40 + rep), replica=rep)
    for n in (0, 1, 1, 3):
        if n:
            eng.step(n)
        for rep in range(n_rep):
            assert eng.digest(rep) == _host_digest(eng, rep), f"{name}: replica {rep} after {eng.status(rep).iteration}"
    eng.close()


@pytest.mark.parametrize("path,precision", [("fast", "fp32"), ("lean", "fp64")])
def test_strip_digest_equals_host_restatement(monkeypatch, path, precision):
    """A strip's digest keys its sites by their global rows (row0 > 0)."""
    L, row0, rows = 128, 48, 32
    p = full_params(dict(C1, L=L))
    S, R, Q = _start(L, 4, precision, 5)
    eng = _engine(monkeypatch, path, p, seeds=1, precision=precision, rows=rows, row0=row0)
    eng.set_state(S[row0:row0 + rows], R[row0:row0 + rows], Q[row0:row0 + rows])
    want = _oracle().state_digest(S[row0:row0 + rows], R[row0:row0 + rows], Q[row0:row0 + rows], L=L, row0=row0)
    assert eng.digest() == _host_digest(eng, row0=row0) == want
    eng.close()


_POISON_CHILD = r"""
import sys, numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {root!r} + "/tests")
import spgg_b200
from helpers import C1, full_params
from oracle import c_oracle
L = 256
eng = spgg_b200.Engine(full_params(dict(C1, L=L)), seeds=9, precision="fp32")
assert eng.describe().startswith("fast"), eng.describe()
rs = np.random.RandomState(3)
eng.set_state(rs.randint(0, 2, (L, L)), rs.randint(-10, 11, (L, L)), rs.uniform(-0.01, 0.01, (L, L, 2, 2)))
eng.step(120)
d = eng.digest()                     # the first synchronising call: it completes the re-run itself
st = eng.status()
assert st.speculation_failures >= 1 and st.iteration == 120, (st.speculation_failures, st.iteration)
S, R, Q = eng.get_state()
assert d == c_oracle.state_digest(S, R, Q), "digest of a chunk with a pending re-run"
print("ok", st.speculation_failures)
"""


def test_digest_after_a_chunk_with_a_pending_rerun():
    env = dict(os.environ, SPGG_NO_RESIDENT="1", SPGG_SPEC_TEST_POISON="5")
    r = subprocess.run([sys.executable, "-c", _POISON_CHILD.format(root=ROOT)], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.parametrize("path,p,precision", [("fast", dict(C1, L=128), "fp32"),
                                              ("k_step", dict(C1, L=64, algorithm="double_qlearning"), "fp64")],
                         ids=["fast_int8", "double_q_fp64"])
def test_every_single_sign_flip_changes_the_digest(monkeypatch, path, p, precision):
    """For 64 sites, one change at a time: the sign of R, the sign of each Q entry, and +0.0 -> -0.0 in Q
    (and in R where R is stored as a double).  Each must change its word of the digest and no other."""
    p = full_params(p)
    L = p["L"]
    eng = _engine(monkeypatch, path, p, seeds=1, precision=precision)
    nq = eng.nq
    S, R, Q = _start(L, nq, precision, 11, zeros=False)
    R[R == 0] = 3.0
    Qf = Q.reshape(L, L, nq)
    sites = np.random.RandomState(12).choice(L * L, 64, replace=False)
    for x in sites:                           # one entry per site is +0.0: its sign flip makes it -0.0
        Qf.flat[x * nq + x % nq] = 0.0
    eng.set_state(S, R, Q)
    d0 = eng.digest()
    missed = []

    def check(what, word):
        eng.set_state(S, R, Q)
        d = eng.digest()
        others = [w for w in range(3) if w != word]
        assert [d[w] for w in others] == [d0[w] for w in others], what
        if d[word] == d0[word]:
            missed.append(what)

    n = 0
    for x in sites:
        i, j = divmod(int(x), L)
        R[i, j] = -R[i, j]
        check(f"R[{i},{j}] sign", 1)
        R[i, j] = -R[i, j]
        n += 1
        for z in range(nq):
            Qf[i, j, z] = -Qf[i, j, z]
            check(f"Q[{i},{j}][{z}] sign ({Qf[i, j, z]!r})", 2)
            Qf[i, j, z] = -Qf[i, j, z]
            n += 1
        if precision == "fp64":                # R is stored as a double: +0.0 and -0.0 differ
            r0 = R[i, j]
            R[i, j] = 0.0
            eng.set_state(S, R, Q)
            d_pos = eng.digest()
            R[i, j] = -0.0
            eng.set_state(S, R, Q)
            if eng.digest()[1] == d_pos[1]:
                missed.append(f"R[{i},{j}] +0.0 -> -0.0")
            R[i, j] = r0
            n += 1
    eng.close()
    assert not missed, f"{len(missed)} of {n} single-value changes left the digest unchanged, e.g. {missed[:4]}"


# ------------------------------------------------------------------ 2. init_random against its restatement
INIT_CASES = [("lean", dict(C1, L=100), "fp32"), ("fast", dict(C1, L=160), "fp32"), ("lean", dict(C1, L=37), "fp64"),
              ("k_step", dict(C2, L=70, algorithm="double_qlearning"), "fp32"),
              ("k_step", dict(C2, L=45, algorithm="double_qlearning"), "fp64")]


@pytest.mark.parametrize("path,p,precision", INIT_CASES,
                         ids=[f"{c[0]}_L{c[1]['L']}_{c[2]}" + ("_dq" if "algorithm" in c[1] else "") for c in INIT_CASES])
def test_init_random_equals_restatement(monkeypatch, path, p, precision):
    p = full_params(p)
    L, seed = p["L"], 0xfeed_0000_0000 + p["L"]
    eng = _engine(monkeypatch, path, p, seeds=1, precision=precision)
    eng.init_random(seed)
    S, R, Q = eng.get_state()
    So, Ro, Qo = _oracle().init_random(L, seed, eng.nq, precision)
    assert np.array_equal(S, So) and np.array_equal(R, Ro) and np.array_equal(Q, Qo)
    assert not np.signbit(R).any()
    assert eng.digest() == _oracle().init_random_digest(L, seed, eng.nq, precision)
    eng.close()


def test_init_random_strips_equal_rows_of_the_lattice(monkeypatch):
    L, seed = 128, 2 ** 33 + 5
    p = full_params(dict(C1, L=L))
    whole = _engine(monkeypatch, "fast", p, seeds=1, precision="fp32")
    whole.init_random(seed)
    Sw, Rw, Qw = whole.get_state()
    total = [0, 0, 0]
    for row0, rows in ((0, 48), (48, 16), (64, 64)):
        e = _engine(monkeypatch, "fast", p, seeds=1, precision="fp32", rows=rows, row0=row0)
        e.init_random(seed)
        S, R, Q = e.get_state()
        assert np.array_equal(S, Sw[row0:row0 + rows]) and np.array_equal(R, Rw[row0:row0 + rows])
        assert np.array_equal(Q, Qw[row0:row0 + rows])
        d = e.digest()
        assert d == _oracle().init_random_digest(L, seed, 4, "fp32", row0=row0, rows=rows)
        total = [(a + b) % M64 for a, b in zip(total, d)]
        e.close()
    assert tuple(total) == whole.digest()
    whole.close()


@pytest.mark.parametrize("path,p,L", [("fast", C1, 32768), ("k_step", dict(C2, algorithm="double_qlearning"), 16384)],
                         ids=["fast_L32768", "double_q_L16384"])
def test_init_random_digest_at_large_L(monkeypatch, path, p, L):
    """The start state of both arms of parity_check and of the bench's large lattices."""
    nq = 8 if "double" in str(p.get("algorithm")) else 4
    _require(GiB, _dev_bytes(L, 1, nq, "fp32", False, path == "fast"))
    seed = 2024
    eng = _engine(monkeypatch, path, full_params(dict(p, L=L)), seeds=1, precision="fp32")
    eng.init_random(seed)
    got = eng.digest()
    eng.close()
    assert got == _oracle().init_random_digest(L, seed, nq, "fp32")


# ------------------------------------------------------------------ 3. L = k*P lattices at epsilon = 0
EPS0 = dict(epsilon=0.0, epsilon_min=0.0)
CHUNKS = (1, 11, 12)


def _diagnose(eng, rep, sim, k):
    """Which P x P blocks and which rows of S and R differ from the tiled oracle state."""
    P = sim.L
    S, R, _ = eng.get_state(rep, want_q=False)
    bad = (S.reshape(k, P, k, P) != sim.S[None, :, None, :]) | \
          (R.reshape(k, P, k, P) != sim.R.astype(np.float64)[None, :, None, :])
    del S, R
    blocks = np.argwhere(bad.any(axis=(1, 3)))
    rows = np.nonzero(bad.any(axis=(2, 3)).reshape(-1))[0]
    if not blocks.size:
        return "S and R equal the tiled oracle state: the Q digest differs"
    return (f"{bad.sum()} S/R mismatches in {len(blocks)} of {k * k} blocks (first {blocks[:5].tolist()}), "
            f"{rows.size} rows (first {rows[:8].tolist()})")


def _compare_rows(full, rows_o, k, precision, int8_r, L, where):
    c = rows_o.shape[0]
    rows, sum_r = full[1:c + 1], full[:c, SUM_R]
    k2 = k * k
    bad = np.nonzero((rows[:, INTS] != k2 * rows_o[:, INTS]).any(axis=1))[0]
    assert bad.size == 0, f"{where}: integer statistics differ from k^2 x the oracle's at row {bad[:1] + 1}"
    if precision == "fp64":
        assert np.array_equal(rows[:, 33], rows_o[:, 33]), f"{where}: global maximum"
        np.testing.assert_allclose(rows[:, 4:11], k2 * rows_o[:, 4:11], rtol=1e-10, atol=1e-9 * k2)
        np.testing.assert_allclose(sum_r, k2 * rows_o[:, SUM_R], rtol=1e-10, atol=1e-9 * k2)
        np.testing.assert_allclose(rows[:, 18:31], k2 * rows_o[:, 18:31], rtol=1e-9, atol=1e-9 * k2)
        return
    assert np.array_equal(rows[:, 33].astype(np.float32), rows_o[:, 33].astype(np.float32)), f"{where}: global maximum"
    # fp32 kernels sum the ratio, the NI percentages and Q per thread in fp32 (k_step_fast: up to 28,000
    # sites a thread here) before the double fold, and the defector Q columns are the total minus the
    # cooperators' column: their error scales with the total of that Q entry, not with the column itself
    np.testing.assert_allclose(rows[:, 4:10], k2 * rows_o[:, 4:10], rtol=1e-5)
    np.testing.assert_allclose(rows[:, 10], k2 * rows_o[:, 10], rtol=1e-4)
    if int8_r:
        assert np.array_equal(sum_r, k2 * rows_o[:, SUM_R]), f"{where}: sums of R differ"
    else:
        np.testing.assert_allclose(sum_r, k2 * rows_o[:, SUM_R], rtol=1e-6, atol=1e-6 * L * L)
    for z in range(4):
        cols = [18 + z, 22 + z, 26 + z]
        scale = np.abs(k2 * rows_o[:, 18 + z])[:, None]
        np.testing.assert_array_less(np.abs(rows[:, cols] - k2 * rows_o[:, cols]),
                                     2e-4 * np.abs(k2 * rows_o[:, cols]) + 1e-6 * scale + 1e-2 * (L / 4096) ** 2,
                                     err_msg=f"{where}: Q sums of entry {z}")
    np.testing.assert_allclose(rows[:, 30], k2 * rows_o[:, 30], rtol=2e-4)


def _periodic_run(monkeypatch, path, plist, P, k, precision, seed):
    c_oracle = _oracle()
    L = k * P
    plist = [full_params(dict(p, L=L, **EPS0)) for p in plist]
    nq = 4
    r_fp32 = precision == "fp32" and any(float(p["rep_gain_C"]) % 1 or float(p["delta_R_D"]) % 1 for p in plist)
    _require(L * L * (8 * nq + 2) + 2 * GiB, _dev_bytes(L, len(plist), nq, precision, r_fp32, path == "fast"))
    rs = np.random.RandomState(seed)
    S0 = rs.randint(0, 2, (P, P)).astype(np.uint8)
    Q0 = rs.uniform(-0.01, 0.01, (P, P, 2, 2))
    if precision == "fp32":
        Q0 = Q0.astype(np.float32).astype(np.float64)
    R0 = np.zeros((P, P))
    eng = _engine(monkeypatch, path, plist if len(plist) > 1 else plist[0], seeds=[seed] * len(plist),
                  precision=precision)
    S_big, Q_big = _tile(S0, k), _tile(Q0, k)
    for rep in range(len(plist)):
        eng.set_state(S_big, np.zeros((L, L)), Q_big, replica=rep)    # R's pages are never written
    del S_big, Q_big
    sims = [c_oracle.Sim(dict(p, L=P), S0, R0, Q0, precision, seed=seed) for p in plist]
    w = c_oracle.digest_weights(L, nq, period=P)
    for rep, sim in enumerate(sims):
        assert eng.digest(rep) == c_oracle.state_digest(sim.S, sim.R, sim.Q, L=L, period=P, weights=w)
    t = 0
    for n, c in enumerate(CHUNKS):
        eng.step(c)
        for rep, sim in enumerate(sims):
            where = f"replica {rep}, chunk {n + 1} (iterations {t + 1}-{t + c})"
            rows_o = sim.run(c)
            assert rows_o.shape[0] == c, f"{where}: the oracle's torus turned uniform"
            assert (rows_o[:, 1] > 0).all() and (rows_o[:, 2] > 0).all(), f"{where}: no switches, nothing tested"
            st = eng.status(rep)
            assert st.stopped_at == -1 and st.iteration == t + c, (st.stopped_at, st.iteration)
            d = eng.digest(rep)
            want = c_oracle.state_digest(sim.S, sim.R.astype(np.float64), sim.Q.astype(np.float64), L=L,
                                         period=P, weights=w)
            if d != want:
                pytest.fail(f"{where}: digest {d} != {want}; {_diagnose(eng, rep, sim, k)}")
            _compare_rows(eng.stats(rep), rows_o, k, precision, bool(st.r_is_int8), L, where)
        t += c
    eng.close()


PERIODIC_CASES = [
    # name, path, params (one per replica), P, k, precision
    ("fast_c1_L32768", "fast", [C1], 512, 64, "fp32"),
    ("fast_c2_L32768", "fast", [C2], 512, 64, "fp32"),
    ("fast_batch2_L32768", "fast", [C1, dict(C1, r=3.6, influence_factor=0.5)], 512, 64, "fp32"),
    ("lean_fracR_L32768", "lean", [FRAC_R], 512, 64, "fp32"),
    ("lean_fp64_L16384", "lean", [C1], 512, 32, "fp64"),
    ("lean_L16380", "lean", [C1], 420, 39, "fp32"),
    ("sarsa_k_step_L16384", "k_step", [dict(C1, algorithm="sarsa")], 512, 32, "fp32"),
    ("expected_sarsa_k_step_L16384", "k_step", [dict(C2, algorithm="expected_sarsa")], 512, 32, "fp32"),
]


@pytest.mark.parametrize("name,path,plist,P,k,precision", PERIODIC_CASES, ids=[c[0] for c in PERIODIC_CASES])
def test_tiled_lattice_at_epsilon_0_vs_oracle(monkeypatch, name, path, plist, P, k, precision):
    _periodic_run(monkeypatch, path, plist, P, k, precision, seed=600 + P)


# ------------------------------------------------------------------ 4. Philox counters at epsilon = 1
def test_every_row_and_word_at_epsilon_1_on_the_fast_path(monkeypatch):
    """Each iteration's S is the Philox action plane and R moves by +1 / -1 into the clamps [-1, 1], which
    clip from iteration 2 on.  S and R digests and the count of C actions (column 3) are compared exactly."""
    c_oracle = _oracle()
    L, P, seed = 32768, 512, 77
    _require(3 * GiB, _dev_bytes(L, 1, 4, "fp32", False, True))
    p = full_params(dict(C1, L=L, epsilon=1.0, epsilon_min=1.0, epsilon_decay=1.0, R_min=-1, R_max=1))
    eng = _engine(monkeypatch, "fast", p, seeds=seed, precision="fp32")
    S_big = _tile(np.random.RandomState(3).randint(0, 2, (P, P)).astype(np.uint8), L // P)
    eng.set_state(S_big, np.zeros((L, L)), np.zeros((L, L, 2, 2)))  # zero pages: nothing is written
    del S_big
    R = np.zeros((L, L), np.int8)
    block = 2048
    for t in (1, 2, 3):
        eng.step(1)
        dS = dR = 0
        n_c = 0
        for i0 in range(0, L, block):
            a = c_oracle.explore_actions(L, seed, t, i0, i0 + block)
            Rb = R[i0:i0 + block]
            np.clip(Rb + np.where(a == 0, 1, -1).astype(np.int8), -1, 1, out=Rb)
            d = c_oracle.state_digest(a, Rb.astype(np.float64), None, L=L, row0=i0)
            dS, dR = (dS + d[0]) % M64, (dR + d[1]) % M64
            n_c += int((a == 0).sum())
        got = eng.digest()
        assert (got[0], got[1]) == (dS, dR), f"iteration {t}: S/R digests differ"
        row = eng.stats()[1]
        assert row[3] == n_c, (t, row[3], n_c)
    assert eng.status().iteration == 3
    eng.close()
