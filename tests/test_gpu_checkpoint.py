"""Checkpoint / resume through the C ABI (SURVEY 8 f4; include/spgg.h: spgg_set_progress): n
iterations in one handle == k iterations, state to the host, handle destroyed, fresh handle,
state uploaded, spgg_set_progress, n-k iterations - bit for bit (S, R, Q, the statistic rows of
the second half, epsilon), on all three kernel paths.  The reference itself can only inject
strategies (S_in_one, spgg.py:51,133,161)."""
import numpy as np
import pytest

from helpers import C1, C2, full_params

pytestmark = pytest.mark.gpu

CASES = [
    # name, params, precision, environment pins, expected path
    ("resident_cluster", dict(C1, L=64), "fp32", {}, "resident"),
    ("resident_grid", dict(C1, L=400), "fp32", {}, "resident"),
    ("fast_tma", dict(C1, L=256), "fp32", {"SPGG_NO_RESIDENT": "1"}, "fast"),
    ("fast_tma_m2_action", dict(C2, L=256), "fp32", {"SPGG_NO_RESIDENT": "1"}, "fast"),
    ("general_fp32", dict(C1, L=100), "fp32", {"SPGG_NO_RESIDENT": "1"}, "general"),
    ("general_fp64", dict(C2, L=48), "fp64", {}, "general"),
    # the other TD rules run on k_step only; Double Q-learning checkpoints both tables
    ("sarsa_fp32", dict(C1, L=100, algorithm="sarsa"), "fp32", {}, "general"),
    ("expected_sarsa_fp64", dict(C2, L=48, algorithm="expected_sarsa"), "fp64", {}, "general"),
    ("double_q_fp32", dict(C1, L=100, algorithm="double_qlearning"), "fp32", {}, "general"),
    ("double_q_fp64", dict(C2, L=48, algorithm="double_qlearning"), "fp64", {}, "general"),
]


@pytest.mark.parametrize("name,p,precision,env,path", CASES, ids=[c[0] for c in CASES])
def test_resume_is_bit_identical(monkeypatch, name, p, precision, env, path):
    import spgg_b200
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    p = full_params(p)
    L, n, k = p["L"], 100, 50
    one = spgg_b200.Engine(p, seeds=31, precision=precision)
    assert one.describe().startswith(path), one.describe()
    rs = np.random.RandomState(9)
    Q0 = rs.uniform(-0.01, 0.01, (L, L, one.nq))   # Double Q-learning: both tables, [site][table][s][a]
    S0 = rs.randint(0, 2, (L, L))
    R0 = np.zeros((L, L))

    one.set_state(S0, R0, Q0)
    one.step(k)
    one.step(n - k)
    rows_one = one.stats()
    S1, R1, Q1 = one.get_state()
    st1 = one.status()

    a = spgg_b200.Engine(p, seeds=31, precision=precision)
    a.set_state(S0, R0, Q0)
    a.step(k)
    ck = a.checkpoint()
    assert ck["iteration"] == k
    a.close()
    b = spgg_b200.Engine(p, seeds=31, precision=precision)
    b.restore(ck)
    assert b.status().iteration == k and b.status().epsilon == ck["epsilon"][0]
    b.step(n - k)
    rows_b = b.stats()
    S2, R2, Q2 = b.get_state()
    st2 = b.status()
    assert np.array_equal(S1, S2), f"{(S1 != S2).sum()} strategy mismatches after the resume"
    assert np.array_equal(R1, R2) and np.array_equal(Q1, Q2)
    assert np.array_equal(rows_one[1:], rows_b[1:])          # same kernels, same fold order
    assert st1.iteration == st2.iteration == n and st1.epsilon == st2.epsilon
    one.close(); b.close()


def test_resume_a_batch_and_the_stale_replica_rule(monkeypatch):
    """The iteration counter is handle-wide: re-seeding one replica of a batch after iterations
    have run starts a new run, and stepping is refused until every replica has a state."""
    import spgg_b200
    ps = [full_params(dict(C1, L=64, r=r)) for r in (3.0, 4.0, 5.0)]
    rs = np.random.RandomState(4)
    st0 = [(rs.randint(0, 2, (64, 64)), np.zeros((64, 64)), rs.uniform(-0.01, 0.01, (64, 64, 2, 2)))
           for _ in ps]
    one = spgg_b200.Engine(ps, seeds=[5, 6, 7], precision="fp32")
    for r, s in enumerate(st0):
        one.set_state(*s, replica=r)
    one.step(60)
    want = [one.get_state(r) for r in range(3)]

    a = spgg_b200.Engine(ps, seeds=[5, 6, 7], precision="fp32")
    for r, s in enumerate(st0):
        a.set_state(*s, replica=r)
    a.step(25)
    ck = a.checkpoint()
    # a new run on the same handle: replica 0 re-seeded, 1 and 2 stale -> stepping refused
    a.set_state(*st0[0], replica=0)
    with pytest.raises(RuntimeError, match="previous run"):
        a.step(1)
    with pytest.raises(RuntimeError):
        a.set_progress(25, ck["epsilon"])
    a.restore(ck)                                            # every replica uploaded, then progress
    a.step(35)
    for r in range(3):
        S, R, Q = a.get_state(r)
        assert np.array_equal(S, want[r][0]) and np.array_equal(R, want[r][1])
        assert np.array_equal(Q, want[r][2])
    one.close(); a.close()


def test_digests_add_up_over_row_blocks():
    """spgg_state_digest: strips of a lattice add up (mod 2^64) to the whole lattice's digest."""
    import spgg_b200
    L = 128
    p = full_params(dict(C1, L=L))
    rs = np.random.RandomState(12)
    S0, R0 = rs.randint(0, 2, (L, L)), rs.randint(-10, 11, (L, L)).astype(np.float64)
    Q0 = rs.uniform(-1, 1, (L, L, 2, 2)).astype(np.float32).astype(np.float64)
    whole = spgg_b200.Engine(p, precision="fp32")
    whole.set_state(S0, R0, Q0)
    dw = whole.digest()
    parts = [0, 0, 0]
    for row0, rows in ((0, 48), (48, 16), (64, 64)):
        e = spgg_b200.Engine(p, precision="fp32", rows=rows, row0=row0)
        e.set_state(S0[row0:row0 + rows], R0[row0:row0 + rows], Q0[row0:row0 + rows])
        d = e.digest()
        parts = [(x + y) % 2 ** 64 for x, y in zip(parts, d)]
        e.close()
    assert tuple(parts) == dw
    S1 = S0.copy(); S1[5, 7] ^= 1
    whole.set_state(S1, R0, Q0)
    d1 = whole.digest()
    assert d1[0] != dw[0] and d1[1:] == dw[1:]
    whole.close()


@pytest.mark.parametrize("precision,gain,loss", [("fp32", 1.0, 1.0), ("fp32", 0.25, 0.75), ("fp32", 0.3, 0.7),
                                                 ("fp64", 0.3, 0.7)])
def test_device_histogram_equals_numpy(precision, gain, loss):
    """rep_hist_* (spgg.py:399-401,626-628): np.histogram(R, bins=20, range=(R_min, R_max)) computed on the
    device - int8 units, fp32 and fp64 reputations, values on and between the bin edges."""
    import spgg_b200
    L = 96
    p = full_params(dict(C1, L=L, rep_gain_C=gain, delta_R_D=loss))
    rs = np.random.RandomState(1)
    eng = spgg_b200.Engine(p, seeds=2, precision=precision)
    eng.set_state(rs.randint(0, 2, (L, L)), np.zeros((L, L)), rs.uniform(-0.01, 0.01, (L, L, 2, 2)))
    for n in (1, 7, 40):
        eng.step(n)
        _S, R, _Q = eng.get_state(want_q=False)
        want_c, want_e = np.histogram(R, bins=20, range=(p["R_min"], p["R_max"]))
        got_c, got_e = eng.r_histogram(20, p["R_min"], p["R_max"])
        assert np.array_equal(got_c, want_c) and got_c.dtype == want_c.dtype
        assert np.array_equal(got_e, want_e)
        want_c, _ = np.histogram(R, bins=7, range=(-3.5, 2.25))      # values outside the range are dropped
        got_c, _ = eng.r_histogram(7, -3.5, 2.25)
        assert np.array_equal(got_c, want_c)
    eng.close()
