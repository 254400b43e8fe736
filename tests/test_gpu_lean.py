"""GPU parity tests of the lean Q-learning update of the general path (csrc/spgg_lean.cuh): the same
iteration as k_step - reference spgg.py:368-592 with algorithms.py:96-133 - with the TD rule compiled
in, the fp64 rewards looked up instead of divided and the Q entries of a row loaded ahead.  Same
thread <-> site mapping, same arithmetic, same summation order: strategies, reputations, Q-tables AND
every statistics column must be bit-identical to k_step (SPGG_NO_LEAN=1).  Both arms run the same
global-maximum kernel, k_gmax_lean, which the oracle tests pin directly (column 33 of the replays)."""
import numpy as np
import pytest

from helpers import C1, C2, full_params, legacy_stream

pytestmark = pytest.mark.gpu

EXACT = [c for c in range(18) if c not in (4, 5, 6, 7, 8, 9, 10)] + [31, 32, 33]


def _engine(*a, **k):
    import spgg_b200
    return spgg_b200.Engine(*a, **k)


def _run(monkeypatch, lean, p, precision, n, chunks, seed=11, replay=None, batch=1):
    monkeypatch.setenv("SPGG_NO_RESIDENT", "1")
    monkeypatch.setenv("SPGG_NO_FAST", "1")
    if lean:
        monkeypatch.delenv("SPGG_NO_LEAN", raising=False)
    else:
        monkeypatch.setenv("SPGG_NO_LEAN", "1")
    L = p["L"]
    plist = [p] * batch if batch > 1 else p
    eng = _engine(plist, seeds=list(range(seed, seed + batch)) if batch > 1 else seed, precision=precision)
    assert ("k_step_lean" in eng.describe()) == lean, eng.describe()
    rs = np.random.RandomState(seed)
    for r in range(batch):
        Q0 = rs.uniform(-0.01, 0.01, (L, L, 2, 2))
        if precision != "fp64":
            Q0 = Q0.astype(np.float32).astype(np.float64)
        eng.set_state(rs.randint(0, 2, (L, L)), np.zeros((L, L)), Q0, replica=r)
    if replay is not None:
        eng.set_replay(*replay)
    for c in chunks:
        eng.step(c)
    out = []
    for r in range(batch):
        out += list(eng.get_state(r)) + [eng.stats(r)]
    eng.close()
    assert sum(chunks) == n
    return out


CASES = [
    # name, params, precision, iterations, chunking
    ("f64_rep_m1_L200", dict(C1, L=200), "fp64", 40, (40,)),
    ("f64_rep_m2_L150", dict(C1, L=150, use_second_order=True, r=3.6), "fp64", 30, (7, 23)),      # partial last tile column
    ("f64_act_m2_L130", dict(C2, L=130), "fp64", 30, (30,)),                                       # 2 columns in the last tile
    ("f64_act_m1_L97", dict(C2, L=97, use_second_order=False, r=3.0), "fp64", 25, (1, 24)),        # one tile column, odd side
    ("f64_rep_m1_L520_frac", dict(C1, L=520, rep_gain_C=0.3, delta_R_D=0.7), "fp64", 24, (24,)),   # interior + edge tiles, TR = 16
    ("f32f_rep_m1_L300", dict(C1, L=300, rep_gain_C=0.3, delta_R_D=0.7), "fp32", 40, (13, 27)),    # fp32 reputations
    ("f32f_rep_m2_L131", dict(C1, L=131, rep_gain_C=0.3, delta_R_D=0.7, use_second_order=True), "fp32", 30, (30,)),
    ("i8_rep_m1_L1100", dict(C1, L=1100), "fp32", 16, (16,)),                                      # side not a multiple of 32
    ("i8_act_m2_L75", dict(C2, L=75), "fp32", 40, (40,)),
    ("i8_rep_m2_L640_kappa0", dict(C1, L=640, use_second_order=True, influence_factor=0.0), "fp32", 20, (20,)),
]


@pytest.mark.parametrize("name,p,precision,n,chunks", CASES, ids=[c[0] for c in CASES])
def test_lean_equals_general_kernel(monkeypatch, name, p, precision, n, chunks):
    p = full_params(p)
    a = _run(monkeypatch, True, p, precision, n, chunks)
    b = _run(monkeypatch, False, p, precision, n, chunks)
    for x, y in zip(a, b):
        assert x.shape == y.shape
        if x.ndim == 2 and x.shape[1] == 40:
            # the two kernels run different persistent grids (2 and 3 CTAs per SM): once a CTA walks several
            # tiles the per-tile partial sums are grouped differently - integer columns stay exact
            assert np.array_equal(x[:, EXACT], y[:, EXACT]), name
            np.testing.assert_allclose(x, y, rtol=1e-12, atol=1e-9, err_msg=name)
            if (p["L"] + 127) // 128 * ((p["L"] + 7) // 8) <= 296:
                bad = sorted(set(np.nonzero(x != y)[1].tolist()))
                assert not bad, f"{name}: statistics columns {bad} differ"
            continue
        assert np.array_equal(x, y), name


def test_lean_replayed_draws_fp64(monkeypatch):
    """Replayed (rand, randint) streams of the reference (spgg.py:409-417) through the lean kernel."""
    L, n = 96, 20
    p = full_params(dict(C1, L=L))
    _, _, u, b = legacy_stream(3, L, n)
    a = _run(monkeypatch, True, p, "fp64", n, (n,), replay=(u, b))
    c = _run(monkeypatch, False, p, "fp64", n, (n,), replay=(u, b))
    for x, y in zip(a, c):
        assert np.array_equal(x, y)


def test_lean_batched_replicas_and_early_exit(monkeypatch):
    """Three replicas per launch; statistics of one replica do not depend on its batch neighbours."""
    p = full_params(dict(C1, L=140))
    a = _run(monkeypatch, True, p, "fp64", 12, (12,), batch=3)
    b = _run(monkeypatch, False, p, "fp64", 12, (12,), batch=3)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    # a lattice that turns uniform stops at the same iteration on both kernels (spgg.py:405)
    L = 64
    q = full_params(dict(C1, L=L, epsilon=0.0, epsilon_min=0.0))
    res = []
    for lean in (True, False):
        monkeypatch.setenv("SPGG_NO_RESIDENT", "1")
        monkeypatch.setenv("SPGG_NO_FAST", "1")
        if lean:
            monkeypatch.delenv("SPGG_NO_LEAN", raising=False)
        else:
            monkeypatch.setenv("SPGG_NO_LEAN", "1")
        eng = _engine(q, seeds=1, precision="fp64")
        Q0 = np.zeros((L, L, 2, 2))
        Q0[..., 1] = 1.0
        eng.set_state(np.random.RandomState(0).randint(0, 2, (L, L)), np.zeros((L, L)), Q0)
        eng.step(6)
        st = eng.status(0)
        res.append((st.stopped_at, st.iteration) + tuple(eng.get_state()) + (eng.stats(),))
        eng.close()
    assert res[0][:2] == res[1][:2] == (1, 1)
    for x, y in zip(res[0][2:], res[1][2:]):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("path,L", [("general", 24), ("fast", 128)])
def test_stopped_replica_keeps_its_state_across_chunks(monkeypatch, path, L):
    """A replica of a batch that stopped (spgg.py:405) in an earlier chunk is not touched by the launches of
    the later ones: its planes - and, on the fast path, its half of the Q ping-pong pair - must be carried to
    whatever parity the running replicas end on (finish_pending in spgg_capi.cu)."""
    monkeypatch.setenv("SPGG_NO_RESIDENT", "1")
    if path == "general":
        monkeypatch.setenv("SPGG_NO_FAST", "1")
    else:
        monkeypatch.delenv("SPGG_NO_FAST", raising=False)
    monkeypatch.delenv("SPGG_NO_LEAN", raising=False)
    p_stop = full_params(dict(C1, L=L, epsilon=0.0, epsilon_min=0.0))
    p_run = full_params(dict(C1, L=L))
    rs = np.random.RandomState(4)
    Q0 = np.zeros((L, L, 2, 2))
    Q0[..., 1] = 1.0                      # everybody prefers to defect: uniform after iteration 1
    S0 = rs.randint(0, 2, (L, L))
    S1 = rs.randint(0, 2, (L, L))
    Q1 = rs.uniform(-0.01, 0.01, (L, L, 2, 2)).astype(np.float32).astype(np.float64)
    eng = _engine([p_stop, p_run], seeds=[1, 2], precision="fp32")
    assert path in eng.describe()
    eng.set_state(S0, np.zeros((L, L)), Q0, replica=0)
    eng.set_state(S1, np.zeros((L, L)), Q1, replica=1)
    eng.step(10)
    assert eng.status(0).stopped_at == 1 and eng.status(1).iteration == 10
    first = eng.get_state(0)
    for n in (5, 4, 1, 6):                 # odd and even chunk lengths: every parity combination
        eng.step(n)
        assert eng.status(0).iteration == 1
        for x, y in zip(first, eng.get_state(0)):
            assert np.array_equal(x, y)
    assert eng.status(1).iteration == 26
    # the running replica is what it would have been alone
    solo = _engine(p_run, seeds=2, precision="fp32")
    solo.set_state(S1, np.zeros((L, L)), Q1)
    solo.step(26)
    for x, y in zip(solo.get_state(), eng.get_state(1)):
        assert np.array_equal(x, y)
    solo.close()
    eng.close()
