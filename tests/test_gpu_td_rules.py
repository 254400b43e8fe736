"""SARSA, Expected SARSA and Double Q-learning on the general kernel (k_step) against the C oracle.

These rules run only on k_step (never on the fast, resident or lean path), selected at run time by
the algorithm code.  Compared here, bit for bit for S, R, Q (both Double-Q tables) and the integer
statistics: fp64 with replayed draws, fp32 with Philox streams 0/1/2 in every reputation storage
mode (int8, int8 in units of 1/2, fp32), fp32 with replayed draw pairs, at sides that leave a
partial last tile column, make CTAs walk several tiles and reach the benchmarked L=4096 geometry;
then the epsilon bookkeeping, batching, chunking and early exit under these rules."""
import numpy as np
import pytest

from helpers import C1, C2, full_params

pytestmark = pytest.mark.gpu

RULES = ["sarsa", "expected_sarsa", "double_qlearning"]
PAIRS = {"qlearning": 1, "sarsa": 3, "expected_sarsa": 1, "double_qlearning": 2}
INTS = [0, 1, 2, 3, 11, 12, 13, 14, 15, 16, 31, 32]
SUM_R = 17

INT8 = dict(C1)                                           # R in int8 units of 1
HALF_R = dict(C1, rep_gain_C=0.5)                         # int8 in units of 1/2
FRAC_R = dict(C1, rep_gain_C=0.3, delta_R_D=0.7)          # fp32 R


def _engine(*a, **k):
    import spgg_b200
    return spgg_b200.Engine(*a, **k)


def _init(p, seed, precision):
    """Random S0 and Q0 (two tables for Double Q-learning), fp32-representable for fp32 runs."""
    L = p["L"]
    rs = np.random.RandomState(seed)
    shape = (L, L, 2, 2, 2) if p.get("algorithm") == "double_qlearning" else (L, L, 2, 2)
    Q0 = rs.uniform(-0.01, 0.01, shape)
    if precision == "fp32":
        Q0 = Q0.astype(np.float32).astype(np.float64)
    S0 = rs.randint(0, 2, (L, L))
    return rs, S0, Q0


def _draw_pairs(rs, algo, n, L):
    pairs = PAIRS[algo]
    return rs.rand(n, pairs, L, L), rs.randint(0, 2, (n, pairs, L, L)).astype(np.uint8)


def _arm(eng, u, b):
    """set_replay takes (n, L, L) for one pair per iteration, (n, pairs, L, L) otherwise."""
    if u.shape[1] == 1:
        eng.set_replay(u[:, 0], b[:, 0])
    else:
        eng.set_replay(u, b)


def _assert_k_step(eng):
    d = eng.describe()
    assert d.startswith("general") and "+ k_step)" in d, d


def _compare(eng, sim, rows_o, precision, n):
    """Engine state and statistic rows == the oracle's.  Float columns: the tolerances of the
    Q-learning parity tests (fp32 sums are grouped per tile, fp64 sums in another order)."""
    L = eng.L
    S, R, Q = eng.get_state()
    full = eng.stats()
    rows = full[1:]
    # the sum of R before the action is recorded by the launch that chooses the action, one row earlier
    sum_r = full[:-1, SUM_R]
    assert rows_o.shape[0] == n and rows.shape == rows_o.shape
    assert np.array_equal(S, sim.S), f"{(S != sim.S).sum()} strategy mismatches"
    if precision == "fp64":
        assert np.array_equal(R, sim.R)
        assert np.array_equal(Q, sim.Q), f"{(Q != sim.Q).sum()} Q mismatches"
    else:
        assert np.array_equal(R, sim.R.astype(np.float64))
        assert np.array_equal(Q.astype(np.float32), sim.Q), f"{(Q.astype(np.float32) != sim.Q).sum()} Q mismatches"
    assert np.array_equal(rows[:, INTS], rows_o[:, INTS])
    if precision == "fp64":
        assert np.array_equal(rows[:, 33], rows_o[:, 33])
        np.testing.assert_allclose(rows[:, 4:11], rows_o[:, 4:11], rtol=1e-10, atol=1e-9)
        np.testing.assert_allclose(sum_r, rows_o[:, SUM_R], rtol=1e-10, atol=1e-9)
        np.testing.assert_allclose(rows[:, 18:31], rows_o[:, 18:31], rtol=1e-9, atol=1e-9)
        return
    assert np.array_equal(rows[:, 33].astype(np.float32), rows_o[:, 33].astype(np.float32))
    big = L >= 4096
    np.testing.assert_allclose(rows[:, 4:11], rows_o[:, 4:11], rtol=1e-5 if big else 1e-6, atol=0 if big else 1e-6)
    if eng.status().r_is_int8:
        assert np.array_equal(sum_r, rows_o[:, SUM_R])   # integer units, scaled once
    else:
        # fp32 partial sums per thread and tile: about one rounding of a 64-site sum per 64 sites
        np.testing.assert_allclose(sum_r, rows_o[:, SUM_R], rtol=1e-6, atol=1e-6 * L * L)
    np.testing.assert_allclose(rows[:, 18:31], rows_o[:, 18:31], rtol=2e-4 if big else 1e-4,
                               atol=1e-2 if big else 1e-3)


# ------------------------------------------------------------------ a. fp64, replayed draws
F64_SHAPES = [
    ("L97_rep_m1", dict(C1, L=97), 40),                                     # odd, one tile column
    ("L130_act_m2", dict(C2, L=130), 30),                                   # two columns in the last tile
    ("L300_rep_m2", dict(C1, L=300, use_second_order=True), 12),            # several tiles per CTA
    ("L520_act_m1", dict(C2, L=520, use_second_order=False, rep_gain_C=0.3, delta_R_D=0.7), 8),
]


@pytest.mark.parametrize("algo", RULES)
@pytest.mark.parametrize("name,p,n", F64_SHAPES, ids=[c[0] for c in F64_SHAPES])
def test_fp64_replay_vs_oracle(algo, name, p, n):
    from oracle import c_oracle
    p = full_params(dict(p, algorithm=algo))
    L = p["L"]
    rs, S0, Q0 = _init(p, 100 + L, "fp64")
    u, b = _draw_pairs(rs, algo, n, L)
    eng = _engine(p, precision="fp64")
    _assert_k_step(eng)
    eng.set_state(S0, np.zeros((L, L)), Q0)
    _arm(eng, u, b)
    eng.step(n)
    sim = c_oracle.Sim(p, S0, np.zeros((L, L)), Q0, "fp64")
    rows_o = sim.run(n, lambda t, L_: (u[t - 1], b[t - 1]))
    _compare(eng, sim, rows_o, "fp64", n)
    eng.close()


# ------------------------------------------------------------------ b. fp32, Philox
F32_CASES = [
    # name, rule, params, iterations
    ("sarsa_int8_L75", "sarsa", dict(INT8, L=75), 40),
    ("expsarsa_halfR_L75", "expected_sarsa", dict(HALF_R, L=75, use_second_order=True), 40),
    ("doubleq_fracR_L75", "double_qlearning", dict(FRAC_R, L=75), 40),
    ("sarsa_halfR_L131", "sarsa", dict(HALF_R, L=131, use_second_order=True), 40),
    ("expsarsa_fracR_L131", "expected_sarsa", dict(FRAC_R, L=131), 40),
    ("doubleq_int8_L131_act", "double_qlearning", dict(C2, L=131), 40),
    ("sarsa_fracR_L256", "sarsa", dict(FRAC_R, L=256, use_second_order=True), 40),
    ("expsarsa_int8_L256_act", "expected_sarsa", dict(C2, L=256, use_second_order=False), 40),
    ("doubleq_halfR_L256", "double_qlearning", dict(HALF_R, L=256), 40),
    ("sarsa_int8_L1000", "sarsa", dict(INT8, L=1000), 16),                  # benchmarked
    ("expsarsa_int8_L1000", "expected_sarsa", dict(INT8, L=1000), 16),
    ("doubleq_int8_L1000", "double_qlearning", dict(INT8, L=1000), 16),
    ("sarsa_int8_L4096", "sarsa", dict(INT8, L=4096), 8),                   # benchmark geometry
    ("doubleq_int8_L4096", "double_qlearning", dict(INT8, L=4096), 8),
]


@pytest.mark.parametrize("name,algo,p,n", F32_CASES, ids=[c[0] for c in F32_CASES])
def test_fp32_philox_vs_oracle_bit_exact(name, algo, p, n):
    from oracle import c_oracle
    p = full_params(dict(p, algorithm=algo))
    L = p["L"]
    _, S0, Q0 = _init(p, 7 + L, "fp32")
    eng = _engine(p, seeds=4242, precision="fp32")
    _assert_k_step(eng)
    assert ("fp32 R" in eng.describe()) == ("fracR" in name), eng.describe()
    eng.set_state(S0, np.zeros((L, L)), Q0)
    eng.step(n)
    sim = c_oracle.Sim(p, S0, np.zeros((L, L)), Q0, "fp32", seed=4242)
    rows_o = sim.run(n)
    _compare(eng, sim, rows_o, "fp32", n)
    eng.close()


# ------------------------------------------------------------------ c. fp32, replayed pairs
@pytest.mark.parametrize("algo,p", [("sarsa", dict(C1, L=131)), ("double_qlearning", dict(C2, L=131))],
                         ids=["sarsa", "double_qlearning"])
def test_fp32_replay_pairs_vs_oracle(algo, p):
    """The REPLAY instantiation of k_step: SARSA's three pairs, Double Q's two (u of pair 1 picks the table)."""
    from oracle import c_oracle
    p = full_params(dict(p, algorithm=algo))
    L, n = p["L"], 30
    rs, S0, Q0 = _init(p, 31, "fp32")
    u, b = _draw_pairs(rs, algo, n, L)
    eng = _engine(p, precision="fp32")
    _assert_k_step(eng)
    eng.set_state(S0, np.zeros((L, L)), Q0)
    _arm(eng, u, b)
    eng.step(n)
    sim = c_oracle.Sim(p, S0, np.zeros((L, L)), Q0, "fp32")
    rows_o = sim.run(n, lambda t, L_: (u[t - 1], b[t - 1]))
    _compare(eng, sim, rows_o, "fp32", n)
    eng.close()


# ------------------------------------------------------------------ d. epsilon edges
@pytest.mark.parametrize("algo", RULES)
def test_epsilon_one_explores_everywhere(algo):
    """epsilon = 1: threshold 2^24, every select and every SARSA next action is a random draw."""
    from oracle import c_oracle
    p = full_params(dict(C1, L=75, epsilon=1.0, epsilon_decay=1.0, algorithm=algo))
    L, n = p["L"], 20
    assert c_oracle.thr24(1.0) == 1 << 24
    _, S0, Q0 = _init(p, 5, "fp32")
    eng = _engine(p, seeds=77, precision="fp32")
    _assert_k_step(eng)
    eng.set_state(S0, np.zeros((L, L)), Q0)
    eng.step(n)
    sim = c_oracle.Sim(p, S0, np.zeros((L, L)), Q0, "fp32", seed=77)
    _compare(eng, sim, sim.run(n), "fp32", n)
    eng.close()


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
@pytest.mark.parametrize("algo", ["sarsa", "expected_sarsa"])
def test_fast_epsilon_decay_across_chunks(algo, precision):
    """epsilon 0.9 halving into epsilon_min = 0.05 within the run: every iteration of the first five
    has its own epsilon, so the policy of the next state (SARSA's threshold, Expected SARSA's
    probabilities) must take the row of the iteration being finished.  Run in chunks of 3 + 9 + 8,
    so that the rows restart at every chunk; fp64 with replayed draws re-armed per chunk."""
    from oracle import c_oracle
    p = full_params(dict(C1, L=97, epsilon=0.9, epsilon_decay=0.5, epsilon_min=0.05, algorithm=algo))
    L, chunks = p["L"], (3, 9, 8)
    n = sum(chunks)
    rs, S0, Q0 = _init(p, 12, precision)
    u, b = _draw_pairs(rs, algo, n, L)
    eng = _engine(p, seeds=5, precision=precision)
    _assert_k_step(eng)
    eng.set_state(S0, np.zeros((L, L)), Q0)
    rows, t0 = [], 0
    for c in chunks:
        if precision == "fp64":
            _arm(eng, u[t0:t0 + c], b[t0:t0 + c])
        eng.step(c)
        rows.append(eng.stats()[1:])
        t0 += c
    sim = c_oracle.Sim(p, S0, np.zeros((L, L)), Q0, precision, seed=5)
    rows_o = sim.run(n, (lambda t, L_: (u[t - 1], b[t - 1])) if precision == "fp64" else None)
    assert eng.status().epsilon == sim.eps == 0.05
    S, R, Q = eng.get_state()
    rows = np.vstack(rows)
    assert np.array_equal(S, sim.S)
    assert np.array_equal(R, sim.R.astype(np.float64))
    assert np.array_equal(Q, sim.Q.astype(np.float64))
    assert np.array_equal(rows[:, INTS], rows_o[:, INTS])
    np.testing.assert_allclose(rows[:, 30], rows_o[:, 30], rtol=1e-6 if precision == "fp32" else 1e-9)


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
@pytest.mark.parametrize("algo", ["sarsa", "expected_sarsa"])
def test_greedy_sarsa_equals_q_learning(monkeypatch, algo, precision):
    """epsilon = epsilon_min = 0: SARSA's next action is the greedy one and Expected SARSA puts all
    weight on it, so both reduce to Q-learning's max.  Q-learning runs k_step_lean, the rule k_step
    (L = 100: no fast path, SPGG_NO_RESIDENT: no resident path), so this also compares the kernels."""
    monkeypatch.setenv("SPGG_NO_RESIDENT", "1")
    L, n = 100, 30
    outs = []
    for rule in ("qlearning", algo):
        p = full_params(dict(C1, L=L, epsilon=0.0, epsilon_min=0.0, algorithm=rule))
        _, S0, Q0 = _init(p, 8, precision)
        eng = _engine(p, seeds=5, precision=precision)
        assert ("k_step_lean" in eng.describe()) == (rule == "qlearning"), eng.describe()
        if rule != "qlearning":
            _assert_k_step(eng)
        eng.set_state(S0, np.zeros((L, L)), Q0)
        eng.step(n)
        st = eng.status()
        assert st.iteration == n and st.stopped_at == -1     # the run did not stop early
        outs.append(eng.get_state() + (eng.stats()[1:],))
        eng.close()
    (Sq, Rq, Qq, rq), (Ss, Rs, Qs, rs_) = outs
    assert 0 < rq[-1, 3] < L * L
    assert np.array_equal(Sq, Ss) and np.array_equal(Rq, Rs)
    assert np.array_equal(Qq, Qs), f"{(Qq != Qs).sum()} Q mismatches"
    assert np.array_equal(rq[:, INTS], rs_[:, INTS])
    assert np.array_equal(rq[:, 33], rs_[:, 33])


# ------------------------------------------------------------------ e. invariances
@pytest.mark.parametrize("algo", RULES)
def test_batched_replicas_equal_single_runs(monkeypatch, algo):
    """Replicas batched in one launch == separate runs, with their own r and influence factor
    (Double Q-learning: 8 Q values per site and replica)."""
    monkeypatch.setenv("SPGG_NO_RESIDENT", "1")
    L, n = 100, 30
    plist = [full_params(dict(C1, L=L, r=r, influence_factor=k, algorithm=algo))
             for r, k in ((3.0, 1.0), (3.6, 0.0), (5.0, 2.0))]
    nq = 8 if algo == "double_qlearning" else 4
    rs = np.random.RandomState(1)
    init = [(rs.randint(0, 2, (L, L)), rs.uniform(-0.01, 0.01, (L, L, nq))) for _ in plist]
    eng = _engine(plist, seeds=[10, 11, 12], precision="fp32")
    assert eng.nq == nq
    _assert_k_step(eng)
    for i, (S0, Q0) in enumerate(init):
        eng.set_state(S0, np.zeros((L, L)), Q0, replica=i)
    eng.step(n)
    for i, (S0, Q0) in enumerate(init):
        single = _engine(plist[i], seeds=10 + i, precision="fp32")
        single.set_state(S0, np.zeros((L, L)), Q0)
        single.step(n)
        for a, b in zip(eng.get_state(i), single.get_state()):
            assert np.array_equal(a, b)
        assert np.array_equal(eng.stats(i), single.stats())
        single.close()
    eng.close()


@pytest.mark.parametrize("algo", RULES)
def test_early_exit_under_td_rules(algo):
    """spgg.py:405 under every TD rule: once the lattice is uniform the loop breaks before acting."""
    from oracle import spgg_numpy
    L = 8
    p = full_params(dict(C1, L=L, epsilon=0.0, epsilon_min=0.0, iterations=10, algorithm=algo))
    # every site prefers to defect in both states -> after iteration 1 all D -> iteration 2 breaks
    Q1 = np.zeros((L, L, 2, 2))
    Q1[..., 1] = 1.0
    Q0 = np.stack([Q1, Q1], axis=2) if algo == "double_qlearning" else Q1
    S0 = np.random.RandomState(0).randint(0, 2, (L, L))
    pairs = PAIRS[algo]
    u = np.full((10, pairs, L, L), 0.5)
    b = np.zeros((10, pairs, L, L), np.uint8)
    eng = _engine(p, precision="fp64")
    _assert_k_step(eng)
    eng.set_state(S0, np.zeros((L, L)), Q0)
    _arm(eng, u, b)
    eng.step(10)
    st = eng.status()
    assert st.stopped_at == 1 and st.iteration == 1
    if algo == "sarsa":
        draws = lambda t, L_: tuple(x for k in range(3) for x in (u[t - 1, k], b[t - 1, k]))  # noqa: E731
    elif algo == "double_qlearning":
        draws = lambda t, L_: (u[t - 1, 0], b[t - 1, 0], u[t - 1, 1])  # noqa: E731
    else:
        draws = lambda t, L_: (u[t - 1, 0], b[t - 1, 0])  # noqa: E731
    q0_np = (Q1.copy(), Q1.copy()) if algo == "double_qlearning" else Q1
    ref = spgg_numpy.simulate(p, S0, np.zeros((L, L)), q0_np, draws)
    S, R, Q = eng.get_state()
    assert np.array_equal(S, ref["Sn_final"]) and np.array_equal(R, ref["R_final"])
    if algo == "double_qlearning":
        assert np.array_equal(Q[:, :, 0], ref["q1_final"]) and np.array_equal(Q[:, :, 1], ref["q2_final"])
    else:
        assert np.array_equal(Q, ref["q_final"])
    assert len(ref["epsilon_history_final"]) == 1 and len(ref["coop_rate_history"]) == 2
    eng.close()
