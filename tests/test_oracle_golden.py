"""CPU tests of the oracle (test infrastructure) against the golden vectors recorded
from the executed reference (``oracle/make_golden.py``), and of the host-side series
assembly on the oracle's statistic rows.  Bit-exact for S, R, Q and integer series."""
import numpy as np
import pytest

from helpers import full_params, load_golden

GOLDEN = ["c1_rep_m1", "c2_act_m2", "rep_m2_r36", "act_m1_k0", "ctor_defaults", "odd_L_fracR"]

FLOAT_SERIES = (
    "it_records_final", "rep_avg_history_final", "epsilon_history_final",
    "neighbor_influence_percent", "payoff_component_history", "rep_component_history",
    "best_neighbor_second_order_percent", "reputation_reward_ratio", "avg_reward_C_history",
    "avg_reward_D_history", "group_comp_d0_history", "group_comp_d3_history",
    "group_comp_d5_history", "avg_q_s0_c_history", "avg_q_s1_d_history",
    "cooperators_q_s0_d_history", "defectors_q_s1_c_history")


def _draws(z):
    return lambda t, L: (z["u"][t - 1], z["b"][t - 1])


@pytest.mark.parametrize("name", GOLDEN)
def test_numpy_oracle_reproduces_reference_bit_for_bit(golden_dir, name):
    from oracle import spgg_numpy
    z, p = load_golden(golden_dir, name)
    p = full_params(p)
    L, n = p["L"], int(z["u"].shape[0])
    out = spgg_numpy.simulate(dict(p, iterations=n), z["s0"].astype(np.int64), np.zeros((L, L)),
                              z["q0"], _draws(z))
    assert np.array_equal(out["Sn_final"], z["s_final"])
    assert np.array_equal(out["R_final"], z["r_final"])
    assert np.array_equal(out["q_final"], z["q_final"])
    for key in ("coop_rate_history", "switch_C_to_D", "switch_D_to_C", "epsilon_history_final"):
        assert np.array_equal(out[key], z["ds_" + key]), key
    for key in FLOAT_SERIES:
        if "ds_" + key in z.files:
            # same NumPy reductions on the same arrays: equal to the last bit
            assert np.array_equal(out[key], z["ds_" + key], equal_nan=True), key
    if "ds_R_snapshot_10" in z.files and 10 in out["snapshots"]:
        assert np.array_equal(out["snapshots"][10][0], z["ds_R_snapshot_10"])
        assert np.array_equal(out["snapshots"][10][1], z["ds_Sn_snapshot_10"])


TD_GOLDEN = ["sarsa_rep_m1", "sarsa_act_m2", "expsarsa_rep_m2", "expsarsa_act_m1"]
DQ_GOLDEN = ["doubleq_rep_m1", "doubleq_act_m2"]


@pytest.mark.parametrize("name", GOLDEN + TD_GOLDEN + DQ_GOLDEN)
def test_c_oracle_fp64_reproduces_reference_bit_for_bit(golden_dir, name):
    """Every TD rule: S, R, Q (both Double-Q tables and their mean) and the integer series."""
    from oracle import c_oracle
    z, p = load_golden(golden_dir, name)
    p = full_params(p)
    L, n = p["L"], int(z["u"].shape[0])
    dq = p.get("algorithm") == "double_qlearning"
    Q0 = np.stack([z["q1_0"], z["q2_0"]], axis=2) if dq else z["q0"]
    sim = c_oracle.Sim(p, z["s0"], np.zeros((L, L)), Q0, "fp64")
    rows = sim.run(n, lambda t, L_: (z["u"][t - 1], z["b"][t - 1]))
    assert rows.shape[0] == n
    assert np.array_equal(sim.S, z["s_final"])
    assert np.array_equal(sim.R, z["r_final"])
    if dq:
        assert np.array_equal(sim.Q[:, :, 0], z["q1_final"])
        assert np.array_equal(sim.Q[:, :, 1], z["q2_final"])
    assert np.array_equal(sim.q_combined, z["q_final"])
    ST = c_oracle.ST
    assert np.array_equal(rows[:, ST["N_CD"]].astype(np.int64), z["ds_switch_C_to_D"])
    assert np.array_equal(rows[:, ST["N_DC"]].astype(np.int64), z["ds_switch_D_to_C"])
    assert np.array_equal(rows[:, ST["NC_OLD"]] / (L * L), z["ds_coop_rate_history"])


@pytest.mark.parametrize("name", GOLDEN)
def test_series_assembly_from_stat_rows_matches_reference_datasets(golden_dir, name):
    """Host logic: statistic rows (sums) -> the reference's HDF5 series.  Rows come from the
    C oracle (same row layout as the device); integer series exact, float means within
    1e-9 relative (the reference uses NumPy's pairwise sums, the rows are plain sums)."""
    import spgg_b200
    from spgg_b200 import series
    from oracle import c_oracle
    z, p = load_golden(golden_dir, name)
    p = full_params(p)
    L, n = p["L"], int(z["u"].shape[0])
    sim = c_oracle.Sim(p, z["s0"], np.zeros((L, L)), z["q0"], "fp64")
    rows = sim.run(n, _draws(z))
    ser = series.assemble(rows, rows[:, spgg_b200._lib.ST_SUM_R], L * L, p, p["epsilon"])
    for key in ("switch_C_to_D", "switch_D_to_C", "coop_rate_history", "epsilon_history_final"):
        assert np.array_equal(ser[key], z["ds_" + key]), key
        assert ser[key].dtype == z["ds_" + key].dtype, key
    for key in FLOAT_SERIES:
        if "ds_" + key in z.files:
            assert ser[key].shape == z["ds_" + key].shape, key
            np.testing.assert_allclose(ser[key], z["ds_" + key], rtol=1e-9, atol=1e-12,
                                       equal_nan=True, err_msg=key)


def test_golden_files_carry_the_full_dataset_contract(golden_dir):
    """The reference writes ~50 datasets (SURVEY.md section 5); the fixture lists them."""
    import json
    z, p = load_golden(golden_dir, "c1_rep_m1")
    names = set(str(s) for s in z["dataset_names"])
    shapes = json.loads(str(z["dataset_shapes"]))
    for k in ("coop_rate_history", "Sn_final", "R_final", "cluster_sizes", "rep_hist_final",
              "rep_bins_final", "switch_C_to_D", "avg_q_s0_c_history",
              "cooperators_q_s1_d_history", "group_comp_d5_history"):
        assert k in names
    assert shapes["Sn_final"][0] == "int64" and shapes["switch_C_to_D"][0] == "int64"
    L = p["L"]
    for a, b in ((L // 2, L // 2), (L // 4, L // 4), (3 * L // 4, 3 * L // 4)):
        assert shapes[f"q_c_pos_{a}_{b}_final"][1] == [0]     # never appended to, spgg.py:345


# ------------------------------------------------------------------ known answers
def test_payoff_known_answers():
    """spgg.py:230-259, 373-377: all-C and all-D lattices, and a single defector."""
    from oracle import spgg_numpy
    r, c, cost = 3.0, 1, 1
    L = 8
    allC = np.zeros((L, L), np.int64)
    P = spgg_numpy.normalised_payoff(allC, r, c, cost)
    # every group has 5 cooperators: 5 * (r - cost) = 10; (10 - (r-5)) / (4r - (r-5))
    assert np.allclose(P, (5 * (r - cost) - (r - 5)) / (4 * r - (r - 5)))
    allD = np.ones((L, L), np.int64)
    P = spgg_numpy.normalised_payoff(allD, r, c, cost)
    assert np.allclose(P, (0 - (r - 5)) / (4 * r - (r - 5)))
    S = np.zeros((L, L), np.int64)
    S[3, 3] = 1
    P = spgg_numpy.normalised_payoff(S, r, c, cost)
    # the defector sits in 5 groups of 4 cooperators each and pays nothing
    assert np.isclose(P[3, 3], (5 * r * 4 / 5 - (r - 5)) / (4 * r - (r - 5)))
    # a site two steps away shares one group (centred between them) with the defector
    assert np.isclose(P[3, 5], ((4 * r + r * 4 / 5) - 5 * cost - (r - 5)) / (4 * r - (r - 5)))


def test_state_encoding_and_offsets():
    """spgg.py:281-310 + the np.roll sign convention (neighbour k of (i,j) = (i-dx, j-dy))."""
    from oracle import spgg_numpy
    assert spgg_numpy.OFFSETS_M1 == ((1, 0), (-1, 0), (0, 1), (0, -1))
    assert len(spgg_numpy.OFFSETS_M2) == 12 and spgg_numpy.OFFSETS_M2[4] == (2, 0)
    L = 7
    R = np.zeros((L, L))
    R[2, 2] = 1.0
    s1 = spgg_numpy.state_of(R, None, 1, "reputation")
    assert s1.sum() == 5 and s1[2, 2] and s1[1, 2] and s1[3, 2] and s1[2, 1] and s1[2, 3]
    s2 = spgg_numpy.state_of(R, None, 2, "reputation")
    assert s2.sum() == 13 and s2[0, 2] and s2[1, 1] and not s2[0, 1]
    S = np.array([[0, 1], [1, 0]])
    assert np.array_equal(spgg_numpy.state_of(None, S, 1, "action"), (S == 0).astype(int))
    X = np.arange(L * L).reshape(L, L)
    assert spgg_numpy.at(X, 1, 0)[3, 4] == X[2, 4] and spgg_numpy.at(X, 0, -1)[3, 6] == X[3, 0]


def test_tie_rules():
    """Greedy tie -> action 0 (algorithms.py:107, np.argmax first max); best-neighbour tie ->
    first offset in the reference order (spgg.py:479-485)."""
    from oracle import spgg_numpy
    L = 6
    p = full_params(dict(L=L, r=3.0, cost=1, alpha=0.5, influence_factor=1.0,
                         use_second_order=False, reward_weight_payoff=1.0, rep_gain_C=1.0))
    S = np.zeros((L, L), np.int64)
    R = np.zeros((L, L))
    Q = np.zeros((L, L, 2, 2))
    u = np.ones((L, L))            # never explore
    b = np.ones((L, L), np.uint8)
    S2, R2, Q2, st = spgg_numpy.qlearning_step(S, R, Q, 0.5, u, b, p)
    assert (S2 == 0).all()         # all ties -> cooperate
    assert (R2 == 1.0).all()


def test_philox_known_answer():
    """Philox4x32-10 known-answer vectors (Random123 kat_vectors)."""
    from oracle import c_oracle
    out = c_oracle.philox([0, 0, 0, 0], [0, 0])
    assert [int(x) for x in out] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    out = c_oracle.philox([0xffffffff] * 4, [0xffffffff] * 2)
    assert [int(x) for x in out] == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    out = c_oracle.philox([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0])
    assert [int(x) for x in out] == [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_threshold_and_reward_table():
    from oracle import c_oracle
    assert c_oracle.thr24(0.5) == 1 << 23
    assert c_oracle.thr24(0.0) == 0 and c_oracle.thr24(1.0) == 1 << 24
    assert c_oracle.thr24(0.01) == int(np.ceil(0.01 * 2 ** 24))
    p = full_params(dict(L=8, r=3.0, cost=1, reward_weight_payoff=0.95))
    tab = c_oracle.reward_table(p)
    # code = SigmaN<<2 | C_old<<1 | coop_new; all-cooperator site that cooperates again
    sn, C, coop = 25, 1, 1
    P = ((3.0 * sn / 5 - 5 * 1.0) - (3.0 - 5)) / (4 * 3.0 - (3.0 - 5))
    assert np.isclose(tab[(sn << 2) | (C << 1) | coop], 0.95 * P + (1 - 0.95) * 0.5, rtol=1e-6)


def test_c_oracle_fp32_follows_fp64_on_short_horizons():
    """The throughput arithmetic (fp32 Q, exact-count reward table) is not bit-compatible
    with the reference; on a short horizon with replayed draws the strategy lattice still
    coincides (SURVEY.md section 4: divergence starts at step 2..500) - here 3 steps."""
    from oracle import c_oracle
    L, n = 32, 3
    p = full_params(dict(L=L, r=3.0, cost=1, alpha=0.8, epsilon_decay=0.99, influence_factor=1.0,
                         use_second_order=False, reward_weight_payoff=0.95, rep_gain_C=1.0))
    rs = np.random.RandomState(11)
    Q0 = rs.uniform(-0.01, 0.01, (L, L, 2, 2))
    S0 = rs.randint(0, 2, (L, L))
    u = rs.rand(n, L, L)
    b = rs.randint(0, 2, (n, L, L)).astype(np.uint8)
    a = c_oracle.Sim(p, S0, np.zeros((L, L)), Q0, "fp64")
    c = c_oracle.Sim(p, S0, np.zeros((L, L)), Q0, "fp32")
    a.run(n, lambda t, L_: (u[t - 1], b[t - 1]))
    c.run(n, lambda t, L_: (u[t - 1], b[t - 1]))
    assert (a.S != c.S).mean() < 0.02
    np.testing.assert_allclose(c.Q, a.Q, rtol=0, atol=2e-2)


@pytest.mark.parametrize("algo", ["sarsa", "expected_sarsa", "double_qlearning"])
def test_c_oracle_fp32_td_rules_follow_fp64_on_short_horizons(algo):
    """As above for the other TD rules, with the draw pairs each consumes (SARSA three, Double Q
    two): the fp32 restatement of k_step stays within the fp64 reference order on 3 steps."""
    from oracle import c_oracle
    L, n = 32, 3
    p = full_params(dict(L=L, r=3.0, cost=1, alpha=0.8, epsilon_decay=0.99, influence_factor=1.0,
                         use_second_order=False, reward_weight_payoff=0.95, rep_gain_C=1.0,
                         algorithm=algo))
    pairs = c_oracle.PAIRS[c_oracle.ALGOS[algo]]
    rs = np.random.RandomState(11)
    Q0 = rs.uniform(-0.01, 0.01, (L, L, 2, 2, 2) if algo == "double_qlearning" else (L, L, 2, 2))
    S0 = rs.randint(0, 2, (L, L))
    u = rs.rand(n, pairs, L, L)
    b = rs.randint(0, 2, (n, pairs, L, L)).astype(np.uint8)
    a = c_oracle.Sim(p, S0, np.zeros((L, L)), Q0, "fp64")
    c = c_oracle.Sim(p, S0, np.zeros((L, L)), Q0, "fp32")
    a.run(n, lambda t, L_: (u[t - 1], b[t - 1]))
    c.run(n, lambda t, L_: (u[t - 1], b[t - 1]))
    assert (a.S != c.S).mean() < 0.02
    np.testing.assert_allclose(c.Q, a.Q, rtol=0, atol=2e-2)
    assert np.abs(c.Q - a.Q).max() > 0                  # the two arithmetics are distinct
    np.testing.assert_allclose(c.q_combined, a.q_combined, rtol=0, atol=2e-2)


@pytest.mark.parametrize("algo", ["qlearning", "sarsa", "expected_sarsa", "double_qlearning"])
@pytest.mark.parametrize("L,second,state", [(37, False, "reputation"), (37, True, "action"),
                                            (64, True, "reputation"), (64, False, "action")])
def test_c_oracle_fp64_equals_numpy_oracle_for_every_td_rule(algo, L, second, state):
    """oracle_step_f64 restates oracle/spgg_numpy.py (pinned to the reference above) for every TD
    rule: S, R, Q (both Double-Q tables) and the integer series bit for bit, odd and even sides."""
    from oracle import c_oracle, spgg_numpy
    n = 25
    p = full_params(dict(L=L, r=3.6, cost=1, alpha=0.8, epsilon_decay=0.9, influence_factor=0.7,
                         use_second_order=second, state_representation=state,
                         reward_weight_payoff=0.95, rep_gain_C=1.0, algorithm=algo, iterations=n))
    pairs = c_oracle.PAIRS[c_oracle.ALGOS[algo]]
    rs = np.random.RandomState(L + 7 * pairs + second)
    Q0 = rs.uniform(-0.01, 0.01, (L, L, 2, 2, 2) if algo == "double_qlearning" else (L, L, 2, 2))
    S0 = rs.randint(0, 2, (L, L))
    u = rs.rand(n, pairs, L, L)
    b = rs.randint(0, 2, (n, pairs, L, L)).astype(np.uint8)
    if algo == "sarsa":
        draws = lambda t, L_: tuple(x for k in range(3) for x in (u[t - 1, k], b[t - 1, k]))  # noqa: E731
    elif algo == "double_qlearning":
        draws = lambda t, L_: (u[t - 1, 0], b[t - 1, 0], u[t - 1, 1])  # noqa: E731
    else:
        draws = lambda t, L_: (u[t - 1, 0], b[t - 1, 0])  # noqa: E731
    q0_np = (Q0[:, :, 0], Q0[:, :, 1]) if algo == "double_qlearning" else Q0
    ref = spgg_numpy.simulate(p, S0.astype(np.int64), np.zeros((L, L)), q0_np, draws)
    sim = c_oracle.Sim(p, S0, np.zeros((L, L)), Q0, "fp64")
    rows = sim.run(n, lambda t, L_: (u[t - 1], b[t - 1]))
    assert rows.shape[0] == n == len(ref["switch_C_to_D"])
    assert np.array_equal(sim.S, ref["Sn_final"])
    assert np.array_equal(sim.R, ref["R_final"])
    if algo == "double_qlearning":
        assert np.array_equal(sim.Q[:, :, 0], ref["q1_final"])
        assert np.array_equal(sim.Q[:, :, 1], ref["q2_final"])
    assert np.array_equal(sim.q_combined, ref["q_final"])
    ST = c_oracle.ST
    assert np.array_equal(rows[:, ST["N_CD"]].astype(np.int64), ref["switch_C_to_D"])
    assert np.array_equal(rows[:, ST["N_DC"]].astype(np.int64), ref["switch_D_to_C"])
    assert np.array_equal(rows[:, ST["NC_OLD"]] / (L * L), ref["coop_rate_history"][:n])
    assert np.array_equal(rows[:, ST["GMAX"]], ref["gmax"])
    for k in range(6):
        assert np.array_equal(rows[:, ST["GROUP0"] + k] / (L * L) * 100, ref[f"group_comp_d{k}_history"])
    # the float statistics are plain sums here and NumPy means there
    np.testing.assert_allclose(rows[:, ST["SUM_NI"]] / (L * L), ref["neighbor_influence_percent"],
                               rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(rows[:, ST["SUM_Q"]] / (L * L), ref["avg_q_s0_c_history"], rtol=1e-9,
                               atol=1e-15)
    assert len(np.unique(sim.S)) == 2                  # the run did not end uniform


def test_philox_streams_of_the_td_rules():
    """The Philox words the step functions draw for a site are those of the documented counters
    (j/4, i, t, stream), word j%4 - the counters k_step's philox_row forms - and the fp32 step
    acts on them: with epsilon = 1 every action is word0 & 1, and Double Q updates table 1 exactly
    where (word1 >> 8) < 2^23."""
    from oracle import c_oracle
    seed = 0x123456789ABCDEF0
    key = [seed & 0xFFFFFFFF, seed >> 32]
    for (t, i, j) in ((1, 0, 0), (7, 5, 13), (3, 36, 31), (2, 4095, 4094)):
        for stream in (0, 1, 2):
            want = int(c_oracle.philox([j // 4, i, t, stream], key)[j % 4])
            assert c_oracle.site_word(seed, t, stream, i, j) == want, (t, i, j, stream)
    L = 37
    p = full_params(dict(L=L, r=3.0, cost=1, epsilon=1.0, epsilon_decay=1.0, influence_factor=0.0,
                         state_representation="action", algorithm="double_qlearning"))
    rs = np.random.RandomState(4)
    Q0 = rs.uniform(-0.01, 0.01, (L, L, 2, 2, 2)).astype(np.float32)
    S0 = rs.randint(0, 2, (L, L))
    sim = c_oracle.Sim(p, S0, np.zeros((L, L)), Q0, "fp32", seed=seed)
    sim.step()
    w0 = np.array([[c_oracle.site_word(seed, 1, 0, i, j) for j in range(L)] for i in range(L)], np.uint64)
    w1 = np.array([[c_oracle.site_word(seed, 1, 1, i, j) for j in range(L)] for i in range(L)], np.uint64)
    assert np.array_equal(sim.S, (w0 & 1).astype(np.uint8))
    upd1 = (w1 >> 8) < (1 << 23)
    changed1 = (sim.Q[:, :, 0] != Q0[:, :, 0]).any(axis=(2, 3))
    changed2 = (sim.Q[:, :, 1] != Q0[:, :, 1]).any(axis=(2, 3))
    assert np.array_equal(changed1, upd1) and np.array_equal(changed2, ~upd1)


def test_early_exit_series_lengths():
    """Uniform lattice: the loop records the pre-action entries and breaks (spgg.py:405):
    T_c = T + 1."""
    from oracle import spgg_numpy
    L = 8
    p = full_params(dict(L=L, iterations=5))
    out = spgg_numpy.simulate(p, np.zeros((L, L), np.int64), np.zeros((L, L)),
                              np.zeros((L, L, 2, 2)), lambda t, L_: (None, None))
    assert len(out["coop_rate_history"]) == 1 and "epsilon_history_final" not in out


def _td_draws(z):
    u, b = z["u"], z["b"]
    if u.ndim == 4:      # (n, pairs, L, L): SARSA draws three pairs per iteration
        return lambda t, L: tuple(x for k in range(u.shape[1]) for x in (u[t - 1, k], b[t - 1, k]))
    return lambda t, L: (u[t - 1], b[t - 1])


@pytest.mark.parametrize("name", TD_GOLDEN)
def test_numpy_oracle_other_td_rules_reproduce_reference(golden_dir, name):
    """SARSA (three draw pairs per iteration, spgg.py:410,433,452) and Expected SARSA
    (algorithms.py:197-234) against the executed reference, bit for bit."""
    from oracle import spgg_numpy
    z, p = load_golden(golden_dir, name)
    p = full_params(p)
    L, n = p["L"], int(z["u"].shape[0])
    assert (z["u"].ndim == 4 and z["u"].shape[1] == 3) == (p["algorithm"] == "sarsa")
    out = spgg_numpy.simulate(dict(p, iterations=n), z["s0"].astype(np.int64), np.zeros((L, L)),
                              z["q0"], _td_draws(z))
    assert np.array_equal(out["Sn_final"], z["s_final"])
    assert np.array_equal(out["R_final"], z["r_final"])
    assert np.array_equal(out["q_final"], z["q_final"])
    for key in ("coop_rate_history", "switch_C_to_D", "neighbor_influence_percent",
                "avg_q_s0_c_history", "cooperators_q_s0_d_history"):
        assert np.array_equal(out[key], z["ds_" + key], equal_nan=True), key


@pytest.mark.parametrize("name", ["doubleq_rep_m1", "doubleq_act_m2"])
def test_numpy_oracle_double_q_reproduces_reference(golden_dir, name):
    """Double Q-learning (algorithms.py:237-341; two tables, table choice drawn per site,
    neighbour term added to both, spgg.py:498-505) against the executed reference."""
    from oracle import spgg_numpy
    z, p = load_golden(golden_dir, name)
    p = full_params(p)
    L, n = p["L"], int(z["u"].shape[0])
    u, b = z["u"], z["b"]
    assert np.array_equal(z["q0"], (z["q1_0"] + z["q2_0"]) / 2)
    out = spgg_numpy.simulate(dict(p, iterations=n), z["s0"].astype(np.int64), np.zeros((L, L)),
                              (z["q1_0"], z["q2_0"]), lambda t, L_: (u[t - 1, 0], b[t - 1, 0], u[t - 1, 1]))
    assert np.array_equal(out["Sn_final"], z["s_final"])
    assert np.array_equal(out["R_final"], z["r_final"])
    assert np.array_equal(out["q1_final"], z["q1_final"]) and np.array_equal(out["q2_final"], z["q2_final"])
    assert np.array_equal(out["q_final"], z["q_final"])
    for key in ("coop_rate_history", "switch_C_to_D", "neighbor_influence_percent", "avg_q_s0_c_history"):
        assert np.array_equal(out[key], z["ds_" + key], equal_nan=True), key


@pytest.mark.parametrize("r,cost,L", [(3.0, 1.0, 64), (3.6, 1.0, 37), (1.0, 0.5, 50), (5.0, 1.0, 20)])
def test_payoff_sums_from_integer_counts(r, cost, L):
    """The kernels' statistics row takes the payoff sums per class (spgg.py:381-392) from exact integer
    counts - sum of P over a class = ((r c SigmaN / 5 - 5 cost C n) - lo n) / span, SigmaN the cooperators
    summed over the five groups of a site (csrc/spgg_kernels.cuh: step_epilogue) - instead of summing the
    per-site payoffs of spgg.py:373-377.  The two agree to rounding (the series are compared to 1e-9)."""
    from oracle import spgg_numpy as sn
    rs = np.random.RandomState(int(r * 10) + L)
    for frac in (0.5, 0.05, 0.95):
        S = (rs.rand(L, L) < frac).astype(np.int64)             # 1 = defector
        P = sn.normalised_payoff(S, r, 1, cost)
        C = (S == 0).astype(np.int64)
        N = sn.group_counts(C)
        sigma = sum(sn.at(N, di, dj) for (di, dj) in ((0, 0), (1, 0), (-1, 0), (0, 1), (0, -1)))
        lo, span = r - 5, 4 * r - (r - 5)
        for cls, mask in (("C", C == 1), ("D", C == 0)):
            n = int(mask.sum())
            direct = float(P[mask].sum())
            from_counts = ((r * 1 * float(sigma[mask].sum()) / 5.0 - 5.0 * cost * (cls == "C") * n) - lo * n) / span
            assert abs(direct - from_counts) <= 1e-12 * max(1.0, abs(direct)) * max(1, n) ** 0.5, (cls, direct, from_counts)
