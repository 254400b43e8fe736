"""The C oracle on uploaded start states, against the NumPy restatement of the reference (CPU only).

Every other oracle test starts from R0 = 0 and Q0 uniform in (-0.01, 0.01).  A run resumed from a
checkpoint, or a drop-in run whose user set ``m.R`` by hand, starts elsewhere: with reputations
beyond the clamps (the reference computes the first state from the raw R and clips it only at the
first update), at a zero start below a floor R_min > 0, and with Q tables whose entries tie (the
greedy choice then takes C, and the TD target's max sees equal values).  Here oracle_step_f64 must
equal oracle/spgg_numpy.py bit for bit on those inputs - S, R, Q (both Double-Q tables) and the
integer series - for every TD rule, both neighbour orders and both state modes.  The GPU tests of
the same starts (tests/test_gpu_start_states.py) take the C oracle as their reference."""
import numpy as np
import pytest

from helpers import full_params

RULES = ["qlearning", "sarsa", "expected_sarsa", "double_qlearning"]
GEOMS = [(37, False, "reputation"), (37, True, "action"), (64, True, "reputation"), (64, False, "action")]
R_KINDS = ["inside", "outside", "floor"]
Q_KINDS = ["zero", "ternary"]


def start_state(L, r_kind, q_kind, algo, seed):
    """(params overrides, S0, R0, Q0) of one start: R0 on the integers within the clamps [-10, 10],
    integers in [-40, 40] (most of them beyond the clamps), or 0 under a floor R_min = 2; Q0 all
    zero or drawn from {-0.01, 0, 0.01} (ties in most sites)."""
    rs = np.random.RandomState(seed)
    extra = {}
    if r_kind == "inside":
        R0 = rs.randint(-10, 11, (L, L)).astype(np.float64)
    elif r_kind == "outside":
        R0 = rs.randint(-40, 41, (L, L)).astype(np.float64)
    else:
        extra = dict(R_min=2)
        R0 = np.zeros((L, L))
    shape = (L, L, 2, 2, 2) if algo == "double_qlearning" else (L, L, 2, 2)
    Q0 = np.zeros(shape) if q_kind == "zero" else rs.choice([-0.01, 0.0, 0.01], shape)
    S0 = rs.randint(0, 2, (L, L))
    return extra, S0, R0, Q0


@pytest.mark.parametrize("q_kind", Q_KINDS)
@pytest.mark.parametrize("r_kind", R_KINDS)
@pytest.mark.parametrize("L,second,state", GEOMS, ids=[f"L{g[0]}_m{2 if g[1] else 1}_{g[2][:3]}" for g in GEOMS])
@pytest.mark.parametrize("algo", RULES)
def test_c_oracle_fp64_equals_numpy_oracle_from_uploaded_starts(algo, L, second, state, r_kind, q_kind):
    from oracle import c_oracle, spgg_numpy
    n = 12
    pairs = c_oracle.PAIRS[c_oracle.ALGOS[algo]]
    seed = 1000 * L + 100 * R_KINDS.index(r_kind) + 10 * Q_KINDS.index(q_kind) + 2 * pairs + second
    extra, S0, R0, Q0 = start_state(L, r_kind, q_kind, algo, seed)
    p = full_params(dict(L=L, r=3.6, cost=1, alpha=0.8, epsilon_decay=0.9, influence_factor=0.7,
                         use_second_order=second, state_representation=state, reward_weight_payoff=0.95,
                         rep_gain_C=1.0, algorithm=algo, iterations=n, **extra))
    rs = np.random.RandomState(seed + 1)
    u = rs.rand(n, pairs, L, L)
    b = rs.randint(0, 2, (n, pairs, L, L)).astype(np.uint8)
    if algo == "sarsa":
        draws = lambda t, L_: tuple(x for k in range(3) for x in (u[t - 1, k], b[t - 1, k]))  # noqa: E731
    elif algo == "double_qlearning":
        draws = lambda t, L_: (u[t - 1, 0], b[t - 1, 0], u[t - 1, 1])  # noqa: E731
    else:
        draws = lambda t, L_: (u[t - 1, 0], b[t - 1, 0])  # noqa: E731
    q0_np = (Q0[:, :, 0].copy(), Q0[:, :, 1].copy()) if algo == "double_qlearning" else Q0.copy()
    ref = spgg_numpy.simulate(p, S0.astype(np.int64), R0, q0_np, draws)
    sim = c_oracle.Sim(p, S0, R0, Q0, "fp64")
    rows = sim.run(n, lambda t, L_: (u[t - 1], b[t - 1]))
    assert rows.shape[0] == n == len(ref["switch_C_to_D"])     # the run did not end uniform
    assert np.array_equal(sim.S, ref["Sn_final"]), f"{(sim.S != ref['Sn_final']).sum()} S mismatches"
    assert np.array_equal(sim.R, ref["R_final"]), f"{(sim.R != ref['R_final']).sum()} R mismatches"
    assert sim.R.min() >= p["R_min"] and sim.R.max() <= p["R_max"]   # the first update clipped every site
    if algo == "double_qlearning":
        assert np.array_equal(sim.Q[:, :, 0], ref["q1_final"])
        assert np.array_equal(sim.Q[:, :, 1], ref["q2_final"])
    assert np.array_equal(sim.q_combined, ref["q_final"])
    ST = c_oracle.ST
    # the first row records the uploaded reputations before anything clips them
    assert rows[0, ST["SUM_R"]] == R0.sum()
    np.testing.assert_allclose(rows[:, ST["SUM_R"]] / (L * L), ref["rep_avg_history_final"], rtol=1e-12, atol=1e-12)
    assert np.array_equal(rows[:, ST["N_CD"]].astype(np.int64), ref["switch_C_to_D"])
    assert np.array_equal(rows[:, ST["N_DC"]].astype(np.int64), ref["switch_D_to_C"])
    assert np.array_equal(rows[:, ST["NC_OLD"]] / (L * L), ref["coop_rate_history"][:n])
    assert np.array_equal(rows[:, ST["GMAX"]], ref["gmax"])
    for k in range(6):
        assert np.array_equal(rows[:, ST["GROUP0"] + k] / (L * L) * 100, ref[f"group_comp_d{k}_history"])
    np.testing.assert_allclose(rows[:, ST["SUM_NI"]] / (L * L), ref["neighbor_influence_percent"],
                               rtol=1e-9, atol=1e-12)


def test_the_starts_reach_the_edges_they_are_meant_to():
    """The inputs above do what they are for: 'outside' puts most sites beyond the clamps (and beyond
    the 5-bit bytes [-16, 15] of the int8 fast path), 'floor' starts below R_min, and ternary Q0
    ties the two actions of a state in a third of the entries."""
    _, _, R0, Q0 = start_state(64, "outside", "ternary", "qlearning", 3)
    assert (np.abs(R0) > 10).mean() > 0.5 and ((R0 > 15) | (R0 < -16)).mean() > 0.4
    assert (Q0[..., 0] == Q0[..., 1]).mean() > 0.25
    extra, _, R0, Q0 = start_state(37, "floor", "zero", "sarsa", 3)
    assert extra["R_min"] > 0 and not R0.any() and not Q0.any()
