"""The unmodified reference against the oracle restatements, the drop-in and the committed
golden fixtures.  Tests that execute the reference (the copy ``oracle/ref_harness.py`` finds, run
with h5py/matplotlib stubs) are skipped where no copy is present; the others compare with what
the fixtures recorded from it."""
import json
import os

import numpy as np
import pytest

from helpers import full_params, load_golden

from oracle import ref_harness

needs_ref = pytest.mark.skipif(not ref_harness.reference_available(),
                               reason="/root/reference not present")
QLEARNING_GOLDEN = ["c1_rep_m1", "c2_act_m2", "rep_m2_r36", "act_m1_k0", "ctor_defaults", "odd_L_fracR"]


@pytest.mark.parametrize("name", ["c1_rep_m1", "c2_act_m2", "rep_m2_r36"])
def test_reference_run_equals_oracles(golden_dir, name):
    """Both oracles against a run the reference recorded: reputation state M=1 r=3 kappa=1,
    action state M=2 r=4 kappa=1, reputation state M=2 r=3.6 kappa=0.5.  S, R, Q bit for bit, and
    every series the run wrote that the NumPy oracle assembles."""
    from oracle import c_oracle, spgg_numpy
    z, params = load_golden(golden_dir, name)
    p = full_params(params)
    L, n = p["L"], int(z["u"].shape[0])
    assert n == params["iterations"]
    draws = lambda t, L_: (z["u"][t - 1], z["b"][t - 1])
    r0 = np.zeros((L, L))                       # spgg.py:129
    out = spgg_numpy.simulate(p, z["s0"].astype(np.int64), r0, z["q0"], draws)
    assert np.array_equal(out["Sn_final"], z["s_final"])
    assert np.array_equal(out["R_final"], z["r_final"])
    assert np.array_equal(out["q_final"], z["q_final"])
    series = [k[3:] for k in z.files if k.startswith("ds_") and k[3:] in out]
    assert {"coop_rate_history", "switch_C_to_D", "neighbor_influence_percent",
            "best_neighbor_second_order_percent", "reputation_reward_ratio"} <= set(series)
    for key in series:
        assert np.array_equal(out[key], z["ds_" + key], equal_nan=True), key
    sim = c_oracle.Sim(p, z["s0"], r0, z["q0"], "fp64")
    sim.run(n, draws)
    assert np.array_equal(sim.S, z["s_final"])
    assert np.array_equal(sim.R, z["r_final"])
    assert np.array_equal(sim.Q, z["q_final"])


def test_reconstructed_legacy_stream_is_what_the_reference_consumes(golden_dir):
    """The ctor draws and per-step draws the reference recorded in each Q-learning fixture, for
    the fixture's pinned seed."""
    from oracle import spgg_numpy
    for name in QLEARNING_GOLDEN:
        z, params = load_golden(golden_dir, name)
        L, n = params["L"], int(z["u"].shape[0])
        Q0, S0, draws = spgg_numpy.legacy_draws(int(z["seed"]), L)
        assert np.array_equal(Q0, z["q0"]) and np.array_equal(S0, z["s0"]), name
        for t in range(1, n + 1):
            u, b = draws(t, L)
            assert np.array_equal(u, z["u"][t - 1]) and np.array_equal(b, z["b"][t - 1]), (name, t)


@pytest.mark.reference
@needs_ref
def test_committed_golden_fixture_is_reproducible(golden_dir):
    """Re-run the reference for one fixture and compare with what is committed."""
    z, params = load_golden(golden_dir, "c1_rep_m1")
    ref = ref_harness.run_reference(int(z["seed"]), **params)
    assert np.array_equal(ref["q_final"], z["q_final"])
    assert np.array_equal(ref["s_final"], z["s_final"])
    assert np.array_equal(ref["u"], z["u"])
    shapes = json.loads(str(z["dataset_shapes"]))
    assert sorted(shapes) == sorted(ref["datasets"])


@pytest.mark.reference
@needs_ref
def test_dropin_class_has_the_reference_signature_and_exports():
    import inspect
    import spgg_b200
    ref_model = ref_harness.import_reference()
    ref_sig = inspect.signature(ref_model.SPGG.__init__)
    our_sig = inspect.signature(spgg_b200.SPGG.__init__)
    assert [(p.name, p.default, p.kind) for p in ref_sig.parameters.values()] == \
           [(p.name, p.default, p.kind) for p in our_sig.parameters.values()]
    for name in ("SPGG", "RLAlgorithm", "QLearning", "SARSA", "ExpectedSARSA", "DoubleQLearning",
                 "create_algorithm"):
        assert hasattr(ref_model, name) and hasattr(spgg_b200, name)
    # attribute surface after construction
    with ref_harness.pinned_seed(5):
        a = ref_model.SPGG(L=10, iterations=3, r=3.0)
    b = spgg_b200.SPGG(L=10, iterations=3, r=3.0, seed=5)
    assert np.array_equal(a.q_table, b.q_table) and np.array_equal(a._Sn, b._Sn)
    for attr in ("R", "params", "folder", "snapshot_iters", "track_positions", "normlize_max",
                 "normlize_min", "reward_weight_rep", "algorithm", "cache", "it_records",
                 "epsilon_history", "rep_avg_history", "q_history"):
        assert hasattr(a, attr) and hasattr(b, attr), attr
    for k, v in a.params.items():
        if k in ("S_in_one",):
            continue
        assert k in b.params, k


@pytest.mark.reference
@needs_ref
def test_runner_folder_name_equals_reference():
    import importlib
    from spgg_b200 import runner
    ref_harness.import_reference()
    ref_runner = importlib.import_module("src.experiments.runner")
    for args in [(3.0, 1.0, False, 0.8, 0.95, 1.0), (3.6, 0.0, True, 0.1, 1.0, 0.5, "action"),
                 (5, 2, True, 0.8, 0.9, 0.25, "reputation", "double_qlearning")]:
        assert runner.get_folder_name(*args) == ref_runner.get_folder_name(*args)


def test_double_q_ctor_draw_order_equals_reference(golden_dir):
    """spgg.py:121-127: uniform q_table (discarded), then table 1, table 2, then randint S - the
    tables and strategies the reference's ctor drew in the Double Q-learning fixtures."""
    import spgg_b200
    for name in ("doubleq_rep_m1", "doubleq_act_m2"):
        z, params = load_golden(golden_dir, name)
        b = spgg_b200.SPGG(**params, seed=int(z["seed"]))
        assert np.array_equal(b.algorithm.q_table_1, z["q1_0"]), name
        assert np.array_equal(b.algorithm.q_table_2, z["q2_0"]), name
        assert np.array_equal(b.q_table, z["q0"]) and np.array_equal(b._Sn, z["s0"]), name
