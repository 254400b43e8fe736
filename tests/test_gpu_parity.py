"""GPU parity tests: the CUDA path (through the C ABI) against the oracle and the
golden vectors recorded from the executed reference.  Bit-exact for S, R and all
integer statistics; Q bit-exact as well (tolerance stated where it is not)."""
import numpy as np
import pytest

from helpers import C1, C2, full_params, legacy_stream, load_golden

pytestmark = pytest.mark.gpu

GOLDEN = ["c1_rep_m1", "c2_act_m2", "rep_m2_r36", "act_m1_k0", "ctor_defaults", "odd_L_fracR"]


def _engine(*a, **k):
    import spgg_b200
    return spgg_b200.Engine(*a, **k)


@pytest.mark.parametrize("name", GOLDEN)
def test_golden_replay_fp64_bit_exact(golden_dir, name):
    """fp64 instantiation + the reference's recorded draws == the reference, bit for bit."""
    import spgg_b200
    from spgg_b200 import series
    z, p = load_golden(golden_dir, name)
    p = full_params(p)
    L, n = p["L"], int(z["u"].shape[0])
    eng = _engine(p, precision="fp64")
    eng.set_state(z["s0"], np.zeros((L, L)), z["q0"])
    eng.set_replay(z["u"], z["b"])
    eng.step(n)
    S, R, Q = eng.get_state()
    assert np.array_equal(S, z["s_final"])
    assert np.array_equal(R, z["r_final"])
    assert np.array_equal(Q, z["q_final"])
    rows = eng.stats()
    ser = series.assemble(rows[1:], rows[:-1, spgg_b200._lib.ST_SUM_R], L * L, p, p["epsilon"])
    for key in ("switch_C_to_D", "switch_D_to_C", "coop_rate_history"):
        assert np.array_equal(ser[key], z["ds_" + key]), key
    for key in [k[3:] for k in z.files if k.startswith("ds_")]:
        if key in ser and ser[key].shape == z["ds_" + key].shape:
            # float statistics: summation order differs from np.sum/np.mean (pairwise)
            np.testing.assert_allclose(ser[key], z["ds_" + key], rtol=1e-9, atol=1e-12,
                                       equal_nan=True, err_msg=key)
    eng.close()


@pytest.mark.parametrize("state", ["reputation", "action"])
@pytest.mark.parametrize("second", [False, True])
@pytest.mark.parametrize("L", [64, 100])
def test_fp64_replay_vs_oracle(state, second, L):
    from oracle import c_oracle
    n = 120
    p = full_params(dict(C1, L=L, use_second_order=second, state_representation=state))
    Q0, S0, u, b = legacy_stream(11 + L, L, n)
    eng = _engine(p, precision="fp64")
    eng.set_state(S0, np.zeros((L, L)), Q0)
    eng.set_replay(u, b)
    eng.step(n)
    S, R, Q = eng.get_state()
    sim = c_oracle.Sim(p, S0, np.zeros((L, L)), Q0, "fp64")
    rows_o = sim.run(n, lambda t, L_: (u[t - 1], b[t - 1]))
    assert np.array_equal(S, sim.S) and np.array_equal(R, sim.R)
    assert np.array_equal(Q, sim.Q)
    rows = eng.stats()[1:]
    ints = [0, 1, 2, 3, 11, 12, 13, 14, 15, 16, 31, 32]
    assert np.array_equal(rows[:, ints], rows_o[:, ints])
    assert np.array_equal(rows[:, 33], rows_o[:, 33])  # gmax is an exact max
    np.testing.assert_allclose(rows[:, 4:11], rows_o[:, 4:11], rtol=1e-10, atol=1e-9)
    # sum of R before the action: recorded by the launch that chooses the action, one row earlier
    np.testing.assert_allclose(eng.stats()[:-1, 17], rows_o[:, 17], rtol=1e-10, atol=1e-9)
    np.testing.assert_allclose(rows[:, 18:31], rows_o[:, 18:31], rtol=1e-9, atol=1e-9)
    eng.close()


@pytest.mark.parametrize("cfg", ["c1", "c2"])
def test_fp64_replay_1000_steps_L200(cfg):
    """north_star: replayed draws, 10^3 steps: S and R bit-exact, Q within 1e-6 relative
    (it is bit-exact)."""
    from oracle import c_oracle
    L, n, chunk = 200, 1000, 250
    p = full_params(dict(C1 if cfg == "c1" else C2, L=L))
    rs = np.random.RandomState(77)
    Q0 = rs.uniform(-0.01, 0.01, (L, L, 2, 2))
    S0 = rs.randint(0, 2, (L, L))
    eng = _engine(p, precision="fp64")
    eng.set_state(S0, np.zeros((L, L)), Q0)
    sim = c_oracle.Sim(p, S0, np.zeros((L, L)), Q0, "fp64")
    for c0 in range(0, n, chunk):
        us = np.empty((chunk, L, L)); bs = np.empty((chunk, L, L), np.uint8)
        for t in range(chunk):
            us[t] = rs.rand(L, L)
            bs[t] = rs.randint(0, 2, (L, L))
        eng.set_replay(us, bs)
        eng.step(chunk)
        sim.run(chunk, lambda t, L_: (us[t - 1 - c0], bs[t - 1 - c0]))
        eng.sync()
    S, R, Q = eng.get_state()
    assert np.array_equal(S, sim.S), f"{(S != sim.S).sum()} strategy mismatches"
    assert np.array_equal(R, sim.R)
    rel = np.abs(Q - sim.Q) / np.maximum(np.abs(sim.Q), 1e-30)
    assert rel.max() <= 1e-6
    assert np.array_equal(Q, sim.Q)
    eng.close()


F32_CASES = [
    ("c1_L100", dict(C1, L=100)),
    ("c1_L128", dict(C1, L=128)),
    ("c2_L200", dict(C2, L=200)),
    ("rep_m2_L256", dict(C1, L=256, use_second_order=True, r=3.6, influence_factor=0.5)),
    ("halfR_L96", dict(C1, L=96, rep_gain_C=0.5)),          # int8 in units of 1/2
    ("fracR_L72", dict(C1, L=72, rep_gain_C=0.3, delta_R_D=0.7, use_second_order=True)),  # fp32 R
    ("act_m1_L520", dict(C2, L=520, use_second_order=False, r=3.0)),
    # 128-aligned sides take the TMA/SWAR fast path (spgg_fast.cuh)
    ("fast_act_m1_L384", dict(C2, L=384, use_second_order=False, r=3.0, reward_weight_payoff=0.9)),
    ("fast_act_m2_L256", dict(C2, L=256)),
    ("fast_rep_m2_L640", dict(C1, L=640, use_second_order=True)),
    ("fast_halfR_L128", dict(C1, L=128, rep_gain_C=0.5, R_min=-7, R_max=7.5)),
    # sides that are multiples of 32 but not of 128: the last tile column is partial (round 2)
    ("fast_part_rep_m1_L160", dict(C1, L=160)),
    ("fast_part_act_m2_L224", dict(C2, L=224)),
    ("fast_part_rep_m2_L416", dict(C1, L=416, use_second_order=True, r=3.6)),
    ("fast_part_act_m1_L288", dict(C2, L=288, use_second_order=False, r=3.0, reward_weight_payoff=0.9)),
]


@pytest.mark.parametrize("name,p", F32_CASES, ids=[c[0] for c in F32_CASES])
def test_fp32_philox_vs_oracle_bit_exact(monkeypatch, name, p):
    """Throughput instantiation (fp32 Q, int8/fp32 R, Philox) == its C restatement.  Lattices
    that fit on chip would run on the resident cluster kernel (tests/test_gpu_resident.py covers
    it); here the per-iteration kernels are pinned: general kernel, or TMA fast path (fast_*)."""
    from oracle import c_oracle
    monkeypatch.setenv("SPGG_NO_RESIDENT", "1")
    p = full_params(p)
    L, n = p["L"], 60
    rs = np.random.RandomState(3)
    Q0 = rs.uniform(-0.01, 0.01, (L, L, 2, 2)).astype(np.float32).astype(np.float64)
    S0 = rs.randint(0, 2, (L, L))
    eng = _engine(p, seeds=4242, precision="fp32")
    if name.startswith("fast_"):
        assert eng.describe().startswith("fast"), eng.describe()
    eng.set_state(S0, np.zeros((L, L)), Q0)
    eng.step(n)
    S, R, Q = eng.get_state()
    sim = c_oracle.Sim(p, S0, np.zeros((L, L)), Q0, "fp32", seed=4242)
    rows_o = sim.run(n)
    assert np.array_equal(S, sim.S)
    assert np.array_equal(R, sim.R.astype(np.float64))
    assert np.array_equal(Q.astype(np.float32), sim.Q)
    rows = eng.stats()[1:]
    ints = [0, 1, 2, 3, 11, 12, 13, 14, 15, 16, 31, 32]
    assert np.array_equal(rows[:, ints], rows_o[:, ints])
    assert np.array_equal(rows[:, 33].astype(np.float32), rows_o[:, 33].astype(np.float32))
    np.testing.assert_allclose(rows[:, 4:11], rows_o[:, 4:11], rtol=1e-6, atol=1e-6)
    sum_r = eng.stats()[:-1, 17]   # sum of R before the action: recorded by the launch that chooses it
    if eng.status().r_is_int8:
        assert np.array_equal(sum_r, rows_o[:, 17])   # integer units, scaled once
    else:
        np.testing.assert_allclose(sum_r, rows_o[:, 17], rtol=1e-6, atol=1e-6 * L * L)
    np.testing.assert_allclose(rows[:, 18:31], rows_o[:, 18:31], rtol=1e-4, atol=1e-3)
    eng.close()


@pytest.mark.parametrize("L", [256, 352])
@pytest.mark.parametrize("second", [False, True])
@pytest.mark.parametrize("state", ["reputation", "action"])
def test_fast_path_equals_general_path(monkeypatch, second, state, L):
    """The TMA/SWAR kernel and the general kernel are two layouts of the same arithmetic (L=352: with a
    partial last tile column)."""
    n = 25
    p = full_params(dict(C1, L=L, use_second_order=second, state_representation=state))
    rs = np.random.RandomState(21)
    Q0 = rs.uniform(-0.01, 0.01, (L, L, 2, 2))
    S0 = rs.randint(0, 2, (L, L))
    outs = []
    monkeypatch.setenv("SPGG_NO_RESIDENT", "1")
    for no_fast in (False, True):
        if no_fast:
            monkeypatch.setenv("SPGG_NO_FAST", "1")
        else:
            monkeypatch.delenv("SPGG_NO_FAST", raising=False)
        eng = _engine(p, seeds=31, precision="fp32")
        eng.set_state(S0, np.zeros((L, L)), Q0)
        eng.step(n)
        outs.append(eng.get_state() + (eng.stats(),))
        eng.close()
    for a, b in zip(*outs):
        if a.ndim == 2 and a.shape[1] == 40:
            exact = [c for c in range(18) if c != 10] + [31, 32, 33]
            assert np.array_equal(a[:, exact], b[:, exact])
            # fp32 partial sums are grouped differently by the two layouts
            np.testing.assert_allclose(a[:, 10], b[:, 10], rtol=1e-5, atol=1e-4)
            np.testing.assert_allclose(a[:, 18:31], b[:, 18:31], rtol=1e-5, atol=1e-4)
        else:
            assert np.array_equal(a, b)


def test_fp32_replay_draws_vs_oracle():
    from oracle import c_oracle
    L, n = 64, 40
    p = full_params(dict(C1, L=L))
    Q0, S0, u, b = legacy_stream(5, L, n)
    Q0 = Q0.astype(np.float32).astype(np.float64)
    eng = _engine(p, precision="fp32")
    eng.set_state(S0, np.zeros((L, L)), Q0)
    eng.set_replay(u, b)
    eng.step(n)
    S, R, Q = eng.get_state()
    sim = c_oracle.Sim(p, S0, np.zeros((L, L)), Q0, "fp32")
    sim.run(n, lambda t, L_: (u[t - 1], b[t - 1]))
    assert np.array_equal(S, sim.S) and np.array_equal(Q.astype(np.float32), sim.Q)
    eng.close()


CHUNK_CASES = [("resident", "qlearning", "philox")] + [
    ("per_iteration", algo, draws) for algo in ("qlearning", "sarsa", "expected_sarsa", "double_qlearning")
    for draws in ("philox", "replay")]


@pytest.mark.parametrize("path,algorithm,draws", CHUNK_CASES, ids=["-".join(c) for c in CHUNK_CASES])
def test_chunking_is_invisible(monkeypatch, path, algorithm, draws):
    """step(7)+step(13) == step(20): the counter-based stream and the skewed pipeline do not
    depend on where the host cuts the run - for every TD rule, with Philox draws or with the
    replayed draw pairs re-armed at every chunk (SARSA's and Double Q's further pairs feed the
    update launched in the next call)."""
    if path == "per_iteration":
        monkeypatch.setenv("SPGG_NO_RESIDENT", "1")
    L = 160
    p = full_params(dict(C1, L=L, use_second_order=True, algorithm=algorithm))
    rs = np.random.RandomState(9)
    nq = 8 if algorithm == "double_qlearning" else 4
    Q0 = rs.uniform(-0.01, 0.01, (L, L, nq))
    S0 = rs.randint(0, 2, (L, L))
    pairs = {"sarsa": 3, "double_qlearning": 2}.get(algorithm, 1)
    u = rs.rand(20, pairs, L, L)
    b = rs.randint(0, 2, (20, pairs, L, L)).astype(np.uint8)
    outs = []
    mixed = False
    for chunks in ((20,), (7, 13), (1,) * 20):
        eng = _engine(p, seeds=99, precision="fp32")
        if algorithm != "qlearning":
            assert eng.describe().endswith("k_step) (fp32 Q, int8 R)"), eng.describe()
        # replayed selects run on the general kernel; on the fast path a chunk's closing update (no select)
        # then runs k_step_fast, so where the chunks end decides which kernel folds an iteration's statistics
        mixed = draws == "replay" and eng.describe().startswith("fast")
        eng.set_state(S0, np.zeros((L, L)), Q0)
        rows = []
        t0 = 0
        for c in chunks:
            if draws == "replay":
                if pairs == 1:
                    eng.set_replay(u[t0:t0 + c, 0], b[t0:t0 + c, 0])
                else:
                    eng.set_replay(u[t0:t0 + c], b[t0:t0 + c])
            eng.step(c)
            t0 += c
            rows.append(eng.stats()[1:])
        outs.append(eng.get_state() + (np.vstack(rows),))
        assert eng.status().iteration == 20
        eng.close()
    for o in outs[1:]:
        for a, b in zip(outs[0], o):
            if mixed and a.ndim == 2 and a.shape[1] == 40:
                # as in test_fast_path_equals_general_path: the two layouts group fp32 partial sums differently
                exact = [c for c in range(18) if c != 10] + [31, 32, 33]
                assert np.array_equal(a[:, exact], b[:, exact])
                np.testing.assert_allclose(a[:, 10], b[:, 10], rtol=1e-5, atol=1e-4)
                np.testing.assert_allclose(a[:, 18:31], b[:, 18:31], rtol=1e-5, atol=1e-4)
            else:
                assert np.array_equal(a, b)


def test_batched_replicas_equal_single_runs(monkeypatch):
    """Replicas batched in one launch (the sweep of runner.py:117-156) == separate runs."""
    monkeypatch.setenv("SPGG_NO_RESIDENT", "1")   # the general kernel's batching; resident: test_gpu_resident.py
    L, n = 100, 30
    plist = [full_params(dict(C1, L=L, r=r, influence_factor=k))
             for r, k in ((3.0, 1.0), (3.6, 0.0), (5.0, 2.0), (1.0, 0.5))]
    rs = np.random.RandomState(1)
    init = [(rs.randint(0, 2, (L, L)), rs.uniform(-0.01, 0.01, (L, L, 2, 2))) for _ in plist]
    eng = _engine(plist, seeds=[10, 11, 12, 13], precision="fp32")
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


def test_batched_replicas_on_the_fast_path_equal_single_runs(monkeypatch):
    """Same as above on 128-aligned lattices (TMA fast path, grid = replicas x CTAs, per-replica
    reward tables, Philox keys and early-exit flags)."""
    monkeypatch.setenv("SPGG_NO_RESIDENT", "1")
    L, n = 256, 40
    plist = [full_params(dict(C1, L=L, r=r, influence_factor=k, reward_weight_payoff=w))
             for r, k, w in ((3.0, 1.0, 0.95), (4.0, 0.0, 1.0), (5.0, 2.0, 0.9))]
    rs = np.random.RandomState(5)
    init = [(rs.randint(0, 2, (L, L)), rs.uniform(-0.01, 0.01, (L, L, 2, 2))) for _ in plist]
    eng = _engine(plist, seeds=[20, 21, 22], precision="fp32")
    for i, (S0, Q0) in enumerate(init):
        eng.set_state(S0, np.zeros((L, L)), Q0, replica=i)
    eng.step(n)
    for i, (S0, Q0) in enumerate(init):
        single = _engine(plist[i], seeds=20 + i, precision="fp32")
        single.set_state(S0, np.zeros((L, L)), Q0)
        single.step(n)
        for a, b in zip(eng.get_state(i), single.get_state()):
            assert np.array_equal(a, b)
        ra, rb = eng.stats(i), single.stats()
        exact = [c for c in range(18) if c != 10] + [31, 32, 33]
        assert np.array_equal(ra[:, exact], rb[:, exact])
        # the per-CTA partial sums are grouped differently when the grid is shared
        np.testing.assert_allclose(ra[:, 18:31], rb[:, 18:31], rtol=1e-5, atol=1e-4)
        single.close()
    eng.close()


def test_early_exit_matches_reference_semantics():
    """spgg.py:405: the loop breaks before acting once the lattice is uniform."""
    from oracle import spgg_numpy
    L = 8
    p = full_params(dict(C1, L=L, epsilon=0.0, epsilon_min=0.0, iterations=10))
    # every site prefers to defect in both states -> after iteration 1 all D -> iteration 2 breaks
    Q0 = np.zeros((L, L, 2, 2))
    Q0[..., 1] = 1.0
    S0 = np.random.RandomState(0).randint(0, 2, (L, L))
    eng = _engine(p, precision="fp64")
    eng.set_state(S0, np.zeros((L, L)), Q0)
    u = np.ones((10, L, L)) * 0.5
    b = np.zeros((10, L, L), np.uint8)
    eng.set_replay(u, b)
    eng.step(10)
    st = eng.status()
    assert st.stopped_at == 1 and st.iteration == 1
    ref = spgg_numpy.simulate(p, S0, np.zeros((L, L)), Q0, lambda t, L_: (u[t - 1], b[t - 1]))
    S, R, Q = eng.get_state()
    assert np.array_equal(S, ref["Sn_final"]) and np.array_equal(R, ref["R_final"])
    assert np.array_equal(Q, ref["q_final"])
    assert len(ref["epsilon_history_final"]) == 1 and len(ref["coop_rate_history"]) == 2
    # uniform initial lattice: nothing runs at all
    eng2 = _engine(p, precision="fp32")
    eng2.set_state(np.zeros((L, L), np.uint8), np.zeros((L, L)), Q0)
    eng2.step(5)
    assert eng2.status().iteration == 0 and eng2.status().stopped_at == 0
    eng.close(); eng2.close()


def test_L4096_32_iterations_vs_oracle_and_invariants():
    """BASELINE config 4, the geometry bench.py times (32 x 256 tiles of 128 x 16 sites walked by
    296 persistent CTAs): 32 iterations fp32 / Philox against the C oracle, S, R, Q and the integer
    statistics bit for bit.  32 iterations take the reputations into both clamps (|R| = 10 needs
    10), move epsilon through 32 thresholds and make every CTA walk its whole tile list; then
    size-independent invariants over a longer run."""
    from oracle import c_oracle
    L, n = 4096, 32
    p = full_params(dict(C1, L=L))
    rs = np.random.RandomState(2)
    Q0 = rs.uniform(-0.01, 0.01, (L, L, 2, 2)).astype(np.float32).astype(np.float64)
    S0 = rs.randint(0, 2, (L, L)).astype(np.uint8)
    eng = _engine(p, seeds=7, precision="fp32")
    assert eng.describe().startswith("fast")
    eng.set_state(S0, np.zeros((L, L)), Q0)
    eng.step(n)
    S, R, Q = eng.get_state()
    rows = eng.stats()[1:]
    sim = c_oracle.Sim(p, S0, np.zeros((L, L)), Q0, "fp32", seed=7)
    rows_o = sim.run(n)
    assert np.array_equal(S, sim.S), f"{(S != sim.S).sum()} strategy mismatches"
    assert np.array_equal(R, sim.R.astype(np.float64))
    assert np.array_equal(Q.astype(np.float32), sim.Q)
    assert R.min() == p["R_min"] and R.max() == p["R_max"]       # both clamps were reached
    ints = [0, 1, 2, 3, 11, 12, 13, 14, 15, 16, 31, 32]
    assert np.array_equal(rows[:, ints], rows_o[:, ints])
    assert np.array_equal(rows[:, 33].astype(np.float32), rows_o[:, 33].astype(np.float32))  # exact max
    np.testing.assert_allclose(rows[:, 4:11], rows_o[:, 4:11], rtol=1e-5)
    assert np.array_equal(eng.stats()[:-1, 17], rows_o[:, 17])   # sum of R before the action: int8 units, scaled once
    np.testing.assert_allclose(rows[:, 18:31], rows_o[:, 18:31], rtol=2e-4, atol=1e-2)
    eng.step(40)
    rows = eng.stats()
    it = rows[1:]
    N = float(L * L)
    assert np.array_equal(it[1:, 0], it[:-1, 3])                 # coop count chains
    assert np.array_equal(it[:, 0] - it[:, 3], it[:, 1] - it[:, 2])  # switches balance
    assert np.array_equal(it[:, 11:17].sum(1), np.full(len(it), N))  # one group per site
    nD = N - it[:, 3]
    assert np.array_equal((it[:, 11:17] * np.arange(6)).sum(1), 5 * nD)  # each D sits in 5 groups
    S2, R2, _ = eng.get_state(want_q=False)
    assert R2.min() >= p["R_min"] and R2.max() <= p["R_max"]
    assert (S2 == 0).sum() == it[-1, 3]
    eng.close()
