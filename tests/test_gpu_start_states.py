"""Every kernel path against the C oracle from uploaded start states.

The other engine-vs-oracle tests start from R0 = 0 and Q0 uniform in (-0.01, 0.01).  A run resumed
from a checkpoint (``Engine.restore``) or a drop-in run whose user set ``m.R`` starts elsewhere, so
here each path is compared with ``c_oracle.Sim`` from:

a. uploaded reputations - on the storage grid within the clamps, integers in [-40, 40] units with
   one row holding -128, -17, -16, 15, 16 and 127 units (k_step_fast's biased bytes hold only
   [-16, 15]; beyond that the next select runs on k_step, which clips every R), and R0 = 0 under a
   floor R_min = 2 - on the resident cluster and grid, the TMA fast path (M = 1 / 2, reputation /
   action state, a partial last tile column, units of 1/2), k_step_lean in int8, fp32 R and fp64,
   and SARSA on k_step;
b. fp64 and fp32-R Q-learning with Philox draws on k_step_lean, up to the benchmarked L = 4096;
c. batches whose replicas differ in r, cost, weights, influence factor, reputation gains and int8
   quantum, each replica against its own oracle and seed;
d. Q tables whose entries tie (the greedy choice takes C, the TD target's max sees equal values),
   at epsilon = 0 and epsilon = 1.

Runs are cut into chunks so that a later chunk's opening select is back on the fast kernel.  The
assertions are those of tests/test_gpu_td_rules.py: S, R and Q bit for bit, the integer statistics
and the global maximum exact, the sum of R of every row (the first one included) exact in int8
storage, float sums to the tolerances of the parity tests."""
import numpy as np
import pytest

from helpers import C1, C2, full_params

pytestmark = pytest.mark.gpu

INTS = [0, 1, 2, 3, 11, 12, 13, 14, 15, 16, 31, 32]
SUM_R = 17
SWITCHES = ("SPGG_NO_RESIDENT", "SPGG_NO_RESIDENT_GRID", "SPGG_NO_FAST", "SPGG_NO_LEAN")
# path -> (switches set, what describe() says)
PATHS = {
    "cluster": ((), "resident: cluster"),
    "grid": ((), "resident: cooperative grid"),
    "fast": (("SPGG_NO_RESIDENT",), "fast: "),
    "lean": (("SPGG_NO_RESIDENT",), "+ k_step_lean)"),
    "k_step": (("SPGG_NO_RESIDENT",), "+ k_step)"),
}
SPECIAL_UNITS = [-128, -17, -16, 15, 16, 127]


def _engine(monkeypatch, path, plist, **kw):
    import spgg_b200
    for s in SWITCHES:
        monkeypatch.delenv(s, raising=False)
    for s in PATHS[path][0]:
        monkeypatch.setenv(s, "1")
    eng = spgg_b200.Engine(plist, **kw)
    assert PATHS[path][1] in eng.describe(), eng.describe()
    return eng


def _quantum(p, precision):
    """The step of the R grid the engine stores (int8 units), or None for fp32 / fp64 R."""
    if precision == "fp64":
        return None
    for k in range(5):
        s = float(1 << k)
        if all(float(p[f]) * s == np.floor(float(p[f]) * s) for f in ("rep_gain_C", "delta_R_D", "R_min", "R_max")):
            return 1.0 / s
    return None


def _r0(p, kind, precision, rs):
    L = p["L"]
    rq = _quantum(p, precision)
    if kind == "inside":
        if rq is None:
            R0 = rs.uniform(p["R_min"], p["R_max"], (L, L))
            return R0.astype(np.float32).astype(np.float64) if precision == "fp32" else R0
        return rs.randint(int(round(p["R_min"] / rq)), int(round(p["R_max"] / rq)) + 1, (L, L)) * rq
    if kind == "outside":
        unit = rq or 1.0
        hi = 19 if unit == 0.5 else 40          # units of 1/2: up to +-9.5
        R0 = rs.randint(-hi, hi + 1, (L, L)).astype(np.float64)
        row = rs.randint(L)
        R0[row, :len(SPECIAL_UNITS)] = SPECIAL_UNITS
        return R0 * unit
    assert kind == "floor" and p["R_min"] > 0
    return np.zeros((L, L))


def _q0(L, kind, precision, rs):
    if kind == "uniform":
        Q0 = rs.uniform(-0.01, 0.01, (L, L, 2, 2))
    elif kind == "zero":
        Q0 = np.zeros((L, L, 2, 2))
    else:
        Q0 = rs.choice([-0.01, 0.0, 0.01], (L, L, 2, 2))
    return Q0.astype(np.float32).astype(np.float64) if precision == "fp32" else Q0


def _compare(eng, rep, sim, rows_o, precision, c, where, may_stop):
    """Engine state and the statistic rows of the chunk just run == the oracle's (test_gpu_td_rules.py).
    A run that turns uniform stops (spgg.py:405) at the same iteration as the oracle's, and only the
    rows of the iterations it ran are compared."""
    L = eng.L
    S, R, Q = eng.get_state(rep)
    full = eng.stats(rep)
    m = rows_o.shape[0]
    assert full.shape[0] == c + 1
    if m < c:
        assert may_stop, f"{where}: the oracle's run ended uniform at iteration {sim.t}"
        st = eng.status(rep)
        assert st.stopped_at == sim.t and st.iteration == sim.t, (st.stopped_at, st.iteration, sim.t)
    rows = full[1:m + 1]
    # the sum of R before the action is recorded by the launch that chooses it, one row earlier
    sum_r = full[:m, SUM_R]
    assert np.array_equal(S, sim.S), f"{where}: {(S != sim.S).sum()} S mismatches"
    if precision == "fp64":
        assert np.array_equal(R, sim.R), f"{where}: {(R != sim.R).sum()} R mismatches"
        assert np.array_equal(Q, sim.Q), f"{where}: {(Q != sim.Q).sum()} Q mismatches"
    else:
        Ro = sim.R.astype(np.float64)
        assert np.array_equal(R, Ro), f"{where}: {(R != Ro).sum()} R mismatches"
        Q32 = Q.astype(np.float32)
        assert np.array_equal(Q32, sim.Q), f"{where}: {(Q32 != sim.Q).sum()} Q mismatches"
    bad = np.nonzero((rows[:, INTS] != rows_o[:, INTS]).any(axis=1))[0]
    assert bad.size == 0, f"{where}: integer statistics differ from row {bad[0] + 1} of the chunk"
    if precision == "fp64":
        assert np.array_equal(rows[:, 33], rows_o[:, 33])
        np.testing.assert_allclose(rows[:, 4:11], rows_o[:, 4:11], rtol=1e-10, atol=1e-9)
        np.testing.assert_allclose(sum_r, rows_o[:, SUM_R], rtol=1e-10, atol=1e-9)
        np.testing.assert_allclose(rows[:, 18:31], rows_o[:, 18:31], rtol=1e-9, atol=1e-9)
        return
    assert np.array_equal(rows[:, 33].astype(np.float32), rows_o[:, 33].astype(np.float32))
    big = L >= 4096
    np.testing.assert_allclose(rows[:, 4:11], rows_o[:, 4:11], rtol=1e-5 if big else 1e-6, atol=0 if big else 1e-6)
    if eng.status(rep).r_is_int8:
        assert np.array_equal(sum_r, rows_o[:, SUM_R]), f"{where}: sums of R differ"   # integer units, scaled once
    else:
        np.testing.assert_allclose(sum_r, rows_o[:, SUM_R], rtol=1e-6, atol=1e-6 * L * L)
    np.testing.assert_allclose(rows[:, 18:31], rows_o[:, 18:31], rtol=2e-4 if big else 1e-4,
                               atol=1e-2 if big else 1e-3)


def _run(monkeypatch, path, plist, starts, precision, chunks, seeds, may_stop=False):
    """One engine (one replica per entry of ``plist``) against one oracle per replica, chunk by chunk."""
    from oracle import c_oracle
    eng = _engine(monkeypatch, path, plist if len(plist) > 1 else plist[0], seeds=list(seeds), precision=precision)
    sims = []
    for i, (p, (S0, R0, Q0)) in enumerate(zip(plist, starts)):
        eng.set_state(S0, R0, Q0, replica=i)
        sims.append(c_oracle.Sim(p, S0, R0, Q0, precision, seed=seeds[i]))
    t = 0
    for k, c in enumerate(chunks):
        eng.step(c)
        for i, sim in enumerate(sims):
            rows_o = sim.run(c)
            if k == 0:
                # the oracle's first row holds the uploaded reputations, before the first update clips
                # them (_compare checks the engine's row 0 against it)
                np.testing.assert_allclose(rows_o[0, SUM_R], starts[i][1].sum(), rtol=1e-6, atol=1e-9)
            _compare(eng, i, sim, rows_o, precision, c,
                     f"replica {i}, chunk {k + 1} (iterations {t + 1}-{t + c})", may_stop)
        t += c
    eng.close()
    return sims


def _start(p, r_kind, q_kind, precision, seed):
    rs = np.random.RandomState(seed)
    L = p["L"]
    R0 = _r0(p, r_kind, precision, rs)
    Q0 = _q0(L, q_kind, precision, rs)
    S0 = rs.randint(0, 2, (L, L))
    return S0, R0, Q0


# ------------------------------------------------------------------ a. uploaded reputations
HALF_FAST = dict(C1, rep_gain_C=0.5, R_min=-7, R_max=7.5)
FRAC_R = dict(C1, rep_gain_C=0.3, delta_R_D=0.7)
R_PATHS = [
    # name, path, params, precision
    ("cluster_L100", "cluster", dict(C1, L=100), "fp32"),
    ("grid_L400", "grid", dict(C1, L=400), "fp32"),
    ("fast_rep_m1_L256", "fast", dict(C1, L=256), "fp32"),
    ("fast_act_m2_L256", "fast", dict(C2, L=256), "fp32"),
    ("fast_part_rep_m2_L160", "fast", dict(C1, L=160, use_second_order=True), "fp32"),
    ("fast_halfR_L128", "fast", dict(HALF_FAST, L=128), "fp32"),
    ("lean_int8_L100", "lean", dict(C1, L=100), "fp32"),
    ("lean_int8_rep_m2_L520", "lean", dict(C1, L=520, use_second_order=True), "fp32"),
    ("lean_fracR_L300", "lean", dict(FRAC_R, L=300), "fp32"),
    ("lean_fp64_L130", "lean", dict(C1, L=130, use_second_order=True), "fp64"),
    ("sarsa_k_step_L131", "k_step", dict(C1, L=131, algorithm="sarsa"), "fp32"),
]
R_KINDS = ["inside", "outside", "floor"]


@pytest.mark.parametrize("r_kind", R_KINDS)
@pytest.mark.parametrize("name,path,p,precision", R_PATHS, ids=[c[0] for c in R_PATHS])
def test_uploaded_reputations_vs_oracle(monkeypatch, name, path, p, precision, r_kind):
    p = full_params(dict(p, R_min=2) if r_kind == "floor" else p)
    S0, R0, Q0 = _start(p, r_kind, "uniform", precision, 50 + p["L"] + R_KINDS.index(r_kind))
    if r_kind == "outside" and path == "fast":
        rq = _quantum(p, precision)
        assert (R0 / rq > 15).any() and (R0 / rq < -16).any()
    _run(monkeypatch, path, [p], [(S0, R0, Q0)], precision, (1, 6, 13), [4242])


@pytest.mark.parametrize("path,L", [("fast", 256), ("cluster", 100), ("lean", 100)])
def test_int8_handle_rejects_unrepresentable_reputations(monkeypatch, path, L):
    p = full_params(dict(C1, L=L))
    S0, R0, Q0 = _start(p, "inside", "uniform", "fp32", 3)
    eng = _engine(monkeypatch, path, p, seeds=1, precision="fp32")
    for bad in (0.3, 200.0):
        R = R0.copy()
        R[L // 2, 3] = bad
        with pytest.raises(ValueError, match="r_storage"):
            eng.set_state(S0, R, Q0)
    eng.set_state(S0, R0, Q0)      # the handle stays usable
    eng.step(2)
    eng.close()


def test_fast_strip_rejects_reputations_beyond_its_bytes(monkeypatch):
    """A strip's boundary rows reach its neighbours from k_step_fast itself, so a fast strip cannot take
    the k_step detour: it accepts R within [-16, 15] int8 units and rejects the rest."""
    L = 256
    p = full_params(dict(C1, L=L))
    rs = np.random.RandomState(8)
    S0 = rs.randint(0, 2, (L // 2, L))
    Q0 = rs.uniform(-0.01, 0.01, (L // 2, L, 2, 2))
    eng = _engine(monkeypatch, "fast", p, seeds=1, precision="fp32", rows=L // 2, row0=0)
    R0 = rs.randint(-16, 16, (L // 2, L)).astype(np.float64)
    R0[0, :2] = (-16, 15)
    eng.set_state(S0, R0, Q0)
    for bad in (16.0, -17.0, 127.0):
        R = R0.copy()
        R[L // 4, 5] = bad
        with pytest.raises(ValueError, match=r"\[-16, 15\]"):
            eng.set_state(S0, R, Q0)
    eng.close()


# ------------------------------------------------------------------ b. fp64 and fp32-R Q-learning, Philox
LEAN_CASES = [
    ("fp64_L97_act_m1", dict(C2, L=97, use_second_order=False), "fp64", (7, 13)),
    ("fp64_L130_act_m2", dict(C2, L=130), "fp64", (7, 13)),
    ("fp64_L300_rep_m2", dict(C1, L=300, use_second_order=True), "fp64", (7, 13)),
    ("fp64_L520_fracgains", dict(FRAC_R, L=520), "fp64", (7, 13)),          # 16-row tiles
    ("fp64_L4096", dict(C1, L=4096), "fp64", (8,)),                          # the benchmarked fp64 geometry
    ("fracR_L300", dict(FRAC_R, L=300), "fp32", (8,)),
    ("fracR_L520", dict(FRAC_R, L=520, use_second_order=True), "fp32", (8,)),
    ("fracR_L1100", dict(FRAC_R, L=1100), "fp32", (8,)),
]


@pytest.mark.parametrize("name,p,precision,chunks", LEAN_CASES, ids=[c[0] for c in LEAN_CASES])
def test_lean_philox_vs_oracle(monkeypatch, name, p, precision, chunks):
    p = full_params(p)
    S0, R0, Q0 = _start(p, "inside", "uniform", precision, 70 + p["L"])
    _run(monkeypatch, "lean", [p], [(S0, R0, Q0)], precision, chunks, [9000 + p["L"]])


# ------------------------------------------------------------------ c. batches whose replicas differ
def test_fp64_batch_of_different_replicas_vs_oracles(monkeypatch):
    """Per-replica reward tables (k_build_valtab) and gains in one fp64 launch."""
    L = 130
    plist = [full_params(dict(C1, L=L, use_second_order=True, **kw)) for kw in (
        dict(r=3.0, cost=1, reward_weight_payoff=0.95, influence_factor=1.0),
        dict(r=4.2, cost=0.5, reward_weight_payoff=0.8, influence_factor=0.0, rep_gain_C=0.5),
        dict(r=5.0, cost=1.5, reward_weight_payoff=1.0, influence_factor=2.0, rep_gain_C=0.3, delta_R_D=0.7))]
    starts = [_start(p, "inside", "uniform", "fp64", 90 + i) for i, p in enumerate(plist)]
    _run(monkeypatch, "lean", plist, starts, "fp64", (7, 13), [21, 22, 23])


QUANTA = [dict(rep_gain_C=1.0, R_min=-10, R_max=10),            # units of 1
          dict(rep_gain_C=0.5, R_min=-7, R_max=7),              # units of 1/2, 14 units each way
          dict(rep_gain_C=0.25, R_min=-3.5, R_max=3.5)]         # units of 1/4, 14 units each way


@pytest.mark.parametrize("path,L,n_rep", [("fast", 256, 3), ("cluster", 100, 5), ("lean", 100, 3)])
def test_int8_batch_of_different_quanta_vs_oracles(monkeypatch, path, L, n_rep):
    """Each replica of a batch stores R in its own int8 quantum (rq per replica)."""
    plist = [full_params(dict(C1, L=L, r=3.0 + 0.4 * i, **QUANTA[i % 3])) for i in range(n_rep)]
    assert [_quantum(p, "fp32") for p in plist[:3]] == [1.0, 0.5, 0.25]
    starts = [_start(p, "inside", "uniform", "fp32", 110 + i) for i, p in enumerate(plist)]
    if path == "cluster":
        monkeypatch.setenv("SPGG_RES_CS8", "1")
    _run(monkeypatch, path, plist, starts, "fp32", (1, 6, 13), [300 + i for i in range(n_rep)])


# ------------------------------------------------------------------ d. ties and epsilon edges
TIE_PATHS = [("cluster", 100, "fp32"), ("grid", 400, "fp32"), ("fast", 256, "fp32"), ("lean", 100, "fp32"),
             ("lean", 130, "fp64")]
EPS = {"eps0": dict(epsilon=0.0, epsilon_min=0.0), "eps1": dict(epsilon=1.0, epsilon_decay=1.0)}


@pytest.mark.parametrize("eps", list(EPS))
@pytest.mark.parametrize("q_kind", ["zero", "ternary"])
@pytest.mark.parametrize("path,L,precision", TIE_PATHS, ids=[f"{c[0]}_L{c[1]}_{c[2]}" for c in TIE_PATHS])
def test_ties_and_epsilon_edges_vs_oracle(monkeypatch, path, L, precision, q_kind, eps):
    """Greedy from an all-zero table: every site ties in the state it lands in, picks C and the lattice is
    uniform after iteration 1 - the run must stop there like the oracle's and stay stopped in the next
    chunk.  The other starts run their 20 iterations."""
    p = full_params(dict(C1, L=L, **EPS[eps]))
    rs = np.random.RandomState(130 + L)
    Q0 = _q0(L, q_kind, precision, rs)
    S0 = rs.randint(0, 2, (L, L))
    stops = q_kind == "zero" and eps == "eps0"
    sim, = _run(monkeypatch, path, [p], [(S0, np.zeros((L, L)), Q0)], precision, (7, 13), [55], may_stop=stops)
    assert sim.t == (1 if stops else 20)
