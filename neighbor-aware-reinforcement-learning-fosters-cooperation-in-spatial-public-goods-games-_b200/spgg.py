"""``SPGG``: the reference's model class (``src/model/spgg.py:39-637``) with the loop body
of ``run`` replaced by the fused CUDA step behind the C ABI.

Same constructor signature, attributes, ``run(filename) -> (coop, def, mean P)`` and
HDF5 dataset names/dtypes/shapes, so ``src/experiments/runner.py`` and the plotting
scripts of the reference work unchanged when ``src.model.SPGG`` is this class
(INTEGRATION.md).  Extra keyword arguments (stored in ``params`` like any other, as the
reference does with ``**params``):

``seed``       int: pins the NumPy stream of the ctor draws (same draws as the reference
               with its ``np.random.seed()`` call pinned) and keys the device Philox stream.
``precision``  ``"fp32"`` (default: throughput instantiation) or ``"fp64"`` (reference
               operation order, no FMA).
``draws``      ``"philox"`` (default, on device) or ``"numpy"``: replay the reference's
               own draw stream (``rand(L,L)`` then ``randint(0,2,(L,L))`` per step); with
               ``precision="fp64"`` and a ``seed`` this reproduces the reference bit for bit.
``device``     CUDA device index (default 0).
``chunk``      iterations per device call (default 4096).
"""
from __future__ import annotations

import os

import numpy as np

from . import _lib as L_
from . import h5lite, series
from .algorithms import RLAlgorithm, create_algorithm
from .engine import Engine

_REF_SNAPSHOTS = (1, 10, 100, 1000, 5000, 10000, 20000, 30000, 40000)   # spgg.py:153


class SPGG:
    def __init__(self, r=2, c=1, cost=0.5, K=0.1, L=50, iterations=1000,
                 num_of_strategies=2, population_type=0, S_in_one=None,
                 alpha=0.1, gamma=0.9, epsilon=0.5, epsilon_decay=0.995,
                 epsilon_min=0.01, influence_factor=1.0, use_second_order=True,
                 lambda_epsilon=0.01, delta_R_C=1, delta_R_D=1, R_min=-10,
                 R_max=10, reward_weight_payoff=1.0, rep_gain_C=0.5,
                 state_representation='reputation', algorithm='qlearning', **params):
        seed = params.get("seed")
        if seed is None:
            np.random.seed()                      # spgg.py:98
            rng = np.random                       # global stream, like the reference
            self._philox_seed = int(np.random.randint(0, 2 ** 31 - 1)) | (
                int(np.random.randint(0, 2 ** 31 - 1)) << 31)
        else:
            rng = np.random.RandomState(int(seed))
            self._philox_seed = int(seed)
        self._rng = rng

        all_params = dict(locals(), **params)     # spgg.py:101-105
        for k in ("self", "params", "rng", "seed"):
            all_params.pop(k, None)
        all_params.update(params)
        self.params = all_params
        for key, val in self.params.items():
            setattr(self, key, val)

        self.reward_weight_rep = 1 - self.reward_weight_payoff        # spgg.py:108
        if state_representation not in ("reputation", "action"):
            # the reference raises this from get_state() inside run() (spgg.py:309)
            self._bad_state = state_representation
        if isinstance(algorithm, str):                                 # spgg.py:111-118
            self.algorithm = create_algorithm(algorithm, alpha, gamma, epsilon, epsilon_decay,
                                              epsilon_min, **params)
        elif isinstance(algorithm, RLAlgorithm):
            self.algorithm = algorithm
        else:
            raise ValueError(f"algorithm must be str or RLAlgorithm, got {type(algorithm)}")

        self.q_table = rng.uniform(low=-0.01, high=0.01, size=(L, L, 2, 2))   # spgg.py:121
        if hasattr(self.algorithm, "initialize_q_tables"):                    # spgg.py:124-127
            self.algorithm.initialize_q_tables(self.q_table.shape, rng)
            self.q_table = self.algorithm.get_combined_q_table()
        self.R = np.zeros((L, L))                                              # spgg.py:129
        self.cache = {}
        self._Sn = S_in_one
        self.create_population()
        self.track_positions = [(L // 2, L // 2), (L // 4, L // 4), (3 * L // 4, 3 * L // 4)]
        self.q_history = {pos: {'q_c': [], 'q_d': []} for pos in self.track_positions}
        self.it_records = []
        self.epsilon_history = []
        self.rep_avg_history = []
        self.influence_counts = []
        self.best_neighbor_type_history = []
        self.normlize_max = 4 * r
        self.normlize_min = r - 5
        int(np.floor(np.log10(self.iterations)))  # spgg.py:152 (raises for iterations <= 0 like the reference)
        self.snapshot_iters = set(_REF_SNAPSHOTS)
        self.folder = None
        self.P = None
        self.kernel_launches = 0

    # ------------------------------------------------------------------ reference helpers
    def create_population(self):
        """spgg.py:158-164."""
        L = self.L
        if self._Sn is None:
            self._Sn = self._rng.randint(0, 2, size=(L, L))
        self._Sn = np.asarray(self._Sn)
        self._S = [(self._Sn == j).astype(int) for j in range(self.num_of_strategies)]
        return self._S

    def update_reputation(self, actions):
        """spgg.py:319-323 (host convenience; the run loop does this on the device)."""
        delta_R = np.where(actions == 0, self.rep_gain_C, -self.delta_R_D)
        self.R = np.clip(self.R + delta_R, self.R_min, self.R_max)

    # ------------------------------------------------------------------ engine plumbing
    def _engine_params(self):
        return dict(L=self.L, r=self.r, c=self.c, cost=self.cost, alpha=self.algorithm.alpha,
                    gamma=self.algorithm.gamma, epsilon=self.algorithm.epsilon,
                    epsilon_decay=self.algorithm.epsilon_decay,
                    epsilon_min=self.algorithm.epsilon_min,
                    influence_factor=self.influence_factor,
                    use_second_order=self.use_second_order, lambda_epsilon=self.lambda_epsilon,
                    delta_R_D=self.delta_R_D, R_min=self.R_min, R_max=self.R_max,
                    reward_weight_payoff=self.reward_weight_payoff, rep_gain_C=self.rep_gain_C,
                    state_representation=self.state_representation,
                    algorithm=getattr(self.algorithm, "name", "qlearning"))

    def run(self, filename):
        """spgg.py:325-637."""
        return run_models([self], [filename])[0]

    def _check_runnable(self):
        if getattr(self, "_bad_state", None) is not None:
            raise ValueError(f"Unknown state_representation: {self._bad_state}. "
                             f"Must be 'reputation' or 'action'")
        # The reference recomputes the TD error of the neighbour-influence statistic with the ctor's alpha and
        # gamma (spgg.py:446-473, 512) while the update itself uses the algorithm object's; the fused kernel
        # has one pair.  An instance that disagrees with the ctor would silently change that statistic.
        if (float(self.algorithm.alpha) != float(self.alpha) or float(self.algorithm.gamma) != float(self.gamma)):
            raise ValueError("the RLAlgorithm instance's alpha / gamma differ from the SPGG ctor's: the reference "
                             "mixes the two in its neighbour-influence statistic (spgg.py:446-473); pass equal values")
        if getattr(self.algorithm, "kernel_tag", None) is None:
            raise ValueError(
                f"algorithm '{getattr(self.algorithm, 'name', type(self.algorithm).__name__)}' is not "
                "built into the fused CUDA step (the reference's four rules are); "
                "there is no CPU fallback")

    def _snapshot(self, eng, i, data_file, snaps, replica=0, deferred=None):
        """State before iteration i acts (spgg.py:397-402).  The device->host copy happens now;
        with ``deferred`` (a list) the histogram and the HDF5 writes are queued so the caller can
        run them while the GPU works on the next chunk."""
        S, R, _ = eng.get_state(replica, want_q=False)
        rep_hist, rep_bins = eng.r_histogram(20, self.R_min, self.R_max, replica)   # np.histogram on the device
        snaps[i] = True

        def write():
            data_file.create_dataset(f"R_snapshot_{i}", data=R)
            data_file.create_dataset(f"rep_hist_{i}", data=rep_hist)
            data_file.create_dataset(f"rep_bins_{i}", data=rep_bins)
            data_file.create_dataset(f"Sn_snapshot_{i}", data=S.astype(np.int64))
        if deferred is None:
            write()
        else:
            deferred.append(write)

    def _write_final(self, data_file, ser, S, R, rep_hist_final, rep_bins_final, cluster_sizes):
        """Dataset names, order and dtypes of spgg.py:595-633.  ``cluster_sizes``: the sizes of the
        4-connected, non-periodic clusters of cooperators (spgg.py:631-633), labelled on the device."""
        for key in ("it_records_final", "epsilon_history_final", "rep_avg_history_final",
                    "coop_rate_history", "switch_C_to_D", "switch_D_to_C",
                    "neighbor_influence_percent", "payoff_component_history",
                    "rep_component_history", "best_neighbor_second_order_percent",
                    "reputation_reward_ratio", "avg_reward_C_history", "avg_reward_D_history"):
            data_file.create_dataset(key, data=ser[key])
        for k in range(6):
            data_file.create_dataset(f"group_comp_d{k}_history", data=ser[f"group_comp_d{k}_history"])
        for grp in ("cooperators", "defectors"):
            for nm in series.Q_NAMES:
                data_file.create_dataset(f"{grp}_{nm}_history", data=ser[f"{grp}_{nm}_history"])
        for nm in series.Q_NAMES:
            data_file.create_dataset(f"avg_{nm}_history", data=ser[f"avg_{nm}_history"])
        for pos in self.track_positions:                               # always empty, spgg.py:345,620-622
            data_file.create_dataset(f"q_c_pos_{pos[0]}_{pos[1]}_final", data=np.zeros(0))
            data_file.create_dataset(f"q_d_pos_{pos[0]}_{pos[1]}_final", data=np.zeros(0))
        data_file.create_dataset("Sn_final", data=S.astype(np.int64))
        data_file.create_dataset("R_final", data=R)
        data_file.create_dataset("rep_hist_final", data=rep_hist_final)
        data_file.create_dataset("rep_bins_final", data=rep_bins_final)
        data_file.create_dataset("cluster_sizes", data=np.asarray(cluster_sizes, dtype=np.int64))


class _HostWorker:
    """Runs queued host jobs (snapshot post-processing) on one background thread, one batch at a
    time; ctypes and NumPy release the GIL, so the jobs overlap the C call that enqueues and the
    GPU that computes the next chunk.  Exceptions resurface in ``join``."""

    def __init__(self):
        self._thread = None
        self._error = None

    def run(self, jobs):
        self.join()
        if not jobs:
            return
        import threading

        def body():
            try:
                for job in jobs:
                    job()
            except BaseException as e:   # re-raised on the caller's thread
                self._error = e
        self._thread = threading.Thread(target=body, daemon=True)
        self._thread.start()

    def join(self):
        if self._thread is not None:
            self._thread.join()
            self._thread = None
        if self._error is not None:
            e, self._error = self._error, None
            raise e


def run_models(models, filenames):
    """``SPGG.run`` for one or several models at once (spgg.py:325-637 for each).  Models that
    share the lattice geometry (L, use_second_order, state_representation, precision) run as
    batched replicas of ONE device handle - the GPU counterpart of the reference's one process
    per parameter tuple (runner.py:117-156).  Returns the list of ``run`` return values."""
    models = list(models)
    for m in models:
        m._check_runnable()
    m0 = models[0]
    L, N, n = m0.L, m0.L * m0.L, len(models)
    precision = m0.params.get("precision", "fp32")
    draws = m0.params.get("draws", "philox")
    chunk_max = int(m0.params.get("chunk", 4096))
    for m in models[1:]:
        if (m.L, bool(m.use_second_order), m.state_representation, m.params.get("precision", "fp32"),
                int(m.iterations), getattr(m.algorithm, "kernel_tag", None)) != (
                L, bool(m0.use_second_order), m0.state_representation, precision,
                int(m0.iterations), getattr(m0.algorithm, "kernel_tag", None)):
            raise ValueError("batched models must share L, use_second_order, state_representation, "
                             "precision, iterations and algorithm")
    if draws == "numpy":
        if n != 1:
            raise ValueError("draws='numpy' (replay of the reference's stream) runs one model at a time")
        chunk_max = max(1, min(chunk_max, (64 << 20) // (27 * N) or 1))
    eps0 = [float(m.algorithm.epsilon) for m in models]
    for m in models:
        snapshots_dir = os.path.join(m.folder, 'plots', 'snapshots') if m.folder else 'snapshots'
        os.makedirs(snapshots_dir, exist_ok=True)                      # spgg.py:365-366
    T = int(m0.iterations)
    cut_points = sorted(i - 1 for i in m0.snapshot_iters if 1 <= i <= T)
    eng = Engine([m._engine_params() for m in models], seeds=[m._philox_seed for m in models],
                 precision=precision, device=int(m0.params.get("device", 0)))
    files = [h5lite.open_file(f, "w") for f in filenames]
    results = []
    worker = _HostWorker()
    try:
        for r, m in enumerate(models):
            q_host = m.q_table
            if eng.nq == 8:   # Double Q-learning: both tables, [site][table][s][a]
                q_host = np.stack([m.algorithm.q_table_1, m.algorithm.q_table_2], axis=2)
            eng.set_state(m._Sn, m.R, q_host, replica=r)
        rows_it = [[] for _ in models]
        sum_r_before = [[] for _ in models]
        stop_sum_r = [0.0] * n
        done = [0] * n
        stopped = [False] * n
        snaps = [{} for _ in models]
        t = 0                                       # iterations launched so far (running replicas are in lockstep)
        while t < T and not all(stopped):
            host_work = []          # snapshot post-processing, run while the GPU computes the chunk
            if t in cut_points or (t == 0 and 1 in m0.snapshot_iters):
                for r, m in enumerate(models):
                    if not stopped[r]:
                        m._snapshot(eng, t + 1, files[r], snaps[r], r, deferred=host_work)
            nxt = min([c for c in cut_points if c > t] + [T])
            k_req = min(nxt - t, chunk_max)
            if draws == "numpy":
                # the reference's stream: per iteration rand(L,L) then randint(0,2,(L,L))
                # (algorithms.py:105,108); SARSA draws three such pairs (spgg.py:410,433,452)
                tag = getattr(m0.algorithm, "kernel_tag", "")
                pairs = {"sarsa": 3, "double_qlearning": 2}.get(tag, 1)
                u = np.empty((k_req, pairs, L, L))
                b = np.zeros((k_req, pairs, L, L), np.uint8)
                for i in range(k_req):
                    for q in range(pairs):
                        u[i, q] = m0._rng.rand(L, L)
                        if not (tag == "double_qlearning" and q == 1):  # Double-Q: rand, randint, rand
                            b[i, q] = m0._rng.randint(0, 2, size=(L, L))
                eng.set_replay(u if pairs > 1 else u[:, 0], b if pairs > 1 else b[:, 0])
            worker.run(host_work)   # histogram + HDF5 writes of the snapshots on a host thread ...
            eng.step(k_req)         # ... while this call enqueues the chunk and the GPU computes it
            for r, m in enumerate(models):
                if stopped[r]:
                    continue
                st = eng.status(r)
                rows = eng.stats(r)
                k = int(st.iteration) - done[r]                         # iterations really completed
                rows_it[r].append(rows[1:k + 1])
                sum_r_before[r].append(rows[:k, L_.ST_SUM_R])
                stop_sum_r[r] = rows[k, L_.ST_SUM_R]
                done[r] += k
                if st.stopped_at >= 0 and st.stopped_at <= done[r]:
                    stopped[r] = True
                    if (done[r] + 1) in m.snapshot_iters and (done[r] + 1) not in snaps[r]:
                        worker.join()
                        m._snapshot(eng, done[r] + 1, files[r], snaps[r], r)   # spgg.py:397 precedes :405
            t += k_req
        worker.join()
        launches = int(eng.status().kernel_launches)
        for r, m in enumerate(models):
            S, R, _ = eng.get_state(r, want_q=False)
            hist_f, bins_f = eng.r_histogram(20, m.R_min, m.R_max, r)
            # scipy.ndimage.label(S == 0) on the device; here, not on the writer thread: one thread per handle
            sizes_f = eng.cluster_sizes(r)
            ri = np.vstack(rows_it[r]) if rows_it[r] else np.zeros((0, L_.NSTAT))
            sb = np.concatenate(sum_r_before[r]) if sum_r_before[r] else np.zeros(0)
            # the schedule the engine ran is the algorithm object's (it may be an instance the caller built)
            ser_params = dict(m.params, epsilon_decay=m.algorithm.epsilon_decay, epsilon_min=m.algorithm.epsilon_min)
            ser = series.assemble(ri, sb, N, ser_params, eps0[r], stopped=stopped[r],
                                  stop_sum_r=stop_sum_r[r] if stopped[r] else 0.0,
                                  stop_all_coop=bool((S == 0).all()))
            # the final datasets go to the file on the host thread while the Q table (the largest array)
            # comes back from the device
            worker.run([lambda m=m, r=r, ser=ser, S=S, R=R, hist_f=hist_f, bins_f=bins_f, sizes_f=sizes_f:
                        m._write_final(files[r], ser, S, R, hist_f, bins_f, sizes_f)])
            Q = eng.get_q(r)
            if eng.nq == 8:
                m.algorithm.q_table_1 = np.ascontiguousarray(Q[:, :, 0])
                m.algorithm.q_table_2 = np.ascontiguousarray(Q[:, :, 1])
                Q = m.algorithm.get_combined_q_table()
            worker.join()
            m.kernel_launches = launches
            # post-run attributes the reference leaves behind
            m.q_table, m.R, m._Sn = Q, R, S.astype(np.int64)
            m._S = [(m._Sn == j).astype(int) for j in range(m.num_of_strategies)]
            if done[r]:                                  # decay_epsilon() done[r] times (algorithms.py:40-42)
                m.algorithm.epsilon = float(series.epsilon_after(
                    m.algorithm.epsilon, m.algorithm.epsilon_decay, m.algorithm.epsilon_min, done[r])[-1])
            m.epsilon = m.algorithm.epsilon
            m.avg_q_history = {k: list(ser[f"avg_{k}_history"]) for k in series.Q_NAMES}
            m.q_history_by_strategy = {
                g: {k: list(ser[f"{g}_{k}_history"]) for k in series.Q_NAMES}
                for g in ("cooperators", "defectors")}
            m.group_composition_history = [list(ser[f"group_comp_d{k}_history"]) for k in range(6)]
            it = ser["it_records_final"]
            mean_P = float(it[-1, 3]) if len(it) else float("nan")
            nC = int((S == 0).sum())
            results.append((nC / N, (N - nC) / N, mean_P))
    finally:
        try:
            worker.join()          # never close a file under the writer thread
        except BaseException:
            pass
        for f in files:
            f.close()
        eng.close()
    return results
