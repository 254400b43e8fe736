/* libspgg_b200 - C ABI of the B200-native SPGG lattice step.
 *
 * The reference (jac0626/Neighbor-Aware-Reinforcement-Learning-...) is pure
 * Python/NumPy and has no FFI of its own; the only boundary of the hot path is
 * the Python class `SPGG` (reference src/model/spgg.py:39-637).  This header
 * is what a Python (ctypes) binding of that class binds instead of the NumPy
 * loop body; every entry point names the reference lines it replaces
 * (paths relative to the reference root).  Plain pointers and sizes only.
 *
 * Conventions: host buffers are caller-owned; device memory is owned by the
 * handle; functions return 0 on success and a negative code on failure, with
 * a message available from spgg_last_error() (thread-local).  One host thread
 * per handle.  All GPU work is enqueued on the stream passed to spgg_step().
 * CUDA is initialised lazily by the first spgg_create() of a process (fork
 * safe until then, reference src/experiments/runner.py:142 forks workers).
 */
#ifndef SPGG_B200_H
#define SPGG_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPGG_ABI_VERSION 2

/* error codes */
#define SPGG_OK 0
#define SPGG_E_INVALID (-1)   /* bad argument (Python side raises ValueError)  */
#define SPGG_E_CUDA (-2)      /* CUDA runtime failure                          */
#define SPGG_E_STATE (-3)     /* call not valid in the handle's current state  */
#define SPGG_E_UNSUPPORTED (-4)

/* precision / arithmetic */
#define SPGG_PREC_FP32 0 /* throughput mode: fp32 float4 Q, int8|fp32 R, exact-count reward table */
#define SPGG_PREC_FP64 1 /* parity mode: fp64 Q and R, reference operation order, no FMA          */

/* state_representation (spgg.py:289-310) */
#define SPGG_STATE_REPUTATION 0
#define SPGG_STATE_ACTION 1

/* algorithm (algorithms.py:344-383) */
#define SPGG_ALGO_QLEARNING 0
#define SPGG_ALGO_SARSA 1          /* algorithms.py:136-178, applied as spgg.py:431-438,450-454 */
#define SPGG_ALGO_EXPECTED_SARSA 2 /* algorithms.py:181-234, spgg.py:455-463 */
#define SPGG_ALGO_DOUBLE_QLEARNING 3 /* algorithms.py:237-341, spgg.py:464-468,498-505: two tables per site */

/* reputation storage in fp32 mode */
#define SPGG_RSTORE_AUTO 0 /* int8 when rep_gain_C, delta_R_D, R_min, R_max are multiples of 2^-k that fit */
#define SPGG_RSTORE_INT8 1
#define SPGG_RSTORE_FP32 2

/* Statistics row: one row of SPGG_NSTAT doubles per iteration and replica.
 * Sums, not means; the host divides (spgg.py:381-394, 419-426, 512-592). */
#define SPGG_NSTAT 40
enum spgg_stat {
  SPGG_ST_NC_OLD = 0,      /* #cooperators in S before the action          spgg.py:383 */
  SPGG_ST_N_CD = 1,        /* C->D switches                                spgg.py:419 */
  SPGG_ST_N_DC = 2,        /* D->C switches                                spgg.py:420 */
  SPGG_ST_NC_NEW = 3,      /* #sites whose action is C                                 */
  SPGG_ST_SUM_P = 4,       /* sum P                                        spgg.py:388 */
  SPGG_ST_SUM_P_C = 5,     /* sum P over previous cooperators              spgg.py:389 */
  SPGG_ST_SUM_P_D = 6,     /* sum P over previous defectors                spgg.py:390 */
  SPGG_ST_SUM_WP_P = 7,    /* sum w_P*P                                    spgg.py:425 */
  SPGG_ST_SUM_REW_C = 8,   /* sum reward over a==C                         spgg.py:542 */
  SPGG_ST_SUM_REW_D = 9,   /* sum reward over a==D                         spgg.py:543 */
  SPGG_ST_SUM_RATIO = 10,  /* sum_{a==C} |w_R*.5|/(|rew|+1e-9)*100         spgg.py:529-536 */
  SPGG_ST_GROUP0 = 11,     /* 11..16: #groups with k=0..5 defectors (new S) spgg.py:586-592 */
  SPGG_ST_SUM_R = 17,      /* sum of R of the state the row index names (row j: R_j) spgg.py:394 */
  SPGG_ST_SUM_Q = 18,      /* 18..21: sum Q[:,:,s,a] after both updates    spgg.py:562-565 */
  SPGG_ST_SUM_Q_C = 22,    /* 22..25: same, previous cooperators           spgg.py:568-583 */
  SPGG_ST_SUM_Q_D = 26,    /* 26..29: same, previous defectors                         */
  SPGG_ST_SUM_NI = 30,     /* sum neighbour-influence percent              spgg.py:512 */
  SPGG_ST_N_BEST_POS = 31, /* #sites with max_diff>0                       spgg.py:521 */
  SPGG_ST_N_BEST_2ND = 32, /* ... whose best neighbour is second order     spgg.py:520 */
  SPGG_ST_GMAX = 33        /* lattice-global max|diff|                     spgg.py:488 */
};

/* Replaces the keyword arguments of SPGG.__init__ that influence the
 * dynamics (spgg.py:50-56); K, population_type, delta_R_C and
 * num_of_strategies are never read by the loop and are not part of the ABI. */
typedef struct spgg_params {
  int32_t L;          /* lattice side (columns; rows too unless a strip)             */
  int32_t rows;       /* rows owned by this handle: L, or the strip height           */
  int32_t row0;       /* global index of the first owned row (strips)                */
  int32_t M;          /* 1 or 2: use_second_order                                    */
  int32_t state_mode; /* SPGG_STATE_*                                                */
  int32_t precision;  /* SPGG_PREC_*                                                 */
  int32_t algorithm;  /* SPGG_ALGO_*                                                 */
  int32_t r_storage;  /* SPGG_RSTORE_*                                               */
  double r, c, cost;
  double alpha, gamma;
  double epsilon, epsilon_decay, epsilon_min;
  double kappa;       /* influence_factor                                            */
  double lambda_eps;
  double rep_gain_C, delta_R_D, R_min, R_max;
  double wP;          /* reward_weight_payoff                                        */
  uint64_t seed;      /* Philox key                                                  */
} spgg_params_t;

typedef struct spgg_status {
  int64_t iteration;   /* completed iterations (state index t: S_t, R_t, Q_t)        */
  int64_t stopped_at;  /* -1, or the t whose S_t is uniform: iteration t+1 breaks (spgg.py:405) */
  double epsilon;      /* epsilon after `iteration` decays (algorithms.py:40-42)     */
  int32_t n_replicas;
  int32_t r_is_int8;
  int64_t kernel_launches; /* kernels launched by this handle so far                 */
  int64_t speculative_launches; /* update launches that guessed the global maximum (below) */
  int64_t speculation_failures; /* ... whose guess was wrong: that iteration and the rest of its chunk were re-run */
} spgg_status_t;

typedef struct spgg_handle spgg_t;

/* SPGG.__init__ (spgg.py:50-156) without the random initial state.  n_replicas
 * independent lattices share L, rows, M, state_mode, precision; everything
 * else may differ per replica (params is an array of n_replicas entries).
 * Replaces one multiprocessing worker per parameter tuple (runner.py:117-156). */
int spgg_create(const spgg_params_t *params, int n_replicas, int device, spgg_t **out);
void spgg_destroy(spgg_t *h);

/* Upload q_table (rows*L*2*2 doubles, layout of spgg.py:121), R (rows*L
 * doubles, spgg.py:129) and _Sn (rows*L bytes, 0=C 1=D, spgg.py:162) of one
 * replica.  Resets that replica's epsilon to its ctor value.
 *
 * The iteration counter (Philox counter word, row index of the statistics) is
 * HANDLE-WIDE.  The first spgg_set_state / spgg_init_random after iterations
 * have run starts a new run: the counter returns to 0 and every OTHER replica
 * of a batch is marked stale; spgg_step / spgg_begin_steps fail with
 * SPGG_E_STATE until each stale replica has been given a state too.  To continue
 * a run instead of starting one, follow the uploads with spgg_set_progress.
 * SPGG_ALGO_DOUBLE_QLEARNING: Q holds both tables, rows*L*2*2*2 doubles laid out
 * [site][table][state][action] (q_table_1, q_table_2 of algorithms.py:245-260). */
int spgg_set_state(spgg_t *h, int replica, const uint8_t *S, const double *R, const double *Q);
int spgg_get_state(spgg_t *h, int replica, uint8_t *S, double *R, double *Q);

/* Checkpoint / resume (SURVEY 8 f4; the reference can only inject strategies, S_in_one
 * spgg.py:51,133,161): declare that the states just uploaded are those after
 * `iteration` completed iterations, with exploration rates epsilon[0..n_replicas)
 * (spgg_query reports both).  The Philox counters, the epsilon schedule
 * (algorithms.py:40-42) and the early-exit bookkeeping continue from there, so
 * n iterations == k iterations + spgg_get_state + spgg_destroy + spgg_create +
 * spgg_set_state + spgg_set_progress + (n-k) iterations, bit for bit. */
int spgg_set_progress(spgg_t *h, int64_t iteration, const double *epsilon);

/* Position-keyed 64-bit digests of one replica's owned rows: out[0] strategies,
 * out[1] reputations, out[2] Q.  A site contributes (hash(global row, column) | 1) *
 * (bits of its value as a double + 1) mod 2^64, so the digests of the strips of a
 * lattice add up (mod 2^64) to the digest of the whole lattice: multi-GPU runs are
 * compared with single-GPU runs without moving a 20 GB state through the host.  The
 * multiplier is odd, so a change of any one value (a sign flip, +0.0 -> -0.0) changes
 * its word.  oracle/spgg_oracle.c: oracle_state_digest computes the same on the host. */
int spgg_state_digest(spgg_t *h, int replica, uint64_t out[3]);

/* np.histogram(R, bins=n_bins, range=(edges[0], edges[n_bins])) of a replica's
 * reputations on the device (rep_hist_* datasets, spgg.py:399-401,626-628): edges
 * are the n_bins+1 values of np.linspace, bins are half-open except the last,
 * the bin index is corrected against the edges as NumPy does.  n_bins <= 64. */
int spgg_r_histogram(spgg_t *h, int replica, int n_bins, const double *edges, int64_t *counts);

/* scipy.ndimage.label(S == which) of one replica on the device (cluster_sizes,
 * spgg.py:631-633): which = 0 selects the cooperators, 1 the defectors; 4-connected,
 * non-periodic unless flags has SPGG_CLUSTER_PERIODIC, which also joins row L-1 to row 0
 * and column L-1 to column 0 (the torus the dynamics live on).  Labels run 1..n in
 * increasing order of each cluster's smallest linear index row*L + col, which is scipy's
 * numbering; the result does not depend on scheduling.  Sees the state spgg_get_state
 * would return.  Whole-lattice handles only (rows == L, rows*L < 2^31; else
 * SPGG_E_UNSUPPORTED; a strip labels through spgg_strip_clusters below).  The result stays
 * on the handle for the two getters below until the next spgg_clusters /
 * spgg_strip_clusters call or until the state changes (spgg_step / spgg_begin_steps,
 * spgg_set_state, spgg_init_random, spgg_set_progress, spgg_strip_rewind); the getters
 * return SPGG_E_STATE without one.  The first call allocates device scratch that the
 * handle keeps until spgg_destroy: 8 bytes a site (union-find parents and set sizes),
 * 2 bits a site (root mask, rank offsets) and room for ceil(L*L/2) int64 sizes, about
 * 12.25 bytes a site in all (206 MB at L=4096, 13.2 GB at L=32768). */
#define SPGG_CLUSTER_PERIODIC 1
int spgg_clusters(spgg_t *h, int replica, int which, int flags, int64_t *n_clusters);
/* After spgg_clusters: sizes[k-1] = #sites of label k, n must equal n_clusters.  After
 * spgg_strip_clusters_resolve: the n_owned clusters whose smallest site lies in this strip,
 * in raster order, i.e. labels first_label+1 .. first_label+n_owned. */
int spgg_cluster_sizes(spgg_t *h, int64_t *sizes, int64_t n);
/* rows*L values, row-major, 0 where not selected; on a strip the labels of the whole lattice
 * (a site of a cluster whose smallest site lies in another strip gets that cluster's label). */
int spgg_cluster_labels(spgg_t *h, int32_t *labels);

/* The same labelling of a lattice split into row strips, one handle (single replica) per
 * rank; the result is defined on the whole L x L lattice and equals spgg_clusters of one
 * handle holding it, bit for bit.  Needs L*L < 2^31 (global site indices are int32), else
 * SPGG_E_UNSUPPORTED.  Per call, on every rank:
 *   1. spgg_strip_clusters labels this strip's rows (replica 0, current state, after
 *      finishing a pending chunk) and writes one boundary record of
 *      spgg_strip_cluster_record_bytes() bytes (device memory; depends on L only) - the
 *      strip's number of clusters and, for each site of its first and last row, its
 *      cluster within the strip, with that cluster's smallest site, raster rank and size;
 *   2. the caller gathers the records of all `world` ranks, in rank order, into one device
 *      buffer on every rank (one all-gather);
 *   3. spgg_strip_clusters_resolve joins the clusters across the strip boundaries (and
 *      across row L-1 | 0 with SPGG_CLUSTER_PERIODIC; the column seam is joined in step 1),
 *      on the device and the same way on every rank.  It returns this strip's number of
 *      owned clusters, the label before the first of them and the number of clusters of
 *      the lattice; spgg_cluster_sizes / spgg_cluster_labels above then serve the result.
 * The records must agree on L, which and flags and their rows must tile [0, L) in rank
 * order (else SPGG_E_INVALID).  A pass that is not resolved yet counts as no result for
 * the getters; the events listed at spgg_clusters discard both.  Scratch: that of
 * spgg_clusters for the strip's rows*L sites, 8 bytes per boundary site (a site of the
 * strip's first or last row) for building the record, whose 16 bytes per boundary site
 * the caller provides, and, in the resolution, 16 bytes per boundary site of every strip. */
int64_t spgg_strip_cluster_record_bytes(spgg_t *h);
int spgg_strip_clusters(spgg_t *h, int which, int flags, void *dev_record);
int spgg_strip_clusters_resolve(spgg_t *h, int world, int rank, const void *dev_records,
                                int64_t *n_owned, int64_t *first_label, int64_t *n_total);

/* Strategy pair counts of one replica on the device: for numpy axis ax and every offset d in
 * 1..max_d, over the torus (indices mod L), n_CC = #sites x that cooperate with x + d*e_ax
 * cooperating too, and n_diff = #sites x whose partner holds the other strategy.
 * out: 2*(max_d+1)*2 int64, out[((ax*(max_d+1)) + d)*2 + k]; ax 0: (i,j)-(i+d,j), ax 1: (i,j)-(i,j+d);
 * k 0: both cooperate, k 1: the two differ; d = 0: {n_C, 0}.  1 <= max_d <= L/2.
 * The rest follows: n_DD = N - n_CC - n_diff, n_CD = n_DC = n_diff/2, and n_diff(ax, 1) / N is
 * the interface density along ax: the fraction of the N nearest-neighbour bonds along that axis
 * that join a cooperator and a defector.  Exact integers, so the result does not depend on scheduling.  Sees
 * the state spgg_get_state would return; changes neither the state, the iteration counter, the
 * statistics rows nor a cluster-labelling result.  Whole-lattice handles only (a strip gets
 * SPGG_E_UNSUPPORTED and counts through spgg_strip_pair_counts below).  Cost: two launches,
 * O(L^2 * max_d / 32) word operations per axis; keeps 32*(max_d+1) bytes of device scratch. */
int spgg_pair_counts(spgg_t *h, int replica, int max_d, int64_t *out);

/* The same counts of a lattice split into row strips, one single-replica handle per rank (a
 * whole-lattice handle is a world of one).  The counts of strip k are those of the pairs whose
 * site x lies in its rows; summed over the ranks they equal spgg_pair_counts of one handle holding
 * the lattice.  The partners of axis 0 reach max_d rows past a strip, so per call, on every rank:
 *   1. spgg_strip_pair_record writes this strip's record (device memory of
 *      spgg_strip_pair_record_bytes(max_d, max_rows) bytes): a header (L, row0, rows, max_d) and
 *      the strip's first min(max_d, rows) rows, packed, padded to max_rows rows.  max_rows must be
 *      the same on every rank, at least min(max_d, rows) of every strip and at most max_d
 *      (min(max_d, largest strip height) fits);
 *   2. the caller gathers the records of all `world` ranks, in rank order, into one device
 *      buffer on every rank (one all-gather);
 *   3. spgg_strip_pair_counts assembles the max_d rows that follow the strip from the records
 *      and writes this strip's counts into out (layout of spgg_pair_counts).
 * Records that disagree on L, max_d or max_rows, or whose rows do not tile [0, L) in rank order,
 * get SPGG_E_INVALID; handles of several replicas SPGG_E_UNSUPPORTED.  Steps 1 and 3 must see the
 * same state.  Scratch: 4*max_d*ceil(L/32) bytes for the assembled rows. */
int64_t spgg_strip_pair_record_bytes(spgg_t *h, int max_d, int max_rows);
int spgg_strip_pair_record(spgg_t *h, int max_d, int max_rows, void *dev_record);
int spgg_strip_pair_counts(spgg_t *h, int world, int rank, const void *dev_records, int max_d,
                           int max_rows, int64_t *out);

/* Block fields of one replica on the device: the lattice cut into B x B blocks of b x b sites,
 * B = ceil(L/b), anchored at site (0, 0), no wrap; block (I, J) covers global rows
 * [I*b, min((I+1)*b, L)) and columns [J*b, min((J+1)*b, L)), so the last block row and column
 * are ragged when b does not divide L.  1 <= b <= L and B*B <= 2^24 (L = 32768 needs b >= 8).
 *   counts[(i*B + J)*2 + k]: int64, k 0 the sites of the block, k 1 its cooperators (S == 0);
 *   sums[((i*B + J)*2 + k)*m + ch]: float64, k 0 over all sites of the block, k 1 over its
 *     cooperators (defectors: the difference); channels ch: with SPGG_BLOCK_R first R as
 *     spgg_get_state returns it (int8 units x quantum), with SPGG_BLOCK_Q then the nq Q entries
 *     in spgg_get_state's order; m = (flags & R) + (flags & Q ? nq : 0).  sums may be null when
 *     flags == 0 (counts only: reads the bit plane alone).
 * i runs over the block rows I0 .. I1 that hold rows of the handle, I = I0 + i: a whole lattice
 * has I0 = 0, I1 = B-1; a strip (rows < L) has I0 = floor(row0/b), I1 = floor((row0+rows-1)/b),
 * and each block holds the contribution of the strip's own rows only, so blocks that straddle
 * a strip boundary are partial and the results of the strips add up to the lattice's.
 * Exactness: counts and int8-storage R sums are exact (the quantum is 2^-k).  fp32 and fp64
 * values are summed in fp64 in an order fixed by (L, row0, rows, b), without floating-point
 * atomics: the same state gives bit-identical sums, whichever kernel path or chunking reached
 * it; a sum of n values x_i differs from the exact one by at most (n-1) 2^-53 sum |x_i|.
 * Sees the state spgg_get_state would return (a pending chunk is finished first); changes
 * neither the state, the iteration counter, the statistics rows, a cluster-labelling result
 * nor the pair-count scratch.  SPGG_E_INVALID: bad replica, b, B, unknown flag bits, null
 * counts, null sums with flags != 0.  Cost: one streaming pass over the bit plane and, if
 * asked, over R and Q; keeps device scratch of 8 bytes per block, plus 16*m bytes per block
 * with flags != 0 and 16*m bytes per piece when b > 32 (pieces per block: ceil(b/32) *
 * ceil(b/256)), grown to the largest call and freed with the handle. */
#define SPGG_BLOCK_R 1
#define SPGG_BLOCK_Q 2
int spgg_block_fields(spgg_t *h, int replica, int b, int flags, int64_t *counts, double *sums);

/* Same distributions as the reference ctor (Q ~ U(-0.01,0.01) spgg.py:121, R = 0
 * spgg.py:129, S ~ Bernoulli(1/2) spgg.py:162) generated on the device from Philox
 * keyed by `seed`; for lattices too large to stage through host memory. */
int spgg_init_random(spgg_t *h, int replica, uint64_t seed);

/* Replay mode: the draw arrays the reference would consume in the next
 * n_steps iterations (algorithms.py:105 `rand(L,L)` and :108
 * `randint(0,2,(L,L))`), each n_steps*rows*L.  Single replica only.  Consumed
 * by the following spgg_step calls; Philox is used once they run out. */
int spgg_set_replay(spgg_t *h, int n_steps, const double *u, const uint8_t *b);
/* Same with n_pairs (rand, randint) pairs per iteration, arrays laid out
 * (n_steps, n_pairs, rows, L): SARSA consumes three pairs per iteration - the action
 * (algorithms.py:145-148 via spgg.py:410), the next action of the update (spgg.py:433) and
 * the next action of the NI statistic (spgg.py:452); Double Q-learning consumes two (the
 * action, and rand(L,L) < 0.5 choosing the table to update, algorithms.py:303 - the second
 * pair's b is ignored); every other rule consumes one. */
int spgg_set_replay_pairs(spgg_t *h, int n_steps, int n_pairs, const double *u, const uint8_t *b);

/* Run n_steps iterations of the loop body spgg.py:368-592 for all replicas
 * (asynchronous on `cuda_stream`, a cudaStream_t or NULL).  One launch for the
 * whole call when the lattices fit in shared memory (one thread-block cluster
 * per replica, csrc/spgg_resident.cuh); otherwise per iteration either the exact
 * pair k_gmax_* (lattice-global max |reward difference|, spgg.py:488) + k_step*, or -
 * TMA fast path - ONE launch that assumes the maximum of the previous iteration,
 * computes the true one as a by-product of the update and compares.  A wrong guess
 * is caught on the device (every later launch of the call returns untouched) and the
 * call is re-run from that iteration by the next synchronising entry point with the
 * value now known, so results never depend on the guess (Q is a ping-pong pair on
 * such handles).  SPGG_NO_SPEC=1 in the environment keeps the exact pair. */
int spgg_step(spgg_t *h, int n_steps, void *cuda_stream);
int spgg_sync(spgg_t *h);

/* Statistic rows of the last spgg_step call: rows [first, first+n) relative
 * to the iteration index at the start of that call (row 0 = starting state:
 * only SPGG_ST_SUM_R is meaningful; row k = iteration start+k). */
int spgg_get_stats(spgg_t *h, int replica, int first, int n, double *rows_out);
int spgg_query(spgg_t *h, int replica, spgg_status_t *out);

/* Which kernels serve this handle, as text ("resident: cluster of 16 CTAs x 352 threads ...",
 * "resident: cooperative grid of 148 CTAs ...", "fast: TMA-staged tiles ...", "general: ...").
 * Writes at most n bytes including the terminating NUL; returns the length it needed. */
int spgg_describe(spgg_t *h, char *buf, int n);

/* Strip decomposition (multi-GPU): boundary rows <-> ghost rows.  pack copies
 * the rows a neighbour needs into two contiguous device buffers of
 * spgg_halo_bytes() each (up = towards row0-1, down = towards row0+rows);
 * unpack fills this strip's ghost rows from the neighbours' buffers. */
int64_t spgg_halo_bytes(spgg_t *h);
int spgg_halo_pack(spgg_t *h, void *dev_to_up, void *dev_to_down, void *cuda_stream);
int spgg_halo_unpack(spgg_t *h, const void *dev_from_up, const void *dev_from_down,
                     void *cuda_stream);
/* Phase-split stepping for strips: select (K with update of iteration j when
 * j>0), then halo exchange, then gmax partial, then all-reduce(max) of the
 * value at spgg_gmax_device_ptr(), repeat. */
int spgg_phase_kernel(spgg_t *h, int do_update, int do_select, void *cuda_stream);
int spgg_phase_gmax(spgg_t *h, void *cuda_stream);
/* One whole iteration inside begin/end: what spgg_step does per iteration (a single
 * speculative launch when the handle can guess the maximum, else k_gmax_* + k_step*). */
int spgg_phase_iteration(spgg_t *h, int do_select, void *cuda_stream);
void *spgg_gmax_device_ptr(spgg_t *h);
/* Strips and the one-launch iteration: the maximum and the uniform-lattice test
 * (spgg.py:405,488) are lattice-global, so a strip's update launch only reports
 * {its own maximum, holds-a-defecting-action, holds-a-cooperating-action, 0} at
 * spgg_strip_report_ptr() (4 floats, device); the ranks max-reduce that vector and
 * spgg_strip_verify() then compares the maximum with the guess, keeps it as the next
 * guess and raises the stop flag.  Per iteration: [spgg_strip_iteration, or the exact
 * pair when spgg_strip_can_speculate() says 0] -> all-reduce(MAX) of the report ->
 * spgg_strip_verify; the halo exchange runs beside the reduce.  After the chunk:
 * spgg_strip_failed() (same answer on every rank) and, if non-zero,
 * spgg_strip_rewind() + the iterations from there again. */
/* Peer-mapped halos (one process per GPU, NVLink): spgg_ipc_export() writes the
 * cudaIpc handles of this strip's six planes (6 x 64 bytes).  A strip attaches the
 * handles of the strip ABOVE it (the owner of row row0-1) with which = 0 and those
 * of the strip BELOW it with which = 1; peer_rows is the number of rows that
 * neighbour owns.  Once both sides are attached every selecting launch of the fast
 * path stores its first / last two rows straight into the neighbours' ghost rows,
 * and the halo pack / send / unpack between launches is not needed (the report
 * all-reduce orders the launches of different GPUs). */
int spgg_ipc_export(spgg_t *h, unsigned char *handles_6x64);
int spgg_ipc_attach(spgg_t *h, int which, const unsigned char *handles_6x64, int peer_rows, int same_as_other);
/* ... and the report itself: with spgg_ring_export / spgg_ring_attach (handles of
 * ALL ranks, in rank order) the last CTA of a launch max-combines its report into a
 * ring slot of every rank with system-scope atomics and counts itself in;
 * spgg_strip_verify() then only waits (on the device) until all ranks are in.  No
 * collective-library call between two launches of the steady state.  A state
 * upload (spgg_set_state / spgg_init_random) and spgg_strip_rewind empty the ring:
 * the caller synchronises the ranks (a barrier) between that and the next launch,
 * and before destroying a handle whose planes and ring the neighbours still map. */
int spgg_ring_export(spgg_t *h, unsigned char *handle64);
int spgg_ring_attach(spgg_t *h, int world, int rank, const unsigned char *handles_world_x64);
int spgg_strip_can_speculate(spgg_t *h, int do_select);
int spgg_strip_iteration(spgg_t *h, int do_select, void *cuda_stream);
void *spgg_strip_report_ptr(spgg_t *h);
int spgg_strip_verify(spgg_t *h, void *cuda_stream);
int spgg_strip_failed(spgg_t *h);
int spgg_strip_rewind(spgg_t *h, int first_failed_launch);
int spgg_begin_steps(spgg_t *h, int n_steps, void *cuda_stream);
int spgg_end_steps(spgg_t *h, void *cuda_stream);

const char *spgg_last_error(void);
int spgg_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SPGG_B200_H */
