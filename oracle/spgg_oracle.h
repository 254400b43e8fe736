/* TEST INFRASTRUCTURE ONLY - C restatement of the reference SPGG step.
 * See spgg_oracle.c for the parity status and the reference citations.
 * Nothing under the product package may include, link or load this. */
#ifndef SPGG_ORACLE_H
#define SPGG_ORACLE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* stat-row layout; identical to the device row layout (include/spgg.h) so the
 * parity tests can compare rows column by column. */
enum {
  OST_NC_OLD = 0,      /* #cooperators before the action (S_{t-1})            spgg.py:383 */
  OST_N_CD = 1,        /* C -> D switches                                      spgg.py:419 */
  OST_N_DC = 2,        /* D -> C switches                                      spgg.py:420 */
  OST_NC_NEW = 3,      /* #sites whose action is cooperate                               */
  OST_SUM_P = 4,       /* sum of normalised payoff P                           spgg.py:388 */
  OST_SUM_P_C = 5,     /* ... over sites with S_{t-1}==C                       spgg.py:389 */
  OST_SUM_P_D = 6,     /* ... over sites with S_{t-1}==D                       spgg.py:390 */
  OST_SUM_WP_P = 7,    /* sum of w_P*P                                         spgg.py:425 */
  OST_SUM_REW_C = 8,   /* sum of reward over a==C                              spgg.py:542 */
  OST_SUM_REW_D = 9,   /* sum of reward over a==D                              spgg.py:543 */
  OST_SUM_RATIO = 10,  /* sum over a==C of |wR*0.5|/(|rew|+1e-9)*100           spgg.py:529-536 */
  OST_GROUP0 = 11,     /* 11..16: #groups with k defectors (k=0..5) in S_t     spgg.py:586-592 */
  OST_SUM_R = 17,      /* sum of R before the action (R_{t-1})                 spgg.py:394 */
  OST_SUM_Q = 18,      /* 18..21: sum of Q[:,:,s,a] after both updates         spgg.py:562-565 */
  OST_SUM_Q_C = 22,    /* 22..25: same over S_{t-1}==C                         spgg.py:568-583 */
  OST_SUM_Q_D = 26,    /* 26..29: same over S_{t-1}==D                                    */
  OST_SUM_NI = 30,     /* sum of neighbour-influence percent                   spgg.py:512 */
  OST_N_BEST_POS = 31, /* #sites with max_diff > 0                             spgg.py:521 */
  OST_N_BEST_2ND = 32, /* ... whose arg-max neighbour is second order          spgg.py:520 */
  OST_GMAX = 33,       /* lattice-global max |diff|                            spgg.py:488 */
  OST_NSTAT = 40
};

/* TD rules: the codes of include/spgg.h (SPGG_ALGO_*) */
enum { OALGO_QLEARNING = 0, OALGO_SARSA = 1, OALGO_EXPECTED_SARSA = 2, OALGO_DOUBLE_QLEARNING = 3 };

typedef struct {
  int32_t L;
  int32_t M;          /* 1 or 2 (use_second_order)           */
  int32_t state_mode; /* 0 = reputation, 1 = action          */
  int32_t algorithm;  /* OALGO_*                             */
  double r, c, cost;
  double alpha, gamma;
  double kappa;       /* influence_factor                    */
  double lambda_eps;
  double rep_gain_C, delta_R_D, R_min, R_max;
  double wP;          /* reward_weight_payoff                */
} oracle_params_t;

/* One iteration, fp64, reference operation order, replayed draws.
 * S: L*L bytes (0=C, 1=D); R: L*L doubles; Q: L*L*4 doubles laid out (s,a), or for
 * Double Q-learning L*L*8 laid out (table,s,a), the two tables of a site side by side.
 * u,b: that iteration's draw pairs, pair k at u + k*L*L (algorithms.py:105,108).  Q-learning
 * and Expected SARSA draw one pair; SARSA three (action, next action of the update, next
 * action of the NI statistic: spgg.py:410,433,452); Double Q-learning two, the table choice
 * being u of pair 1 (update table 1 <=> u < 0.5, algorithms.py:302).
 * If u == NULL the draws come from Philox4x32-10 with the integer threshold thr24
 * (explore <=> (word>>8) < thr24; random action = word&1): the action from counter
 * (j/4, i, step, 0), SARSA's next actions from (j/4, i, step, 1) and (j/4, i, step, 2),
 * Double Q's table choice from (j/4, i, step, 1) (table 1 <=> (word>>8) < 2^23).
 * eps / thr24 are those of iteration `step`: the select and SARSA's / Expected SARSA's
 * policy of the next state use the same epsilon.
 * stats: OST_NSTAT doubles (may be NULL); the Q sums are over the mean of the two tables
 * for Double Q-learning (algorithms.py:263). Returns 0. */
int oracle_step_f64(const oracle_params_t *p, uint8_t *S, double *R, double *Q,
                    double eps, const double *u, const uint8_t *b,
                    uint64_t seed, uint32_t step, uint32_t thr24, double *stats);

/* One iteration with the throughput-mode arithmetic: fp32 Q, fp32 R, rewards
 * from the integer table rew[SigmaN][C_old][coop_new] (exact-count payoff),
 * explicit fmaf, Philox draws (or replayed u,b when u != NULL; u compared in
 * double against eps).  Draws, Q layout and TD rules as oracle_step_f64. */
int oracle_step_f32(const oracle_params_t *p, uint8_t *S, float *R, float *Q,
                    double eps, const double *u, const uint8_t *b,
                    uint64_t seed, uint32_t step, uint32_t thr24, double *stats);

/* Philox4x32-10, exposed for known-answer tests. */
void oracle_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);

/* the Philox word both step functions draw for site (i,j) at iteration `step` from stream
 * `stream` (0: action, 1 and 2: SARSA's next actions, 1: Double Q's table choice) */
uint32_t oracle_site_word(uint64_t seed, uint32_t step, uint32_t stream, int i, int j);

/* explore threshold used by both implementations: ceil(eps * 2^24) clamped to [0, 2^24] */
uint32_t oracle_thr24(double eps);

/* reward table of the throughput mode: 128 floats indexed (SigmaN<<2 | C_old<<1 | coop_new) */
void oracle_reward_table(const oracle_params_t *p, float *tab128);

int oracle_num_threads(void);

/* spgg_state_digest restated (csrc/spgg_kernels.cuh: k_state_digest): out[0] strategies, out[1]
 * reputations, out[2] Q, each the sum mod 2^64 over sites of (hash | 1) * (value bits + 1).
 * S: bytes (0 = C, else D); R, Q (nq = 4 or 8 per site): the values as the device holds them,
 * widened to double (int8 units times rq, fp32, fp64).  Q == NULL leaves out[2] = 0.
 * period == 0: the arrays hold `rows` rows of an L-wide lattice starting at global row row0.
 * period == P: they hold a P x P state, and the digest is that of the L x L lattice (L % P == 0,
 * rows from row0) whose site (i, j) holds the value of (i % P, j % P).
 * w: NULL, or the multipliers oracle_digest_weights computed for the same geometry, which makes
 * repeated digests of a periodic lattice cost P*P instead of L*L hashes.  Returns 0, or -1 when
 * P does not divide L. */
int oracle_state_digest(int L, int row0, int rows, int period, int nq, const uint8_t *S,
                        const double *R, const double *Q, const uint64_t *w, uint64_t out[3]);
/* w: (rows * L or P * P) * (2 + nq) multipliers, per slot S, R, Q[0..nq) */
int oracle_digest_weights(int L, int row0, int rows, int period, int nq, uint64_t *w);

/* spgg_init_random restated (k_init_random): rows [row0, row0 + rows) of an L x L lattice.  Q
 * entry z of table t at site (i, j) from Philox counter (j, i, t, 1) word z, rounded to float
 * when fp32; strategy word w of row i from counter (w / 4, i, 0, 2) word w % 4, bits beyond
 * column L - 1 masked; R = 0. */
void oracle_init_random(int L, int row0, int rows, int nq, int fp32, uint64_t seed, uint8_t *S, double *R,
                        double *Q);
/* the digest of that state, without holding it: for lattices too large for host memory */
int oracle_init_random_digest(int L, int row0, int rows, int nq, int fp32, uint64_t seed, uint64_t out[3]);

/* actions (0 = C, 1 = D) of rows [i0, i1) at iteration `step` when epsilon = 1: every site
 * explores, and its action is bit 0 of its stream-0 Philox word (oracle_site_word) */
void oracle_explore_actions(int L, int i0, int i1, uint64_t seed, uint32_t step, uint8_t *a);

#ifdef __cplusplus
}
#endif
#endif
