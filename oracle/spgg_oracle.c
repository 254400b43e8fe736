/* TEST INFRASTRUCTURE ONLY.
 *
 * Plain-C, per-site restatement of one iteration of the reference's SPGG loop
 * (reference paths relative to /root/reference):
 *   src/model/spgg.py:368-592   (SPGG.run loop body)
 *   src/model/algorithms.py:96-133 (QLearning.select_action / update_q_table)
 *   src/model/algorithms.py:136-341 (SARSA, Expected SARSA, Double Q-learning), applied as
 *   spgg.py:431-473,498-505, in the operation order of oracle/spgg_numpy.py
 * It is the checker for the CUDA path; the product never links or loads it.
 * Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs do.
 *
 * Parity status: PINNED.  oracle_step_f64 is compared bit-for-bit (S, R, Q and
 * the integer statistics) against the executed reference through
 * oracle/spgg_numpy.py, the golden fixtures in tests/golden/ and, inside the
 * build container, the reference itself (tests/test_oracle_vs_reference.py).
 * The reference has no tests/golden vectors of its own (SURVEY.md section 4).
 *
 * oracle_step_f32 restates the *throughput-mode* arithmetic of the CUDA
 * kernel (fp32 Q, exact-count reward table, explicit fmaf, Philox draws); it
 * has no bit-level counterpart in the reference and is pinned statistically
 * (cooperation-rate curves inside the reference's seed-to-seed band) and
 * against oracle_step_f64 on dyadic parameter sets where both are exact.  For every TD rule
 * it follows k_step (csrc/spgg_kernels.cuh: td_update_f32 and the Double-Q branch).
 *
 * The end of the file restates two helpers of the C ABI that the large-lattice tests check
 * against: spgg_state_digest (also for a lattice that tiles a smaller state) and
 * spgg_init_random, plus the actions of an iteration at epsilon = 1.
 *
 * Build with -ffp-contract=off (see oracle/Makefile): the reference is NumPy,
 * every operation is individually rounded.
 */
#include "spgg_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* neighbour offsets (dx,dy) in the reference's enumeration order;
 * neighbour k of (i,j) is (i-dx, j-dy) because np.roll(X,(dx,dy))[i,j]==X[i-dx,j-dy].
 * spgg.py:479-485 */
static const int OFF[12][2] = {{1, 0},  {-1, 0}, {0, 1},  {0, -1}, {2, 0},  {-2, 0},
                               {0, 2},  {0, -2}, {1, 1},  {1, -1}, {-1, 1}, {-1, -1}};
/* groups a site belongs to, in the summation order of spgg.py:373-377:
 * centres (i,j), (i-1,j), (i+1,j), (i,j-1), (i,j+1) */
static const int GRP[5][2] = {{0, 0}, {-1, 0}, {1, 0}, {0, -1}, {0, 1}};

static inline int wrapi(int a, int L) {
  a %= L;
  return a < 0 ? a + L : a;
}
#define IDX(i, j) ((size_t)wrapi((i), L) * (size_t)L + (size_t)wrapi((j), L))

int oracle_num_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

/* ---------------------------------------------------------------- Philox */
static inline void philox_round(uint32_t c[4], const uint32_t k[2]) {
  const uint64_t p0 = (uint64_t)0xD2511F53u * c[0];
  const uint64_t p1 = (uint64_t)0xCD9E8D57u * c[2];
  const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k[0];
  const uint32_t n1 = (uint32_t)p1;
  const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k[1];
  const uint32_t n3 = (uint32_t)p0;
  c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
}

void oracle_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  uint32_t c[4] = {ctr[0], ctr[1], ctr[2], ctr[3]};
  uint32_t k[2] = {key[0], key[1]};
  for (int r = 0; r < 10; ++r) {
    philox_round(c, k);
    k[0] += 0x9E3779B9u;
    k[1] += 0xBB67AE85u;
  }
  memcpy(out, c, sizeof(c));
}

uint32_t oracle_thr24(double eps) {
  double t = ceil(eps * 16777216.0);
  if (t < 0) t = 0;
  if (t > 16777216.0) t = 16777216.0;
  return (uint32_t)t;
}

/* draw word of site (i,j) at iteration `step` from stream `stream`: counter = (j>>2, row, step,
 * stream), word index j&3 - one Philox call serves four consecutive sites of a row.  Stream 0 is
 * the action, streams 1 and 2 the further draws of SARSA and Double Q-learning. */
static inline uint32_t site_word(uint64_t seed, uint32_t step, uint32_t stream, int i, int j) {
  uint32_t ctr[4] = {(uint32_t)(j >> 2), (uint32_t)i, step, stream};
  uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
  uint32_t w[4];
  oracle_philox4x32_10(ctr, key, w);
  return w[j & 3];
}

uint32_t oracle_site_word(uint64_t seed, uint32_t step, uint32_t stream, int i, int j) {
  return site_word(seed, step, stream, i, j);
}

/* the update's further draws of site (i,j): SARSA's next actions for the TD target (ex1, rn1)
 * and for the NI statistic (ex2, rn2), spgg.py:433,452; Double Q's table choice upd1,
 * algorithms.py:302.  Replayed: pairs 1 and 2 of u, b (n_sites apart).  Philox: streams 1, 2. */
typedef struct {
  int ex1, rn1, ex2, rn2, upd1;
} td_draws_t;

static td_draws_t td_draws(int algo, double eps, const double *u, const uint8_t *b, size_t n_sites,
                           uint64_t seed, uint32_t step, uint32_t thr24, int i, int j, size_t x) {
  td_draws_t d = {0, 0, 0, 0, 0};
  if (algo == OALGO_SARSA) {
    if (u) {
      d.ex1 = (u[n_sites + x] < eps); d.rn1 = b[n_sites + x];
      d.ex2 = (u[2 * n_sites + x] < eps); d.rn2 = b[2 * n_sites + x];
    } else {
      const uint32_t w1 = site_word(seed, step, 1u, i, j), w2 = site_word(seed, step, 2u, i, j);
      d.ex1 = ((w1 >> 8) < thr24); d.rn1 = (int)(w1 & 1u);
      d.ex2 = ((w2 >> 8) < thr24); d.rn2 = (int)(w2 & 1u);
    }
  } else if (algo == OALGO_DOUBLE_QLEARNING) {
    if (u) d.upd1 = (u[n_sites + x] < 0.5);
    else d.upd1 = ((site_word(seed, step, 1u, i, j) >> 8) < (1u << 23));
  }
  return d;
}

/* value of the next state's row (x0, x1) in the TD target: max (algorithms.py:125), Q[s',a']
 * with a' eps-greedy (:142-150,169) or the eps-greedy expectation (:212-224), in the order of
 * oracle/spgg_numpy.py */
static double next_f64(int algo, double x0, double x1, double eps, int ex, int rn) {
  if (algo == OALGO_QLEARNING) return fmax(x0, x1);
  const int greedy = (x1 > x0) ? 1 : 0;
  if (algo == OALGO_SARSA) return (ex ? rn : greedy) ? x1 : x0;
  const double po = eps / 2.0, pg = (1.0 - eps) + po;
  return (greedy ? po : pg) * x0 + (greedy ? pg : po) * x1;
}

/* the same in the kernel's fp32 arithmetic (k_step: next_value; epsilon rounded to float once) */
static float next_f32(int algo, float x0, float x1, float e, int ex, int rn) {
  if (algo == OALGO_QLEARNING) return fmaxf(x0, x1);
  const int greedy = (x1 > x0) ? 1 : 0;
  if (algo == OALGO_SARSA) return (ex ? rn : greedy) ? x1 : x0;
  const float po = e * 0.5f, pg = (1.0f - e) + po;
  return fmaf(greedy ? pg : po, x1, (greedy ? po : pg) * x0);
}

/* k_step's q_max: the first argument on a tie */
static inline float qmaxf(float x, float y) { return x > y ? x : (y > x ? y : x); }

/* ------------------------------------------------------------ shared bits */
static void count_groups(int L, const uint8_t *S, uint8_t *N) {
  /* spgg.py:23-36 on the cooperator mask */
#pragma omp parallel for schedule(static)
  for (int i = 0; i < L; ++i)
    for (int j = 0; j < L; ++j) {
      int n = (S[IDX(i, j)] == 0) + (S[IDX(i + 1, j)] == 0) + (S[IDX(i - 1, j)] == 0) +
              (S[IDX(i, j + 1)] == 0) + (S[IDX(i, j - 1)] == 0);
      N[(size_t)i * L + j] = (uint8_t)n;
    }
}

static void zero_stats(double *st) {
  if (st) memset(st, 0, sizeof(double) * OST_NSTAT);
}

/* =================================================================== fp64 */
int oracle_step_f64(const oracle_params_t *p, uint8_t *S, double *R, double *Q, double eps,
                    const double *u, const uint8_t *b, uint64_t seed, uint32_t step,
                    uint32_t thr24, double *stats) {
  const int L = p->L;
  const size_t n_sites = (size_t)L * L;
  const int nk = (p->M == 2) ? 12 : 4;
  const int nst = nk + 1;
  const double rc = p->r * p->c;
  double g[6];
  for (int n = 0; n < 6; ++n) g[n] = rc * (double)n / 5.0; /* spgg.py:256 */
  const double lo = p->r - 5.0;                            /* spgg.py:149 */
  const double span = 4.0 * p->r - lo;                     /* spgg.py:148,377 */
  const double wP = p->wP, wR = 1.0 - p->wP;               /* spgg.py:108 */
  const int algo = p->algorithm, dq = (algo == OALGO_DOUBLE_QLEARNING), nq = dq ? 8 : 4;

  uint8_t *N = (uint8_t *)malloc(n_sites);
  uint8_t *a = (uint8_t *)malloc(n_sites);
  uint8_t *s_old = (uint8_t *)malloc(n_sites);
  uint8_t *s_new = (uint8_t *)malloc(n_sites);
  double *Rn = (double *)malloc(n_sites * sizeof(double));
  double *P = (double *)malloc(n_sites * sizeof(double));
  double *rew = (double *)malloc(n_sites * sizeof(double));
  zero_stats(stats);

  count_groups(L, S, N);

  /* payoff of the configuration before the action: spgg.py:373-377 */
#pragma omp parallel for schedule(static)
  for (int i = 0; i < L; ++i)
    for (int j = 0; j < L; ++j) {
      const size_t x = (size_t)i * L + j;
      const double C = (S[x] == 0) ? 1.0 : 0.0, D = 1.0 - C;
      double tot = 0.0;
      for (int q = 0; q < 5; ++q) {
        const double share = g[N[IDX(i + GRP[q][0], j + GRP[q][1])]];
        const double term = (share - p->cost) * C + share * D;
        tot = (q == 0) ? term : tot + term;
      }
      P[x] = (tot - lo) / span;
    }

  /* state, action, reputation: spgg.py:409-415, algorithms.py:102-110 */
#pragma omp parallel for schedule(static)
  for (int i = 0; i < L; ++i)
    for (int j = 0; j < L; ++j) {
      const size_t x = (size_t)i * L + j;
      int s;
      if (p->state_mode == 1) {
        s = (S[x] == 0);
      } else {
        double acc = 0.0;
        acc += R[x];
        for (int k = 0; k < nk; ++k) acc += R[IDX(i - OFF[k][0], j - OFF[k][1])];
        s = (acc / (double)nst > 0.0);
      }
      s_old[x] = (uint8_t)s;
      int explore, rnd;
      if (u) {
        explore = (u[x] < eps);
        rnd = b[x];
      } else {
        const uint32_t w = site_word(seed, step, 0u, i, j);
        explore = ((w >> 8) < thr24);
        rnd = (int)(w & 1u);
      }
      const double *q = Q + nq * x + 2 * s;
      int greedy;
      if (dq) /* the policy acts on the mean of the two tables (algorithms.py:263,283-290) */
        greedy = ((q[1] + q[5]) / 2.0 > (q[0] + q[4]) / 2.0) ? 1 : 0;
      else
        greedy = (q[1] > q[0]) ? 1 : 0; /* np.argmax: first max */
      a[x] = (uint8_t)(explore ? rnd : greedy);
      double rn = R[x] + (a[x] == 0 ? p->rep_gain_C : -p->delta_R_D); /* spgg.py:321 */
      rn = fmax(rn, p->R_min);
      rn = fmin(rn, p->R_max);
      Rn[x] = rn;
    }

  /* new state + rewards: spgg.py:423-427 */
#pragma omp parallel for schedule(static)
  for (int i = 0; i < L; ++i)
    for (int j = 0; j < L; ++j) {
      const size_t x = (size_t)i * L + j;
      int s;
      if (p->state_mode == 1) {
        s = (a[x] == 0);
      } else {
        double acc = 0.0;
        acc += Rn[x];
        for (int k = 0; k < nk; ++k) acc += Rn[IDX(i - OFF[k][0], j - OFF[k][1])];
        s = (acc / (double)nst > 0.0);
      }
      s_new[x] = (uint8_t)s;
      const double rr = (a[x] == 0) ? 0.5 : 0.0;
      rew[x] = wP * P[x] + wR * rr;
    }

  /* lattice-global max |diff|: spgg.py:486-488 */
  double gmax = 0.0;
#pragma omp parallel for schedule(static) reduction(max : gmax)
  for (int i = 0; i < L; ++i)
    for (int j = 0; j < L; ++j) {
      const size_t x = (size_t)i * L + j;
      for (int k = 0; k < nk; ++k) {
        const double d = fabs(rew[IDX(i - OFF[k][0], j - OFF[k][1])] - rew[x]);
        if (d > gmax) gmax = d;
      }
    }

  /* updates + statistics */
  double acc_st[OST_NSTAT];
  memset(acc_st, 0, sizeof(acc_st));
  /* plain sequential accumulation: statistics are compared with a tolerance */
  for (int i = 0; i < L; ++i)
    for (int j = 0; j < L; ++j) {
      const size_t x = (size_t)i * L + j;
      const int s = s_old[x], sn = s_new[x], act = a[x], e = 2 * s + act;
      const td_draws_t dr = td_draws(algo, eps, u, b, n_sites, seed, step, thr24, i, j, x);
      double best = 0.0;
      int kstar = 0;
      for (int k = 0; k < nk; ++k) {
        const double d = rew[IDX(i - OFF[k][0], j - OFF[k][1])] - rew[x];
        if (k == 0 || d > best) {
          best = d;
          kstar = k;
        }
      }
      const double lam = p->kappa * fmax(0.0, best) / (gmax + p->lambda_eps); /* spgg.py:489 */
      const int a_star = a[IDX(i - OFF[kstar][0], j - OFF[kstar][1])];
      const double nu = lam * ((a_star == act) ? 1.0 : -1.0);
      double *q = Q + nq * x;
      double td2, qm[4];
      const double *qs = q; /* the table the statistics see */
      if (dq) {
        /* algorithms.py:292-341: the chosen table's target is the other table's row maximum of s' */
        double *qa = q, *qb = q + 4;
        const double nxa = fmax(qb[2 * sn], qb[2 * sn + 1]), nxb = fmax(qa[2 * sn], qa[2 * sn + 1]);
        if (dr.upd1) qa[e] = qa[e] + p->alpha * (rew[x] + p->gamma * nxa - qa[e]);
        else qb[e] = qb[e] + p->alpha * (rew[x] + p->gamma * nxb - qb[e]);
        /* TD error of the combined table after the write (spgg.py:464-468) */
        for (int z = 0; z < 4; ++z) qm[z] = (qa[z] + qb[z]) / 2.0;
        td2 = rew[x] + p->gamma * fmax(qm[2 * sn], qm[2 * sn + 1]) - qm[e];
        qa[e] += nu; /* spgg.py:498-505: both tables */
        qb[e] += nu;
        for (int z = 0; z < 4; ++z) qm[z] = (qa[z] + qb[z]) / 2.0;
        qs = qm;
      } else {
        const double q0 = q[e];
        const double mx = next_f64(algo, q[2 * sn], q[2 * sn + 1], eps, dr.ex1, dr.rn1);
        const double td = rew[x] + p->gamma * mx - q0; /* algorithms.py:128 */
        const double qtd = q0 + p->alpha * td;         /* algorithms.py:131 */
        /* NI statistic uses the table after the TD write (spgg.py:446-473,512) */
        q[e] = qtd;
        const double mx2 = next_f64(algo, q[2 * sn], q[2 * sn + 1], eps, dr.ex2, dr.rn2);
        td2 = rew[x] + p->gamma * mx2 - qtd;
        q[e] = qtd + nu; /* spgg.py:509 */
      }
      const double pct = fabs(nu) / (fabs(p->alpha * td2) + fabs(nu) + 1e-8) * 100.0;

      const int wasC = (S[x] == 0);
      acc_st[OST_NC_OLD] += wasC;
      acc_st[OST_N_CD] += (wasC && act == 1);
      acc_st[OST_N_DC] += (!wasC && act == 0);
      acc_st[OST_NC_NEW] += (act == 0);
      acc_st[OST_SUM_P] += P[x];
      acc_st[wasC ? OST_SUM_P_C : OST_SUM_P_D] += P[x];
      acc_st[OST_SUM_WP_P] += wP * P[x];
      acc_st[act == 0 ? OST_SUM_REW_C : OST_SUM_REW_D] += rew[x];
      if (act == 0) acc_st[OST_SUM_RATIO] += fabs(wR * 0.5) / (fabs(rew[x]) + 1e-9) * 100.0;
      acc_st[OST_SUM_R] += R[x];
      for (int z = 0; z < 4; ++z) {
        acc_st[OST_SUM_Q + z] += qs[z];
        acc_st[(wasC ? OST_SUM_Q_C : OST_SUM_Q_D) + z] += qs[z];
      }
      acc_st[OST_SUM_NI] += pct;
      if (best > 0.0) {
        acc_st[OST_N_BEST_POS] += 1;
        acc_st[OST_N_BEST_2ND] += (kstar >= 4);
      }
      const int nd = (a[IDX(i, j)] == 1) + (a[IDX(i + 1, j)] == 1) + (a[IDX(i - 1, j)] == 1) +
                     (a[IDX(i, j + 1)] == 1) + (a[IDX(i, j - 1)] == 1);
      acc_st[OST_GROUP0 + nd] += 1;
    }
  acc_st[OST_GMAX] = gmax;
  if (stats) memcpy(stats, acc_st, sizeof(acc_st));

  memcpy(S, a, n_sites);
  memcpy(R, Rn, n_sites * sizeof(double));
  free(N); free(a); free(s_old); free(s_new); free(Rn); free(P); free(rew);
  return 0;
}

/* =================================================================== fp32 */
void oracle_reward_table(const oracle_params_t *p, float *tab) {
  const double rc = p->r * p->c;
  const double lo = p->r - 5.0, span = 4.0 * p->r - lo;
  const double wP = p->wP, wR = 1.0 - p->wP;
  for (int code = 0; code < 128; ++code) {
    const int sn = code >> 2, C = (code >> 1) & 1, coop = code & 1;
    /* exact-count payoff: sum over the 5 groups of (rc*N/5 - cost*C) */
    const double tot = rc * (double)sn / 5.0 - (C ? 5.0 * p->cost : 0.0);
    const double P = (tot - lo) / span;
    tab[code] = (float)(wP * P + wR * (coop ? 0.5 : 0.0));
  }
}

static double payoff_from_count(const oracle_params_t *p, int sn, int C) {
  const double rc = p->r * p->c;
  const double lo = p->r - 5.0, span = 4.0 * p->r - lo;
  const double tot = rc * (double)sn / 5.0 - (C ? 5.0 * p->cost : 0.0);
  return (tot - lo) / span;
}

int oracle_step_f32(const oracle_params_t *p, uint8_t *S, float *R, float *Q, double eps,
                    const double *u, const uint8_t *b, uint64_t seed, uint32_t step,
                    uint32_t thr24, double *stats) {
  const int L = p->L;
  const size_t n_sites = (size_t)L * L;
  const int nk = (p->M == 2) ? 12 : 4;
  const int nst = nk + 1;
  const float alpha = (float)p->alpha, gamma = (float)p->gamma, kappa = (float)p->kappa;
  const float leps = (float)p->lambda_eps;
  const float gainC = (float)p->rep_gain_C, lossD = (float)p->delta_R_D;
  const float rmin = (float)p->R_min, rmax = (float)p->R_max;
  const double wP = p->wP, wR = 1.0 - p->wP;
  const int algo = p->algorithm, dq = (algo == OALGO_DOUBLE_QLEARNING), nq = dq ? 8 : 4;
  float tab[128];
  oracle_reward_table(p, tab);

  uint8_t *N = (uint8_t *)malloc(n_sites);
  uint8_t *SN = (uint8_t *)malloc(n_sites);
  uint8_t *a = (uint8_t *)malloc(n_sites);
  uint8_t *s_old = (uint8_t *)malloc(n_sites);
  uint8_t *s_new = (uint8_t *)malloc(n_sites);
  float *Rn = (float *)malloc(n_sites * sizeof(float));
  float *rew = (float *)malloc(n_sites * sizeof(float));
  zero_stats(stats);

  count_groups(L, S, N);
#pragma omp parallel for schedule(static)
  for (int i = 0; i < L; ++i)
    for (int j = 0; j < L; ++j) {
      int sn = 0;
      for (int q = 0; q < 5; ++q) sn += N[IDX(i + GRP[q][0], j + GRP[q][1])];
      SN[(size_t)i * L + j] = (uint8_t)sn;
    }

#pragma omp parallel for schedule(static)
  for (int i = 0; i < L; ++i)
    for (int j = 0; j < L; ++j) {
      const size_t x = (size_t)i * L + j;
      int s;
      if (p->state_mode == 1) {
        s = (S[x] == 0);
      } else {
        float acc = R[x];
        for (int k = 0; k < nk; ++k) acc += R[IDX(i - OFF[k][0], j - OFF[k][1])];
        s = (acc / (float)nst > 0.0f);
      }
      s_old[x] = (uint8_t)s;
      int explore, rnd;
      if (u) {
        explore = (u[x] < eps);
        rnd = b[x];
      } else {
        const uint32_t w = site_word(seed, step, 0u, i, j);
        explore = ((w >> 8) < thr24);
        rnd = (int)(w & 1u);
      }
      const float *q = Q + nq * x + 2 * s;
      int greedy;
      if (dq) /* k_step's q_mean of the two tables */
        greedy = ((q[1] + q[5]) / 2.0f > (q[0] + q[4]) / 2.0f) ? 1 : 0;
      else
        greedy = (q[1] > q[0]) ? 1 : 0;
      a[x] = (uint8_t)(explore ? rnd : greedy);
      float rn = R[x] + (a[x] == 0 ? gainC : -lossD);
      rn = fmaxf(rn, rmin);
      rn = fminf(rn, rmax);
      Rn[x] = rn;
    }

#pragma omp parallel for schedule(static)
  for (int i = 0; i < L; ++i)
    for (int j = 0; j < L; ++j) {
      const size_t x = (size_t)i * L + j;
      int s;
      if (p->state_mode == 1) {
        s = (a[x] == 0);
      } else {
        float acc = Rn[x];
        for (int k = 0; k < nk; ++k) acc += Rn[IDX(i - OFF[k][0], j - OFF[k][1])];
        s = (acc / (float)nst > 0.0f);
      }
      s_new[x] = (uint8_t)s;
      rew[x] = tab[(SN[x] << 2) | ((S[x] == 0) << 1) | (a[x] == 0)];
    }

  float gmax = 0.0f;
#pragma omp parallel for schedule(static) reduction(max : gmax)
  for (int i = 0; i < L; ++i)
    for (int j = 0; j < L; ++j) {
      const size_t x = (size_t)i * L + j;
      for (int k = 0; k < nk; ++k) {
        const float d = fabsf(rew[IDX(i - OFF[k][0], j - OFF[k][1])] - rew[x]);
        if (d > gmax) gmax = d;
      }
    }
  const float inv_den = 1.0f / (gmax + leps);

  double acc_st[OST_NSTAT];
  memset(acc_st, 0, sizeof(acc_st));
  for (int i = 0; i < L; ++i)
    for (int j = 0; j < L; ++j) {
      const size_t x = (size_t)i * L + j;
      const int s = s_old[x], sn = s_new[x], act = a[x], e = 2 * s + act;
      const td_draws_t dr = td_draws(algo, eps, u, b, n_sites, seed, step, thr24, i, j, x);
      float best = 0.0f;
      int kstar = 0;
      for (int k = 0; k < nk; ++k) {
        const float d = rew[IDX(i - OFF[k][0], j - OFF[k][1])] - rew[x];
        if (k == 0 || d > best) {
          best = d;
          kstar = k;
        }
      }
      const float lam = (kappa * fmaxf(0.0f, best)) * inv_den;
      const int a_star = a[IDX(i - OFF[kstar][0], j - OFF[kstar][1])];
      const float nu = (a_star == act) ? lam : -lam;
      float *q = Q + nq * x;
      float td2, qm[4];
      const float *qs = q; /* the table the statistics see */
      if (dq) {
        /* k_step's Double-Q branch: separately rounded products and sums, means by division */
        float *t1 = q, *t2 = q + 4;
        const float nx1 = qmaxf(t2[2 * sn], t2[2 * sn + 1]), nx2 = qmaxf(t1[2 * sn], t1[2 * sn + 1]);
        if (dr.upd1) t1[e] = t1[e] + alpha * ((rew[x] + gamma * nx1) - t1[e]);
        else t2[e] = t2[e] + alpha * ((rew[x] + gamma * nx2) - t2[e]);
        for (int z = 0; z < 4; ++z) qm[z] = (t1[z] + t2[z]) / 2.0f;
        td2 = (rew[x] + gamma * qmaxf(qm[2 * sn], qm[2 * sn + 1])) - qm[e];
        t1[e] = t1[e] + nu;
        t2[e] = t2[e] + nu;
        for (int z = 0; z < 4; ++z) qm[z] = (t1[z] + t2[z]) / 2.0f;
        qs = qm;
      } else {
        /* td_update_f32 */
        const float ef = (float)eps;
        const float q0 = q[e];
        const float mx = next_f32(algo, q[2 * sn], q[2 * sn + 1], ef, dr.ex1, dr.rn1);
        const float td = fmaf(gamma, mx, rew[x]) - q0;
        const float qtd = fmaf(alpha, td, q0);
        q[e] = qtd;
        const float mx2 = next_f32(algo, q[2 * sn], q[2 * sn + 1], ef, dr.ex2, dr.rn2);
        td2 = fmaf(gamma, mx2, rew[x]) - qtd;
        q[e] = qtd + nu;
      }
      const double pct =
          (double)fabsf(nu) / ((double)fabsf(alpha * td2) + (double)fabsf(nu) + 1e-8) * 100.0;

      const int wasC = (S[x] == 0);
      const double Px = payoff_from_count(p, SN[x], wasC);
      acc_st[OST_NC_OLD] += wasC;
      acc_st[OST_N_CD] += (wasC && act == 1);
      acc_st[OST_N_DC] += (!wasC && act == 0);
      acc_st[OST_NC_NEW] += (act == 0);
      acc_st[OST_SUM_P] += Px;
      acc_st[wasC ? OST_SUM_P_C : OST_SUM_P_D] += Px;
      acc_st[OST_SUM_WP_P] += wP * Px;
      const double rewd = wP * Px + wR * (act == 0 ? 0.5 : 0.0);
      acc_st[act == 0 ? OST_SUM_REW_C : OST_SUM_REW_D] += rewd;
      if (act == 0) acc_st[OST_SUM_RATIO] += fabs(wR * 0.5) / (fabs(rewd) + 1e-9) * 100.0;
      acc_st[OST_SUM_R] += R[x];
      for (int z = 0; z < 4; ++z) {
        acc_st[OST_SUM_Q + z] += qs[z];
        acc_st[(wasC ? OST_SUM_Q_C : OST_SUM_Q_D) + z] += qs[z];
      }
      acc_st[OST_SUM_NI] += pct;
      if (best > 0.0f) {
        acc_st[OST_N_BEST_POS] += 1;
        acc_st[OST_N_BEST_2ND] += (kstar >= 4);
      }
      const int nd = (a[IDX(i, j)] == 1) + (a[IDX(i + 1, j)] == 1) + (a[IDX(i - 1, j)] == 1) +
                     (a[IDX(i, j + 1)] == 1) + (a[IDX(i, j - 1)] == 1);
      acc_st[OST_GROUP0 + nd] += 1;
    }
  acc_st[OST_GMAX] = gmax;
  if (stats) memcpy(stats, acc_st, sizeof(acc_st));

  memcpy(S, a, n_sites);
  memcpy(R, Rn, n_sites * sizeof(float));
  free(N); free(SN); free(a); free(s_old); free(s_new); free(Rn); free(rew);
  return 0;
}

/* ================================================================ digests */
/* k_state_digest (csrc/spgg_kernels.cuh): site (i, j) of global row i adds to each word
 * (hash | 1) * (bits of its value as a double + 1) mod 2^64, the hash keyed by (i, j) and the
 * word (S, R, Q entry z).  The odd multiplier is invertible mod 2^64, so a change of one value
 * changes the sum. */
static inline uint64_t digest_mix(uint64_t x) {
  x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
  return x;
}

static inline uint64_t dbits(double v) {
  uint64_t u;
  memcpy(&u, &v, sizeof(u));
  return u;
}

/* multipliers of the value slot (a, b): with period 0 those of site (row0 + a, b), with period P
 * the sum over the sites (a + uP, b + vP) of the L x L lattice that carry that slot's value */
static void slot_weights(int L, int row0, int period, int nq, int a, int b, uint64_t *w) {
  const int k = period ? L / period : 1, step = period ? period : 0;
  for (int m = 0; m < 2 + nq; ++m) w[m] = 0;
  for (int u = 0; u < k; ++u)
    for (int v = 0; v < k; ++v) {
      const uint64_t key = ((uint64_t)(uint32_t)(row0 + a + u * step) << 32) | (uint32_t)(b + v * step);
      w[0] += digest_mix(key * 3 + 1) | 1u;
      w[1] += digest_mix(key * 3 + 2) | 1u;
      for (int z = 0; z < nq; ++z) w[2 + z] += digest_mix(key * 3 + 3 + ((uint64_t)(z + 1) << 58)) | 1u;
    }
}

static int digest_geometry(int L, int rows, int period, int *nr, int *nc) {
  if (period) {
    if (period < 1 || L % period != 0) return -1;
    *nr = *nc = period;
  } else {
    *nr = rows; *nc = L;
  }
  return 0;
}

int oracle_digest_weights(int L, int row0, int rows, int period, int nq, uint64_t *w) {
  int nr, nc;
  if (digest_geometry(L, rows, period, &nr, &nc)) return -1;
  const int nw = 2 + nq;
#pragma omp parallel for schedule(dynamic, 1)
  for (int a = 0; a < nr; ++a)
    for (int b = 0; b < nc; ++b) slot_weights(L, row0, period, nq, a, b, w + ((size_t)a * nc + b) * nw);
  return 0;
}

int oracle_state_digest(int L, int row0, int rows, int period, int nq, const uint8_t *S,
                        const double *R, const double *Q, const uint64_t *w, uint64_t out[3]) {
  int nr, nc;
  if (digest_geometry(L, rows, period, &nr, &nc)) return -1;
  const int nw = 2 + nq;
  uint64_t dS = 0, dR = 0, dQ = 0;
#pragma omp parallel for schedule(dynamic, 1) reduction(+ : dS, dR, dQ)
  for (int a = 0; a < nr; ++a)
    for (int b = 0; b < nc; ++b) {
      const size_t x = (size_t)a * nc + b;
      uint64_t ws[2 + 8];
      const uint64_t *wx = ws;
      if (w) wx = w + x * nw;
      else slot_weights(L, row0, period, nq, a, b, ws);
      dS += wx[0] * (uint64_t)((S[x] != 0) + 1);
      dR += wx[1] * (dbits(R[x]) + 1);
      if (Q)
        for (int z = 0; z < nq; ++z) dQ += wx[2 + z] * (dbits(Q[x * nq + z]) + 1);
    }
  out[0] = dS; out[1] = dR; out[2] = Q ? dQ : 0;
  return 0;
}

/* ============================================================ k_init_random */
/* Q entry z of table t of site (i, j): Philox counter (j, row0 + i, t, 1), word z; the device
 * evaluates -0.01 + 0.02 * u as one fused multiply-add in double, then rounds to the Q type */
static inline double init_q(uint32_t word, int fp32) {
  const double uu = (double)(word >> 8) * (1.0 / 16777216.0);
  const double q = fma(0.02, uu, -0.01);
  return fp32 ? (double)(float)q : q;
}

/* strategy word wi of global row gi: counter (wi >> 2, gi, 0, 2), word wi & 3, masked beyond L */
static inline uint32_t init_s_word(uint64_t seed, int L, int gi, int wi) {
  const uint32_t ctr[4] = {(uint32_t)(wi >> 2), (uint32_t)gi, 0u, 2u};
  const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
  uint32_t w[4];
  oracle_philox4x32_10(ctr, key, w);
  uint32_t word = w[wi & 3];
  const int rem = L - wi * 32;
  if (rem < 32) word &= (1u << rem) - 1u;
  return word;
}

static inline void init_q_site(uint64_t seed, int gi, int j, int nq, int fp32, double *q) {
  const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
  for (int t = 0; t < nq / 4; ++t) {
    const uint32_t ctr[4] = {(uint32_t)j, (uint32_t)gi, (uint32_t)t, 1u};
    uint32_t w[4];
    oracle_philox4x32_10(ctr, key, w);
    for (int z = 0; z < 4; ++z) q[4 * t + z] = init_q(w[z], fp32);
  }
}

void oracle_init_random(int L, int row0, int rows, int nq, int fp32, uint64_t seed, uint8_t *S, double *R,
                        double *Q) {
  const int nW = (L + 31) >> 5;
#pragma omp parallel for schedule(static)
  for (int i = 0; i < rows; ++i) {
    for (int wi = 0; wi < nW; ++wi) {
      const uint32_t word = init_s_word(seed, L, row0 + i, wi);
      for (int c = wi * 32; c < L && c < wi * 32 + 32; ++c) S[(size_t)i * L + c] = (uint8_t)((word >> (c & 31)) & 1u);
    }
    for (int j = 0; j < L; ++j) {
      const size_t x = (size_t)i * L + j;
      R[x] = 0.0;
      init_q_site(seed, row0 + i, j, nq, fp32, Q + x * nq);
    }
  }
}

int oracle_init_random_digest(int L, int row0, int rows, int nq, int fp32, uint64_t seed, uint64_t out[3]) {
  if (nq != 4 && nq != 8) return -1;
  const int nW = (L + 31) >> 5;
  uint64_t dS = 0, dR = 0, dQ = 0;
#pragma omp parallel for schedule(dynamic, 1) reduction(+ : dS, dR, dQ)
  for (int i = 0; i < rows; ++i)
    for (int wi = 0; wi < nW; ++wi) {
      const uint32_t word = init_s_word(seed, L, row0 + i, wi);
      for (int j = wi * 32; j < L && j < wi * 32 + 32; ++j) {
        uint64_t ws[2 + 8];
        double q[8];
        slot_weights(L, row0, 0, nq, i, j, ws);
        init_q_site(seed, row0 + i, j, nq, fp32, q);
        dS += ws[0] * (uint64_t)(((word >> (j & 31)) & 1u) + 1);
        dR += ws[1] * (dbits(0.0) + 1);
        for (int z = 0; z < nq; ++z) dQ += ws[2 + z] * (dbits(q[z]) + 1);
      }
    }
  out[0] = dS; out[1] = dR; out[2] = dQ;
  return 0;
}

/* ======================================================== epsilon = 1 actions */
void oracle_explore_actions(int L, int i0, int i1, uint64_t seed, uint32_t step, uint8_t *a) {
  const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
#pragma omp parallel for schedule(static)
  for (int i = i0; i < i1; ++i)
    for (int j4 = 0; j4 < L; j4 += 4) {
      const uint32_t ctr[4] = {(uint32_t)(j4 >> 2), (uint32_t)i, step, 0u};
      uint32_t w[4];
      oracle_philox4x32_10(ctr, key, w);
      for (int z = 0; z < 4 && j4 + z < L; ++z) a[(size_t)(i - i0) * L + j4 + z] = (uint8_t)(w[z] & 1u);
    }
}
