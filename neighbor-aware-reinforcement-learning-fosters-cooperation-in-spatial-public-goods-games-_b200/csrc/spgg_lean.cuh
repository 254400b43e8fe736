// Kernels of the general path, for the lattices the TMA fast path does not take - reference precision (fp64 Q
// and R, spgg.py:121,129), fp32 reputations, lattice sides that are not multiples of 32:
//   k_gmax_lean  the global maximum of every iteration, whatever the TD rule;
//   k_step_lean  the Q-learning iteration of k_step (spgg_kernels.cuh) with the same thread <-> site mapping, the
//                same arithmetic in the same order and therefore the same results bit for bit, statistics included
//                (tests/test_gpu_lean.py compares the two with SPGG_NO_LEAN=1).  The site code both kernels share
//                (constants, lambda denominator, Philox words, arg-max neighbour, fp32 update) is written once in spgg_kernels.cuh.
//
// k_step carries every TD rule, the replay of up to three draw streams and the select-only / update-only
// launches behind runtime switches; ncu counted 570 instructions per site for its select-only launch alone
// (profiles/r02_fp64_lean.md).  What k_step_lean does differently:
//   * Q-learning and "update" are compile-time facts (the host launches it for algo 0, do_update = 1);
//   * the reward of an fp64 code is a table lookup (KArgs::valtab, built once per handle by k_build_valtab
//     with payoff_f64 / reward_f64 themselves) instead of an fp64 division per staged site;
//   * tiles are staged with every global load of a thread in flight at once (stage_tile in spgg_kernels.cuh,
//     shared with k_step): no division per element, the code -> reward pass fused into the code load, ghost
//     columns read instead of wrapped;
//   * the Q entries of a pair of the four sites a thread owns in a row (and their replayed draws) are loaded
//     before the first of them is processed, and the Q rows of the CTA's next tile are prefetched into L2;
//   * interior tiles store with plain stores (no ghost-copy tests per cell);
//   * no fp64 division ever sees an exactly-zero numerator (ddiv_zero_safe, rep_state): __ddiv_rn's slow path,
//     84 instructions per call, was taken by two divisions of nearly every site.
#pragma once
#include "spgg_dispatch.h"
#include "spgg_kernels.cuh"

namespace spgg {

// {reward, ratio statistic} of every fp64 reward code (index code >> 1), reference operation order
// (spgg.py:256-257,373-377,424-427; the ratio of spgg.py:430 for cooperating codes)
__global__ void k_build_valtab(const RepConst *rc_all, double *tab) {
  const int rep = blockIdx.y;
  const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (1u << VALTAB_BITS)) return;
  const RepConst &rc = rc_all[rep];
  const uint32_t code = idx << 1;
  double v = 0.0, ratio = 0.0;
  bool ok = true;
#pragma unroll
  for (int q = 0; q < 5; ++q) ok = ok && (((code >> (15 - 3 * q)) & 7u) <= 5u);
  if (ok) {
    v = reward_f64(code, payoff_f64(code, rc), rc);
    if ((code >> 1) & 1u)
      ratio = __dmul_rn(__ddiv_rn(fabs(__dmul_rn(rc.wR, 0.5)), __dadd_rn(fabs(v), 1e-9)), 100.0);
  }
  double *dst = tab + (((size_t)rep << VALTAB_BITS) + idx) * 2;
  dst[0] = v;
  dst[1] = ratio;
}

template <bool B>
struct BoolC { static constexpr bool value = B; };

// Lattice-global max |reward difference| over neighbour pairs (spgg.py:486-488): tiles staged row by row with
// the rewards looked up while they land, and every unordered pair taken once (|x - y| == |y - x| exactly): from
// each site towards (i+1,j), (i,j+1) and, second order, (i+2,j), (i,j+2), (i+1,j+1), (i+1,j-1).  The maximum of
// a set does not depend on the order.  One atomic per CTA (non-negative IEEE values order like unsigned ints).
template <class Md, int M>
__global__ void __launch_bounds__(MAX_THREADS) k_gmax_lean(GArgs a) {
  typedef typename Md::Code Code;
  typedef typename Md::Val Val;
  const Geom &g = a.g;
  const int rep = blockIdx.x / g.ctas_per_rep, cta = blockIdx.x % g.ctas_per_rep;
  pdl_launch_dependents();
  pdl_wait();
  const int stop = a.stop_at[rep];
  if (stop >= 0 && a.j > stop) return;

  extern __shared__ __align__(16) unsigned char smem[];
  Val *sm_val = reinterpret_cast<Val *>(smem);
  float *sm_tab = reinterpret_cast<float *>(smem + align_up(sizeof(Val) * (g.TR + 2 * HR) * SMW, 16));
  __shared__ RepConst s_rc;
  load_rep_const<Md::kFp64 ? 0 : 1>(s_rc, a.rc + rep, sm_tab);

  const Code *code_in = reinterpret_cast<const Code *>(a.code_in) + (long long)rep * g.plane_stride;
  const double *vtab = a.valtab ? a.valtab + ((size_t)rep << (VALTAB_BITS + 1)) : nullptr;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  Val lmax = Val(0);
  // one of each +/- pair of c_off: neighbour (i-dx, j-dy)
  constexpr int NP = (M == 2) ? 6 : 2;
  constexpr int kPair[6] = {1, 3, 5, 7, 11, 10};

  const int n_tiles = g.n_tx * g.n_ty;
  for (int tile = cta; tile < n_tiles; tile += g.ctas_per_rep) {
    const int ty = tile / g.n_tx, tx = tile - ty * g.n_tx;
    const int r0 = ty * g.TR, c0 = tx * TC;
    __syncthreads();
    stage_tile<Md, M, false>(g, r0, c0, code_in, nullptr, nullptr, s_rc, sm_tab, vtab, sm_val, nullptr, nullptr, nullptr);
    __syncthreads();
    for (int rr = warp; rr < g.TR; rr += nw) {
      if (r0 + rr >= g.rows) break;
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) {
        const int cc = k4 * 32 + lane;
        if (c0 + cc >= g.L) continue;
        const int sr = rr + HR, sc = cc + HP;
        const Val vx = sm_val[sr * SMW + sc];
#pragma unroll
        for (int k = 0; k < NP; ++k) {
          const Val vk = sm_val[(sr - c_off[kPair[k]][0]) * SMW + (sc - c_off[kPair[k]][1])];
          Val d;
          if constexpr (Md::kFp64) d = fabs(__dsub_rn(vk, vx));
          else d = fabsf(__fsub_rn(vk, vx));
          lmax = d > lmax ? d : lmax;
        }
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const Val other = __shfl_down_sync(0xffffffffu, lmax, o);
    lmax = other > lmax ? other : lmax;
  }
  __shared__ Val s_wmax[MAX_THREADS / 32];
  if (lane == 0) s_wmax[warp] = lmax;
  __syncthreads();
  if (threadIdx.x == 0) {
    Val m = s_wmax[0];
    for (int w = 1; w < nw; ++w) m = s_wmax[w] > m ? s_wmax[w] : m;
    Val *dst = reinterpret_cast<Val *>(a.gmax) + (long long)rep * a.cap + a.rel;
    if constexpr (Md::kFp64)
      atomicMax(reinterpret_cast<unsigned long long *>(dst), (unsigned long long)__double_as_longlong(m));
    else
      atomicMax(reinterpret_cast<unsigned int *>(dst), __float_as_uint(m));
  }
}

// sites of a row whose Q (and draws) k_step_lean loads before it processes the first of them
// (measured at L=4096 in fp64: batches of 4 sites 648 us per iteration, pairs 630)
constexpr int LEAN_BATCH = 2;

// 2 CTAs per SM: with 3 (80 registers, 336 B of spills) the fp64 iteration at L=4096 took 835 us instead of 611
// (profiles/r02_fp64_lean.md)
template <class Md, int M, bool ACTION, bool REPLAY>
__global__ void __launch_bounds__(MAX_THREADS, 2) k_step_lean(KArgs a) {
  typedef typename Md::Q QT;
  typedef typename Md::R RT;
  typedef typename Md::Code Code;
  typedef typename Md::Val Val;
  constexpr bool kI8 = (sizeof(RT) == 1);
  const Geom &g = a.g;
  const int rep = blockIdx.x / g.ctas_per_rep, cta = blockIdx.x % g.ctas_per_rep;
  pdl_launch_dependents();
  pdl_wait();
  const int stop = a.stop_at[rep];
  if (stop >= 0 && a.j > stop) return;
  constexpr bool upd = true;
  const bool sel = (a.do_select != 0) && !(stop >= 0 && a.j == stop);

  extern __shared__ __align__(16) unsigned char smem[];
  // the layout of the largest tile (16 rows) whatever g.TR is: the offsets are immediates instead of values
  // the compiler recomputes inside the loop (spgg_create sizes the dynamic shared memory accordingly)
  constexpr SmemLayout<Md> lay(LEAN_TR_MAX);
  Val *sm_val = reinterpret_cast<Val *>(smem + lay.off_val);
  RT *sm_R = reinterpret_cast<RT *>(smem + lay.off_R);
  Code *sm_code = reinterpret_cast<Code *>(smem + lay.off_code);
  uint8_t *sm_C = smem + lay.off_C;
  uint8_t *sm_N = smem + lay.off_N;
  float *sm_tab = reinterpret_cast<float *>(smem + lay.off_tab);
  float *sm_ratio = sm_tab + 128;
  double *sm_red = reinterpret_cast<double *>(smem + lay.off_red);
  __shared__ RepConst s_rc;
  __shared__ int s_is_last;

  load_rep_const<2>(s_rc, a.rc + rep, sm_tab);
  const RepConst &rc = s_rc;
  const double *vtab = a.valtab ? a.valtab + ((size_t)rep << (VALTAB_BITS + 1)) : nullptr;

  QT *Qp = reinterpret_cast<QT *>(a.Q) + (long long)rep * g.site_stride * 4;
  const RT *R_in = reinterpret_cast<const RT *>(a.R_in) + (long long)rep * g.plane_stride;
  RT *R_out = reinterpret_cast<RT *>(a.R_out) + (long long)rep * g.plane_stride;
  const Code *code_in = reinterpret_cast<const Code *>(a.code_in) + (long long)rep * g.plane_stride;
  Code *code_out = reinterpret_cast<Code *>(a.code_out) + (long long)rep * g.plane_stride;
  const uint32_t *S_in = a.S_in + (long long)rep * g.bits_stride;
  uint32_t *S_out = a.S_out + (long long)rep * g.bits_stride;

  Val inv_den = Val(0), den = Val(1);
  lambda_den<Md>(a, rep, rc, den, inv_den);
  const long long tab_idx = (long long)(a.rel + 1) * g.n_rep + rep;
  const uint32_t thr = sel ? a.thr_tab[tab_idx] : 0u;
  const double eps = (sel && REPLAY) ? a.eps_tab[tab_idx] : 0.0;

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;

  // per-thread statistics, accumulated in k_step's order (site by site: tile, row, k4)
  // (32-bit counters: a thread sees at most a few 10^5 sites per launch, SigmaN <= 25 each)
  uint32_t cls_n[4] = {0, 0, 0, 0}, cls_sn[4] = {0, 0, 0, 0};
  uint32_t grp[6] = {0, 0, 0, 0, 0, 0};
  uint32_t n_best = 0, n_best2 = 0, n_sel_coop = 0;
  double sumQ[4] = {0, 0, 0, 0}, sumQC[4] = {0, 0, 0, 0};
  double sumNI = 0.0, sumR = 0.0, sumRatio = 0.0;

  const int n_tiles = g.n_tx * g.n_ty;
  for (int tile = cta; tile < n_tiles; tile += g.ctas_per_rep) {
    const int ty = tile / g.n_tx, tx = tile - ty * g.n_tx;
    const int r0 = ty * g.TR, c0 = tx * TC;
    const bool full = (c0 + TC <= g.L) && (r0 + g.TR <= g.rows);
    // no cell of this tile has a periodic copy (ghost column / ghost row / ghost word)
    const bool interior = full && c0 >= GC && c0 + TC <= g.L - GC &&
                          (!g.wrap_rows || (r0 >= GH && r0 + g.TR <= g.rows - GH));
    __syncthreads();
    {  // the Q rows of this CTA's next tile on their way into L2 while this tile is computed
      const int nt = tile + g.ctas_per_rep;
      if (nt < n_tiles) {
        const int nty = nt / g.n_tx, ntx = nt - nty * g.n_tx;
        const int nrow = nty * g.TR, ncol = ntx * TC;
        constexpr int kLineSites = 128 / (int)(4 * sizeof(QT));      // sites per 128-byte line
        const int lines = TC / kLineSites;
        for (int e = threadIdx.x; e < g.TR * lines; e += blockDim.x) {
          const int rr = e / lines, cs = ncol + (e - rr * lines) * kLineSites;
          if (nrow + rr < g.rows && cs < g.L)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(Qp + ((long long)(nrow + rr) * g.L + cs) * 4));
        }
      }
    }
    // ---- stage the halo'd tiles: reward codes (+ their rewards), reputations, cooperator flags
    stage_tile<Md, M, true>(g, r0, c0, code_in, R_in, S_in, rc, sm_tab, vtab, sm_val, sm_code, sm_R, sm_C);
    __syncthreads();
    {
      // N = cooperators in the 5-site group centred on each site (spgg.py:23-36) of S_j, tile + one-site ring
      const int nr = g.TR + 2;
      for (int r = warp; r < nr; r += nw) {
        const int base = (r - 1 + HR) * SMW + HP;
#pragma unroll
        for (int q = 0; q < (TC + 2 + 31) / 32; ++q) {
          const int cc = q * 32 + lane - 1;
          if (cc < TC + 1) {
            const int idx = base + cc;
            sm_N[idx] = (uint8_t)(sm_C[idx] + sm_C[idx + SMW] + sm_C[idx - SMW] + sm_C[idx + 1] + sm_C[idx - 1]);
          }
        }
      }
    }
    __syncthreads();

    unsigned pk_n = 0;
    unsigned long long pk_sn = 0, pk_grp = 0;
    float tq[4] = {0.f, 0.f, 0.f, 0.f}, tqc[4] = {0.f, 0.f, 0.f, 0.f};
    float tni = 0.f, tratio = 0.f, trf = 0.f;
    int tri = 0;

    auto do_row = [&](auto fullc, auto interiorc, int rr) {
      constexpr bool FULL = decltype(fullc)::value;
      constexpr bool INTERIOR = decltype(interiorc)::value;
      const int i = r0 + rr;
      const int sr = rr + HR;
      uint32_t w4[4] = {0, 0, 0, 0};
      if (sel && !REPLAY) philox_row(c0, g.row0 + i, (uint32_t)(a.j + 1), 0u, rc, lane, w4);
      // ---- everything that comes from global memory for a batch of LEAN_BATCH sites, before the first is processed
#pragma unroll
      for (int kb = 0; kb < 4; kb += LEAN_BATCH) {
      QT q[4][4];
      [[maybe_unused]] double ru[4] = {0, 0, 0, 0};    // replayed draws
      [[maybe_unused]] uint8_t rb[4] = {0, 0, 0, 0};
      [[maybe_unused]] double rat[4] = {0, 0, 0, 0};   // fp64: ratio statistic of the site's code (second table column)
      const long long site_row = (long long)i * g.L + c0 + lane;
#pragma unroll
      for (int k4 = kb; k4 < kb + LEAN_BATCH; ++k4) {
        const bool valid = FULL || (c0 + 32 * k4 + lane < g.L);
        const long long site = site_row + 32 * k4;
        if (valid) {
          if constexpr (Md::kFp64) {
            const double2 lo2 = reinterpret_cast<const double2 *>(Qp)[site * 2];
            const double2 hi2 = reinterpret_cast<const double2 *>(Qp)[site * 2 + 1];
            q[k4][0] = lo2.x; q[k4][1] = lo2.y; q[k4][2] = hi2.x; q[k4][3] = hi2.y;
          } else {
            const float4 v = reinterpret_cast<const float4 *>(Qp)[site];
            q[k4][0] = v.x; q[k4][1] = v.y; q[k4][2] = v.z; q[k4][3] = v.w;
          }
          if constexpr (REPLAY) {
            if (sel) { ru[k4] = a.u[site]; rb[k4] = a.b[site]; }
          }
          if constexpr (Md::kFp64)
            rat[k4] = __ldg(vtab + 2 * (size_t)(sm_code[sr * SMW + 32 * k4 + lane + HP] >> 1) + 1);   // 0 for defecting codes
        } else {
          q[k4][0] = q[k4][1] = q[k4][2] = q[k4][3] = QT(0);
        }
      }
#pragma unroll
      for (int k4 = kb; k4 < kb + LEAN_BATCH; ++k4) {
        const int cc = k4 * 32 + lane;
        const int col = c0 + cc;
        const bool valid = FULL || (col < g.L);
        const int sc = cc + HP;
        const int sidx = sr * SMW + sc;
        int a_new = 0;
        if (valid) {
          const long long site = site_row + 32 * k4;
          QT q0_ = q[k4][0], q1_ = q[k4][1], q2_ = q[k4][2], q3_ = q[k4][3];
          const RT r_old = sm_R[sidx];
          const int Ccur = sm_C[sidx];
          // post-action state of iteration j == pre-action state of iteration j+1 (spgg.py:409/423)
          const int s_new = ACTION ? Ccur : rep_state<RT, M>(sm_R, sr, sc);
          if constexpr (kI8) tri += (int)r_old;
          else if constexpr (sizeof(RT) == 4) trf += r_old;
          else sumR += r_old;

          const Code code = sm_code[sidx];
          const int s = code & 1u, coop = (code >> 1) & 1u, wasC = (code >> 2) & 1u;
          const int act = coop ^ 1;
          const Val vx = sm_val[sidx];
          // neighbour-aware term inputs: spgg.py:486-494 (first arg-max wins)
          const auto bn = best_neighbour<Md, M>(sm_val, sr, sc, vx);
          const Val best = bn.d;
          const int bidx = bn.idx, kstar = bn.k;
          const bool same = (((sm_code[bidx] >> 1) & 1u) == (unsigned)coop);
          const int e = 2 * s + act;
          const QT qe = sel4<QT>(e, q0_, q1_, q2_, q3_);
          const QT na = s_new ? q2_ : q0_, nb = s_new ? q3_ : q1_;  // pre-update row of s'
          QT qfin;
          if constexpr (Md::kFp64) {
            const double mx = fmax(na, nb);                                              // algorithms.py:125
            const double td = __dsub_rn(__dadd_rn(vx, __dmul_rn(rc.gamma, mx)), qe);     // algorithms.py:128
            const double qtd = __dadd_rn(qe, __dmul_rn(rc.alpha, td));                   // algorithms.py:131
            const double num = __dmul_rn(rc.kappa, fmax(0.0, best));
            const double na2 = (s_new == s && act == 0) ? qtd : na;
            const double nb2 = (s_new == s && act == 1) ? qtd : nb;
            const double td2 = __dsub_rn(__dadd_rn(vx, __dmul_rn(rc.gamma, fmax(na2, nb2))), qtd);
            // A site without a better neighbour has an exactly-zero numerator: lambda is that zero and the NI
            // statistic adds +0.  Both divisions of the other sites sit in ONE block the optimiser cannot
            // speculate (the empty volatile asm): a division it evaluates for every lane sends the zero
            // numerators through __ddiv_rn's slow path, 84 instructions per call (profiles/r02_fp64_lean.md);
            // once domains have formed whole warps skip the block.
            double lam = num;                                                            // spgg.py:489
            if (!(num == 0.0 && den > 0.0)) {
              asm volatile("");
              lam = __ddiv_rn(num, den);
              const double an = fabs(lam);
              sumNI += __dmul_rn(ddiv_zero_safe(an, __dadd_rn(__dadd_rn(fabs(__dmul_rn(rc.alpha, td2)), an), 1e-8)), 100.0);  // spgg.py:512
            }
            const double nu = same ? lam : -lam;                                         // spgg.py:494-495
            qfin = __dadd_rn(qtd, nu);                                                   // spgg.py:509
            pk_sn += (unsigned long long)sigma_n_of_code(code) << (16 * (wasC * 2 + coop));
            if (coop) sumRatio += rat[k4];
          } else {
            auto next_value = [](float x0, float x1, bool) { return fmaxf(x0, x1); };
            qfin = td_update_f32(rc, vx, qe, na, nb, s, s_new, act, best, same, inv_den, next_value, tni);
            pk_sn += (unsigned long long)(code >> 3) << (16 * (wasC * 2 + coop));
            if (rc.has_ratio && coop) tratio += sm_ratio[code >> 1];
          }
          q0_ = (e == 0) ? qfin : q0_;
          q1_ = (e == 1) ? qfin : q1_;
          q2_ = (e == 2) ? qfin : q2_;
          q3_ = (e == 3) ? qfin : q3_;
          pk_n += 1u << (8 * (wasC * 2 + coop));
          if (best > Val(0)) { n_best += 1u; n_best2 += (kstar >= 4); }
          pk_grp += 1ull << (10 * (5 - (int)sm_N[sidx]));                                // spgg.py:586-592
          if constexpr (Md::kFp64) {
            sumQ[0] += q0_; sumQ[1] += q1_; sumQ[2] += q2_; sumQ[3] += q3_;
            if (wasC) { sumQC[0] += q0_; sumQC[1] += q1_; sumQC[2] += q2_; sumQC[3] += q3_; }
          } else {
            const float m = wasC ? 1.0f : 0.0f;
            tq[0] += q0_; tq[1] += q1_; tq[2] += q2_; tq[3] += q3_;
            tqc[0] = fmaf(m, q0_, tqc[0]); tqc[1] = fmaf(m, q1_, tqc[1]);
            tqc[2] = fmaf(m, q2_, tqc[2]); tqc[3] = fmaf(m, q3_, tqc[3]);
          }

          if (sel) {
            int explore, rnd;
            if constexpr (REPLAY) {
              explore = ru[k4] < eps;  // algorithms.py:105
              rnd = rb[k4];            // algorithms.py:108
            } else {
              explore = (w4[k4] >> 8) < thr;
              rnd = (int)(w4[k4] & 1u);
            }
            const QT ga = s_new ? q2_ : q0_, gb = s_new ? q3_ : q1_;
            const int greedy = (gb > ga) ? 1 : 0;  // np.argmax, tie -> 0   algorithms.py:107
            a_new = explore ? rnd : greedy;        // algorithms.py:109
            n_sel_coop += (a_new == 0);
            RT r_new;                              // spgg.py:321-323
            if constexpr (kI8) {
              int t = (int)r_old + (a_new == 0 ? rc.gain_i : -rc.loss_i);
              t = max(t, rc.rmin_i);
              t = min(t, rc.rmax_i);
              r_new = (RT)t;
            } else if constexpr (sizeof(RT) == 4) {
              const float t = __fadd_rn(r_old, a_new == 0 ? rc.gainC_f : -rc.lossD_f);
              r_new = fminf(fmaxf(t, rc.rmin_f), rc.rmax_f);
            } else {
              const double t = __dadd_rn(r_old, a_new == 0 ? rc.gainC : -rc.lossD);
              r_new = fmin(fmax(t, rc.rmin), rc.rmax);
            }
            const int n5[5] = {sm_N[sidx], sm_N[sidx - SMW], sm_N[sidx + SMW], sm_N[sidx - 1], sm_N[sidx + 1]};
            const Code cnew = pack_code<Md>(n5, Ccur, a_new ^ 1, s_new);
            if constexpr (INTERIOR) {
              const long long o = (long long)(i + GH) * g.pitchB + CPAD + col;
              code_out[o] = cnew;
              R_out[o] = r_new;
            } else {
              store_cell<Code>(code_out, g, i, col, cnew);
              store_cell<RT>(R_out, g, i, col, r_new);
            }
          }
          if constexpr (Md::kFp64) {
            reinterpret_cast<double2 *>(Qp)[site * 2] = make_double2(q0_, q1_);
            reinterpret_cast<double2 *>(Qp)[site * 2 + 1] = make_double2(q2_, q3_);
          } else {
            reinterpret_cast<float4 *>(Qp)[site] = make_float4(q0_, q1_, q2_, q3_);
          }
        }
        if (sel) {
          const uint32_t word = __ballot_sync(0xffffffffu, valid && a_new);
          const int wi = (c0 >> 5) + k4;
          if (lane == 0) {
            if constexpr (INTERIOR) S_out[(long long)(i + GH) * g.pitchW + WPAD + wi] = word;
            else if (wi * 32 < g.L) store_bits_word(S_out, g, i, wi, word);
          }
        }
      }
      }   // batch
    };

    if (interior) {
      for (int rr = warp; rr < g.TR; rr += nw) do_row(BoolC<true>{}, BoolC<true>{}, rr);
    } else {
      for (int rr = warp; rr < g.TR; rr += nw) {
        if (r0 + rr >= g.rows) break;
        do_row(BoolC<false>{}, BoolC<false>{}, rr);
      }
    }
    // flush the per-tile packed counters
#pragma unroll
    for (int z = 0; z < 4; ++z) {
      cls_n[z] += (pk_n >> (8 * z)) & 0xffu;
      cls_sn[z] += (uint32_t)((pk_sn >> (16 * z)) & 0xffffull);
      sumQ[z] += (double)tq[z];
      sumQC[z] += (double)tqc[z];
    }
#pragma unroll
    for (int z = 0; z < 6; ++z) grp[z] += (uint32_t)((pk_grp >> (10 * z)) & 0x3ffull);
    sumNI += (double)tni;
    sumRatio += (double)tratio;
    sumR += (double)tri + (double)trf;
  }

  StepSums sums;
#pragma unroll
  for (int z = 0; z < 4; ++z) { sums.cls_n[z] = cls_n[z]; sums.cls_sn[z] = cls_sn[z]; sums.sumQ[z] = sumQ[z]; sums.sumQC[z] = sumQC[z]; }
#pragma unroll
  for (int z = 0; z < 6; ++z) sums.grp[z] = grp[z];
  sums.n_best = n_best; sums.n_best2 = n_best2; sums.n_sel_coop = n_sel_coop;
  sums.sumNI = sumNI; sums.sumR = sumR; sums.sumRatio = sumRatio;
  step_epilogue<Md>(a, rep, cta, rc, sums, sm_red, &s_is_last, upd, sel);
}

}  // namespace spgg
