// SPGG lattice step for sm_100a - kernels.
//
// One iteration t of the reference loop (src/model/spgg.py:368-592, Q-learning
// rule src/model/algorithms.py:96-133) is split along its data dependencies
// (DESIGN.md "step decomposition"):
//
//   k_gmax*<t>  light: reads the per-site reward codes of iteration t, produces the
//               lattice-global max |reward difference|           (spgg.py:486-488)
//   k_step<t>   heavy, fused: finishes iteration t (TD update algorithms.py:122-131,
//               neighbour-aware update spgg.py:478-509, statistics spgg.py:512-592)
//               while Q is in registers, then - because the post-action state of
//               iteration t is the pre-action state of t+1 (spgg.py:423 vs 409) -
//               chooses the action of iteration t+1 (algorithms.py:102-110), updates
//               the reputation (spgg.py:319-323) and emits the reward code of t+1.
//
// Q is read once and written once per iteration; R, the strategy bits and the
// one-byte reward code are the only other per-site traffic.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace spgg {

constexpr int GH = 2;            // ghost rows on each side of every lattice plane
constexpr int CPAD = 16;         // ghost columns (elements) on each side of the code / R planes
constexpr int WPAD = 4;          // ghost words on each side of a strategy bit row
constexpr int GC = 2;            // ghost columns actually kept current (>= max halo)
constexpr int TC = 128;          // tile columns: one warp covers a 128-site row segment
constexpr int HP = 4;            // smem column pad on each side (>= widest halo)
constexpr int SMW = TC + 2 * HP; // smem row stride (elements)
constexpr int HR = 2;            // smem row halo (rows) on each side
constexpr int NSTAT = 40;
constexpr int MAX_THREADS = 256;

// stat-row columns (mirror of include/spgg.h)
enum {
  ST_NC_OLD = 0, ST_N_CD = 1, ST_N_DC = 2, ST_NC_NEW = 3, ST_SUM_P = 4, ST_SUM_P_C = 5,
  ST_SUM_P_D = 6, ST_SUM_WP_P = 7, ST_SUM_REW_C = 8, ST_SUM_REW_D = 9, ST_SUM_RATIO = 10,
  ST_GROUP0 = 11, ST_SUM_R = 17, ST_SUM_Q = 18, ST_SUM_Q_C = 22, ST_SUM_Q_D = 26,
  ST_SUM_NI = 30, ST_N_BEST_POS = 31, ST_N_BEST_2ND = 32, ST_GMAX = 33,
  // scratch columns used between the per-CTA partials and the final row (fp32 mode)
  ST_X_SN0 = 34, /* 34..37: sum of SigmaN per class (C_old*2+coop) */
  ST_X_NSEL = 38 /* #cooperating actions chosen by the select phase */
};

// neighbour offsets (dx,dy), reference order spgg.py:479-485; neighbour k of (i,j) is
// (i-dx, j-dy) because np.roll(X,(dx,dy))[i,j] == X[i-dx, j-dy].
__device__ __constant__ const int8_t c_off[12][2] = {
    {1, 0}, {-1, 0}, {0, 1}, {0, -1}, {2, 0}, {-2, 0},
    {0, 2}, {0, -2}, {1, 1}, {1, -1}, {-1, 1}, {-1, -1}};

// per-replica constants, built on the host (spgg_capi.cu: build_repconst)
struct RepConst {
  float rewtab[128];   // fp32 mode reward by (SigmaN<<2 | C_old<<1 | coop_new)
  float ratiotab[128]; // fp32 mode |wR*.5|/(|rew|+1e-9)*100 for coop codes, else 0
  uint32_t pkeys[20];  // Philox round keys: [2r] = seed_lo + r*0x9E3779B9, [2r+1] = seed_hi + r*0xBB67AE85
  double g[6];         // rc*n/5                                     spgg.py:256
  double cost, lo, span, wP, wR, rc;
  double alpha, gamma, kappa, leps;
  double gainC, lossD, rmin, rmax; // reputation step / clip, real units   spgg.py:321-323
  double rq;                       // int8 quantum: R_real = R_int8 * rq
  float alpha_f, gamma_f, kappa_f, leps_f;
  float gainC_f, lossD_f, rmin_f, rmax_f;
  int gain_i, loss_i, rmin_i, rmax_i;
  uint32_t seed_lo, seed_hi;
  int has_ratio;
  int pad_;
};

struct Geom {
  int L, rows, row0, wrap_rows;
  int pitchB;   // elements per row of the code / R planes: CPAD + roundup(L,16) + CPAD
  int pitchW;   // 32-bit words per row of the strategy bit plane: WPAD + roundup(words,4) + WPAD
  int n_tx, n_ty, TR;
  int ctas_per_rep, n_rep;
  long long plane_stride; // elements per replica, (rows+2GH)*pitchB
  long long bits_stride;  // words per replica, (rows+2GH)*pitchW
  long long site_stride;  // sites per replica, rows*L
};

#ifndef SPGG_MAX_RING
#define SPGG_MAX_RING 16
#endif
constexpr int RING_SLOTS = 4, RING_WORDS = 4;   // per slot: max bits, any D, any C, arrivals

struct KArgs {
  Geom g;
  const RepConst *rc;
  void *Q;
  const void *R_in;
  void *R_out;
  const void *code_in;
  void *code_out;
  const uint32_t *S_in;
  uint32_t *S_out;
  const void *gmax;        // Val[n_rep][cap]
  // fp64 mode: {reward, reward-ratio statistic} of every reward code, [n_rep][1 << 17][2], indexed by code >> 1
  // (k_build_valtab: the same operations in the same order as payoff_f64 / reward_f64, so a lookup is the
  // bit-identical value without the fp64 division per staged site); nullptr: compute
  const double *valtab;
  double *stats;           // [n_rep][cap][NSTAT]
  double *partials;        // [n_rep][ctas_per_rep][NSTAT]
  unsigned *tickets;       // [n_rep]
  int *stop_at;            // [n_rep], -1 = running
  const double *eps_tab;   // [cap+1][n_rep]: eps used at iteration (start + idx)
  const uint32_t *thr_tab; // same shape, ceil(eps*2^24)
  const double *u;         // replay draws of iteration j+1 (or nullptr)
  const uint8_t *b;
  // TD rule (general kernel only): 0 Q-learning, 1 SARSA, 2 Expected SARSA (algorithms.py:96-234)
  int algo;
  const double *u2, *u3;   // SARSA: replayed draws of iteration j for the update's next action
  const uint8_t *b2, *b3;  //        (spgg.py:433) and for the NI statistic's (spgg.py:452); or nullptr
  int j;                   // absolute iteration index this launch finishes (state index)
  int rel;                 // j - (iteration at start of the spgg_step call)
  int cap;                 // rows per replica in stats/gmax tables
  int do_update, do_select;
  // Speculative global maximum (fast path, spgg_fast.cuh).  The lattice-global max |reward difference| of
  // iteration j (spgg.py:488) is also max over sites of the best signed neighbour difference the update
  // computes anyway, so every update launch produces it as a by-product (atomicMax into gmax[rep][rel]).
  // With spec != 0 the launch does not wait for a k_gmax pass: it uses the previous iteration's value
  // (gcarry[rep]) and the last CTA compares; on a mismatch it records rel in *bad_at, every later launch of
  // the chunk returns at once, and the host re-runs from there with the (now known) exact value.
  int spec;                // 0 exact (gmax[rep][rel] was computed by k_gmax_*), 1 guess = gcarry[rep], 2 test hook: a wrong guess
  float *gcarry;           // [n_rep] exact maximum of the last finished iteration (written by every update launch)
  int *bad_at;             // handle-wide: INT_MAX, or the first rel whose speculation failed
  // Row strips (one lattice over several GPUs): the maximum and the uniform-lattice test of spgg.py:405 are
  // lattice-global, so a strip only REPORTS - gvec[rel] = {its own maximum, 1 if it holds a defecting action,
  // 1 if it holds a cooperating action, 0} - and k_strip_verify, run after the ranks have max-reduced that
  // vector, does what the last CTA does for a whole lattice (compare with the guess, gcarry, stop flag)
  float *gvec;             // [cap][4] or nullptr (whole lattice)
  // Strips with peer-mapped planes (cudaIpc, NVLink): the boundary tiles store their first / last GH rows
  // straight into the ghost rows of the strip above ([0]) / below ([1]) - the OUTPUT planes of this launch
  // on that GPU - so no halo message is packed, sent and unpacked between two launches.  nullptr: no peer.
  void *peer_code[2];
  void *peer_R[2];
  uint32_t *peer_S[2];
  int peer_rows[2];        // rows the neighbour owns (its bottom ghost rows start at that row index)
  // ... and a 4-slot ring of {max bits, any D, any C, arrivals} per strip, mapped by every rank: the last CTA
  // of a launch max-combines its report into slot (gen & 3) of EVERY rank and then counts itself in; the
  // one-thread kernel k_ring_verify of each rank waits until all ranks are in and takes the verdict.  No
  // collective library call between two launches.  ring_world == 0: no ring (NCCL all-reduce of gvec).
  unsigned *ring_peer[SPGG_MAX_RING];
  int ring_world, gen;
#ifdef SPGG_TRACE
  unsigned long long *trace;  // debug builds only: per CTA {start ns, end ns, smid, tiles}
#endif
};

// programmatic dependent launch: let the next kernel of the stream be scheduled while this one
// drains, and wait (in the next kernel) until everything before it has completed and is visible
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ------------------------------------------------------------------ Philox4x32-10
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                              uint32_t k0, uint32_t k1, uint32_t (&out)[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// the same generator with the ten round keys read from a table (shared memory: the key
// schedule then costs five 16-byte loads instead of 18 integer adds per call)
__device__ __forceinline__ void philox4x32_10_keys(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                   const uint32_t *keys, uint32_t (&out)[4]) {
  uint32_t k[20];
#pragma unroll
  for (int q = 0; q < 5; ++q) {
    const uint4 v = reinterpret_cast<const uint4 *>(keys)[q];
    k[4 * q] = v.x; k[4 * q + 1] = v.y; k[4 * q + 2] = v.z; k[4 * q + 3] = v.w;
  }
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k[2 * r];
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k[2 * r + 1];
    c3 = lo0;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// ------------------------------------------------------------------ modes
// Reward code of a site for iteration t (one per site, written by k_step<t-1>):
//   bit0 = s_t   (state in which a_t was chosen)            spgg.py:409
//   bit1 = coop_t (a_t == 0)                                algorithms.py:109
//   bit2 = C_{t-1} (S_{t-1} == 0, the strategy the payoff P refers to)  spgg.py:373
//   fp32 mode: bits 3..7 = SigmaN = sum over the site's 5 groups of #cooperators (0..25)
//   fp64 mode: bits 3..17 = N of the 5 groups in the reference's summation order
//              (centres (i,j),(i-1,j),(i+1,j),(i,j-1),(i,j+1); spgg.py:373-377), 3 bits each
struct ModeF32I8 {
  typedef float Q; typedef int8_t R; typedef uint8_t Code; typedef float Val;
  static constexpr bool kFp64 = false;
};
struct ModeF32F {
  typedef float Q; typedef float R; typedef uint8_t Code; typedef float Val;
  static constexpr bool kFp64 = false;
};
struct ModeF64 {
  typedef double Q; typedef double R; typedef uint32_t Code; typedef double Val;
  static constexpr bool kFp64 = true;
};

template <class Md>
__device__ __forceinline__ typename Md::Code pack_code(const int (&n)[5], int C, int coop, int s) {
  if constexpr (Md::kFp64) {
    return (typename Md::Code)((n[0] << 15) | (n[1] << 12) | (n[2] << 9) | (n[3] << 6) |
                               (n[4] << 3) | (C << 2) | (coop << 1) | s);
  } else {
    return (typename Md::Code)(((n[0] + n[1] + n[2] + n[3] + n[4]) << 3) | (C << 2) |
                               (coop << 1) | s);
  }
}

// normalised payoff P of a site from its code, fp64, reference operation order
// (spgg.py:256-257 per group, summed left to right spgg.py:373-377, normalised :377)
__device__ __forceinline__ double payoff_f64(uint32_t code, const RepConst &rc) {
  const double C = (double)((code >> 2) & 1u), D = 1.0 - C;
  double tot = 0.0;
#pragma unroll
  for (int q = 0; q < 5; ++q) {
    const double share = rc.g[(code >> (15 - 3 * q)) & 7u];
    const double term =
        __dadd_rn(__dmul_rn(__dsub_rn(share, rc.cost), C), __dmul_rn(share, D));
    tot = (q == 0) ? term : __dadd_rn(tot, term);
  }
  return __ddiv_rn(__dsub_rn(tot, rc.lo), rc.span);
}
// reward spgg.py:424-427
__device__ __forceinline__ double reward_f64(uint32_t code, double P, const RepConst &rc) {
  const double rr = ((code >> 1) & 1u) ? 0.5 : 0.0;
  return __dadd_rn(__dmul_rn(rc.wP, P), __dmul_rn(rc.wR, rr));
}

constexpr int VALTAB_BITS = 17;   // code >> 1: coop, C_old and the five 3-bit group counts

// sum of the five 3-bit group counts of an fp64-mode code (bits 3..17): SigmaN of the fp32 modes
__device__ __forceinline__ uint32_t sigma_n_of_code(uint32_t code) {
  const uint32_t x = code >> 3;
  const uint32_t a = x & 070707u, b = (x >> 3) & 0707u;          // digits 0,2,4 / 1,3 spaced 6 bits apart
  return (((a * 010101u) >> 12) & 63u) + (((b * 0101u) >> 6) & 63u);
}

template <class Md>
__device__ __forceinline__ typename Md::Val val_of_code(typename Md::Code code, const RepConst &rc,
                                                        const float *sm_tab, const double *valtab = nullptr) {
  if constexpr (Md::kFp64) {
    if (valtab) return __ldg(valtab + 2 * (size_t)(code >> 1));
    return reward_f64(code, payoff_f64(code, rc), rc);
  } else {
    return sm_tab[code >> 1];
  }
}

// num / den, correctly rounded, without __ddiv_rn's slow path for an exactly-zero numerator over a positive
// denominator (the quotient is that zero, sign included): most sites have no better neighbour, so the
// neighbour-aware term's numerator kappa max(0, best) is an exact zero for them (spgg.py:489)
// (the optimiser must not see that the replaced operand is only used where z is false - it would fold the
// select away and divide the zero after all, which is what happened: hence the empty asm)
__device__ __forceinline__ double opaque(double x) {
  asm("" : "+d"(x));
  return x;
}
__device__ __forceinline__ double ddiv_zero_safe(double num, double den) {
  const bool z = (num == 0.0) && (den > 0.0);
  const double q = __ddiv_rn(opaque(z ? 1.0 : num), den);
  return z ? num : q;
}

// reputation state spgg.py:292-307: (sum over self + offsets of R)/n > 0, reference order
template <class RT, int M>
__device__ __forceinline__ int rep_state(const RT *smR, int sr, int sc) {
  constexpr int NK = (M == 2) ? 12 : 4;
  if constexpr (sizeof(RT) == 1) {
    int acc = smR[sr * SMW + sc];
#pragma unroll
    for (int k = 0; k < NK; ++k) acc += smR[(sr - c_off[k][0]) * SMW + (sc - c_off[k][1])];
    return acc > 0;
  } else if constexpr (sizeof(RT) == 4) {
    float acc = smR[sr * SMW + sc];
#pragma unroll
    for (int k = 0; k < NK; ++k)
      acc = __fadd_rn(acc, smR[(sr - c_off[k][0]) * SMW + (sc - c_off[k][1])]);
    return __fdiv_rn(acc, (float)(NK + 1)) > 0.0f;
  } else {
    double acc = smR[sr * SMW + sc];
#pragma unroll
    for (int k = 0; k < NK; ++k)
      acc = __dadd_rn(acc, smR[(sr - c_off[k][0]) * SMW + (sc - c_off[k][1])]);
    // sign of acc / n: that of acc, unless the quotient underflows (|acc| below 1e-300: divide).  The division
    // must stay inside its branch: evaluated for every lane (what the optimiser does with a pure expression) a
    // ZERO numerator - the common case while reputations are small integers - sends __ddiv_rn through its
    // slow path (84 instructions per call, profiles/r02_fp64_lean.md)
    const bool plain = fabs(acc) > 1e-300 || acc == 0.0;
    int st = acc > 0.0;
    if (!plain) {
      asm volatile("");   // not to be speculated: see above
      st = __ddiv_rn(acc, (double)(NK + 1)) > 0.0;
    }
    return st;
  }
}

__device__ __forceinline__ int wrap_col(int col, int L) {
  if (col < 0) {
    col += L;
    if (col < 0) col = ((col % L) + L) % L;
  } else if (col >= L) {
    col -= L;
    if (col >= L) col %= L;
  }
  return col;
}

// generic tile loader: plane element (prow, col) for the tile rows [r0-H, r0+TR+H) and
// columns [c0-H, c0+TC+H) into smem[(rr+HR)*SMW + cc+HP]; columns wrap, rows use ghosts.
template <class T, int H>
__device__ __forceinline__ void load_tile(T *sm, const T *plane, const Geom &g, int r0, int c0,
                                          int TR) {
  constexpr int NC = TC + 2 * H;
  const int nr = TR + 2 * H;
  for (int e = threadIdx.x; e < nr * NC; e += blockDim.x) {
    const int rr = e / NC - H, cc = e % NC - H;
    const int prow = r0 + rr + GH;
    T v = T(0);
    if (prow >= 0 && prow < g.rows + 2 * GH) {
      const int col = wrap_col(c0 + cc, g.L);
      v = plane[(long long)prow * g.pitchB + CPAD + col];
    }
    sm[(rr + HR) * SMW + cc + HP] = v;
  }
}

// strategy bits -> cooperator flags (1 = cooperator), halo 2
__device__ __forceinline__ void load_coop_tile(uint8_t *sm, const uint32_t *bits, const Geom &g,
                                               int r0, int c0, int TR) {
  constexpr int H = 2, NC = TC + 2 * H;
  const int nr = TR + 2 * H;
  for (int e = threadIdx.x; e < nr * NC; e += blockDim.x) {
    const int rr = e / NC - H, cc = e % NC - H;
    const int prow = r0 + rr + GH;
    uint8_t v = 0;
    if (prow >= 0 && prow < g.rows + 2 * GH) {
      const int col = wrap_col(c0 + cc, g.L);
      const uint32_t w = bits[(long long)prow * g.pitchW + WPAD + (col >> 5)];
      v = (uint8_t)(((w >> (col & 31)) & 1u) ^ 1u);
    }
    sm[(rr + HR) * SMW + cc + HP] = v;
  }
}

// deterministic block reduction of NV doubles held per thread; result in sm_red[0..NV).
// Warp stage: groups of 32 values go through one transposing butterfly (at each of five levels a
// lane keeps half of its values and hands the other half to its partner: 31 shuffles reduce 32
// values at once and lane z ends with the warp sum of value z); the remaining NV % 32 values take
// the classic five-step tree.
template <int NV>
__device__ __forceinline__ void block_reduce_bfly(double (&v)[NV], double *sm_red /* [8][NV] */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  constexpr int NG = NV / 32;
#pragma unroll
  for (int gI = 0; gI < NG; ++gI) {
    double w[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) w[i] = v[32 * gI + i];
#pragma unroll
    for (int lvl = 0; lvl < 5; ++lvl) {
      const int o = 16 >> lvl, half = 16 >> lvl;
      const bool hi = (lane & o) != 0;
#pragma unroll
      for (int i = 0; i < half; ++i) {
        const double keep = hi ? w[i + half] : w[i];
        const double send = hi ? w[i] : w[i + half];
        w[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
      }
    }
    sm_red[warp * NV + 32 * gI + lane] = w[0];
  }
#pragma unroll
  for (int i = 32 * NG; i < NV; ++i) {
    double x = v[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
    if (lane == 0) sm_red[warp * NV + i] = x;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double x = 0.0;
    for (int w = 0; w < nw; ++w) x += sm_red[w * NV + threadIdx.x];
    sm_red[threadIdx.x] = x;
  }
  __syncthreads();
}

// the same with one five-step tree per value: fewer live registers (the general kernel keeps its
// occupancy), five times the shuffles
template <int NV>
__device__ __forceinline__ void block_reduce(double (&v)[NV], double *sm_red /* [8][NV] */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    double x = v[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
    if (lane == 0) sm_red[warp * NV + i] = x;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double x = 0.0;
    for (int w = 0; w < nw; ++w) x += sm_red[w * NV + threadIdx.x];
    sm_red[threadIdx.x] = x;
  }
  __syncthreads();
}

// Last CTA of a replica: fold the per-CTA partial rows in a fixed order (deterministic) using
// the whole block: group q of NSTAT threads adds CTAs q, q+G, q+2G, ...; the G group sums
// are then added in order.  Result in sm_red[0..NSTAT).
__device__ __forceinline__ void fold_partials(const double *pp, int n_ctas, double *sm_red /* [8][NSTAT] */) {
  const int groups = min((int)blockDim.x / NSTAT, 8);
  const int q = threadIdx.x / NSTAT, z = threadIdx.x - q * NSTAT;
  if (q < groups) {
    double x = 0.0;
    // sixteen independent L2 loads in flight per thread: this fold is the tail of every launch
#pragma unroll 16
    for (int c = q; c < n_ctas; c += groups) x += __ldcg(pp + (long long)c * NSTAT + z);
    sm_red[q * NSTAT + z] = x;
  }
  __syncthreads();
  if (threadIdx.x < NSTAT) {
    double x = sm_red[threadIdx.x];
    for (int k = 1; k < groups; ++k) x += sm_red[k * NSTAT + threadIdx.x];
    sm_red[threadIdx.x] = x;
  }
  __syncthreads();
}

__device__ __forceinline__ size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }


// ------------------------------------------------------------------ plane stores
// A value of site (i, col) goes to its own cell plus the periodic copies other tiles read:
// ghost columns (always) and ghost rows (when this handle owns every row).
template <class T>
__device__ __forceinline__ void store_cell(T *plane, const Geom &g, int i, int col, T v) {
  int gcol = -1;
  if (col < GC) gcol = CPAD + g.L + col;
  else if (col >= g.L - GC) gcol = CPAD + col - g.L;
  long long rowoff = (long long)(i + GH) * g.pitchB;
  plane[rowoff + CPAD + col] = v;
  if (gcol >= 0) plane[rowoff + gcol] = v;
  if (g.wrap_rows) {
    if (i < GH) {
      rowoff = (long long)(i + g.rows + GH) * g.pitchB;
      plane[rowoff + CPAD + col] = v;
      if (gcol >= 0) plane[rowoff + gcol] = v;
    }
    if (i >= g.rows - GH) {
      rowoff = (long long)(i - g.rows + GH) * g.pitchB;
      plane[rowoff + CPAD + col] = v;
      if (gcol >= 0) plane[rowoff + gcol] = v;
    }
  }
}
// strategy word wi of row i (ghost words only exist when L is a multiple of 32)
__device__ __forceinline__ void store_bits_word(uint32_t *S, const Geom &g, int i, int wi, uint32_t word) {
  const int nW = (g.L + 31) >> 5;
  const bool gw = (g.L & 31) == 0;
  const int gl = (gw && wi == nW - 1) ? WPAD - 1 : -1;  // left ghost word <- last data word
  const int gr = (gw && wi == 0) ? WPAD + nW : -1;      // right ghost word <- first data word
  long long rowoff = (long long)(i + GH) * g.pitchW;
  S[rowoff + WPAD + wi] = word;
  if (gl >= 0) S[rowoff + gl] = word;
  if (gr >= 0) S[rowoff + gr] = word;
  if (g.wrap_rows) {
    if (i < GH) {
      rowoff = (long long)(i + g.rows + GH) * g.pitchW;
      S[rowoff + WPAD + wi] = word;
      if (gl >= 0) S[rowoff + gl] = word;
      if (gr >= 0) S[rowoff + gr] = word;
    }
    if (i >= g.rows - GH) {
      rowoff = (long long)(i - g.rows + GH) * g.pitchW;
      S[rowoff + WPAD + wi] = word;
      if (gl >= 0) S[rowoff + gl] = word;
      if (gr >= 0) S[rowoff + gr] = word;
    }
  }
}

// =================================================================== global maximum (k_gmax_lean, spgg_lean.cuh)
struct GArgs {
  Geom g;
  const RepConst *rc;
  const void *code_in;
  void *gmax;          // Val[n_rep][cap], zeroed at the start of the spgg_step call
  const double *valtab; // see KArgs
  const int *stop_at;
  int j, rel, cap;
};

// Stages the halo'd planes of a tile with every global load of a thread in flight at once (the general
// kernel's element loops expose one memory round trip per element: ncu, profiles/r02_fp64_lean.md).
// A warp owns the staged rows r = warp, warp + nw, warp + 2 nw of rows -2 .. TR+1:
//   phase A  raw loads: reward codes and reputations (halo M; ghost columns and ghost rows of the planes hold
//            the periodic images, store_cell keeps GC >= M of them current) and the six strategy words of a row
//   phase B  stores of codes / reputations / cooperator flags, and the reward-table lookups (fp64) of all rows
//   phase C  reward stores
// STEP = false stages the rewards only (k_gmax_lean).
template <class Md, int M, bool STEP>
__device__ __forceinline__ void stage_tile(const Geom &g, int r0, int c0, const typename Md::Code *code_in,
                                           const typename Md::R *R_in, const uint32_t *S_in, const RepConst &rc,
                                           const float *sm_tab, const double *vtab, typename Md::Val *sm_val,
                                           typename Md::Code *sm_code, typename Md::R *sm_R, uint8_t *sm_C) {
  typedef typename Md::Code Code;
  typedef typename Md::R RT;
  typedef typename Md::Val Val;
  constexpr int NQ = (TC + 4 + 31) / 32, MAXIT = 3;   // (TR + 4) rows / nw warps <= 3 for every geometry spgg_create picks
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  if ((g.TR + 4 + nw - 1) / nw > MAXIT) __trap();      // a geometry this staging does not cover must not run silently
  const int cmax = g.L + GC;                       // first column without a current image
  // strategy words can be taken whole where no column of the halo'd tile wraps
  const bool wordpath = STEP && c0 >= 32 && c0 + TC + 2 <= g.L;
  Code cv[MAXIT][NQ];
  RT rv[MAXIT][NQ];
  uint32_t sw[MAXIT];
#pragma unroll
  for (int it = 0; it < MAXIT; ++it) {
    const int r = warp + it * nw, rr = r - 2, prow = r0 + rr + GH;
    const bool rowok = r < g.TR + 4 && prow < g.rows + 2 * GH;
    const bool in_cr = rowok && rr >= -M && rr < g.TR + M;
    const long long rowoff = (long long)prow * g.pitchB + CPAD + c0;
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      const int cc = q * 32 + lane - 2;
      const bool ok = in_cr && cc >= -M && cc < TC + M && c0 + cc < cmax;
      cv[it][q] = ok ? code_in[rowoff + cc] : Code(0);
      if constexpr (STEP) rv[it][q] = ok ? R_in[rowoff + cc] : RT(0);
    }
    if constexpr (STEP)
      sw[it] = (wordpath && rowok && lane < 6) ? S_in[(long long)prow * g.pitchW + WPAD + (c0 >> 5) - 1 + lane] : 0u;
  }
  Val vv[MAXIT][NQ];
#pragma unroll
  for (int it = 0; it < MAXIT; ++it) {
    const int r = warp + it * nw, rr = r - 2;
    const bool rowact = r < g.TR + 4;
    const bool in_cr = rowact && rr >= -M && rr < g.TR + M;
    const int base = (rr + HR) * SMW + HP;
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      const int cc = q * 32 + lane - 2;
      if constexpr (Md::kFp64) vv[it][q] = __ldg(vtab + 2 * (size_t)(cv[it][q] >> 1));   // code 0 is a valid entry
      else vv[it][q] = sm_tab[cv[it][q] >> 1];
      if constexpr (STEP) {
        if (in_cr && cc >= -M && cc < TC + M) {
          sm_code[base + cc] = cv[it][q];
          sm_R[base + cc] = rv[it][q];
        }
        // cooperator flag of the cell: bit cc & 31 of word (cc + 32) >> 5 of the six (c0 is a multiple of 32)
        const uint32_t w = __shfl_sync(0xffffffffu, sw[it], (cc + 32) >> 5);
        const bool rowok = r0 + rr + GH < g.rows + 2 * GH;      // rows below the ghost rows read as defectors
        if (wordpath && rowact && cc < TC + 2) sm_C[base + cc] = rowok ? (uint8_t)((~w >> (cc & 31)) & 1u) : (uint8_t)0;
      }
    }
  }
#pragma unroll
  for (int it = 0; it < MAXIT; ++it) {
    const int r = warp + it * nw, rr = r - 2;
    const bool in_cr = r < g.TR + 4 && rr >= -M && rr < g.TR + M;
    const int base = (rr + HR) * SMW + HP;
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      const int cc = q * 32 + lane - 2;
      if (in_cr && cc >= -M && cc < TC + M) sm_val[base + cc] = vv[it][q];
    }
  }
  if constexpr (STEP) {
    if (!wordpath) load_coop_tile(sm_C, S_in, g, r0, c0, g.TR);   // edge tile columns: per-cell wrap
  }
}

// =================================================================== k_step
template <class Md>
struct SmemLayout {
  size_t off_code, off_val, off_R, off_C, off_N, off_tab, off_red, total;
  __host__ __device__ constexpr explicit SmemLayout(int TR)
      : off_code(0), off_val(0), off_R(0), off_C(0), off_N(0), off_tab(0), off_red(0), total(0) {
    const size_t n = (size_t)(TR + 2 * HR) * SMW;
    size_t o = 0;
    off_val = o;  o = (o + sizeof(typename Md::Val) * n + 15) / 16 * 16;
    off_R = o;    o = (o + sizeof(typename Md::R) * n + 15) / 16 * 16;
    off_code = o; o = (o + sizeof(typename Md::Code) * n + 15) / 16 * 16;
    off_C = o;    o = (o + n + 15) / 16 * 16;
    off_N = o;    o = (o + n + 15) / 16 * 16;
    off_tab = o;  o = (o + 256 * sizeof(float) + 15) / 16 * 16;
    off_red = o;  o = (o + sizeof(double) * (MAX_THREADS / 32) * NSTAT + 15) / 16 * 16;
    total = o;
  }
};

template <class T>
__device__ __forceinline__ T sel4(int e, T a0, T a1, T a2, T a3) {
  const T lo = (e & 1) ? a1 : a0, hi = (e & 1) ? a3 : a2;
  return (e & 2) ? hi : lo;
}

// per-thread statistics of a launch, handed to step_epilogue (k_step and k_step_lean share the fold)
struct StepSums {
  unsigned long long cls_n[4], cls_sn[4], grp[6], n_best, n_best2, n_sel_coop;
  double sumQ[4], sumQC[4], sumNI, sumR, sumRatio;
};

// per-CTA partial row, then the last CTA of the replica folds the rows in a fixed order (deterministic)
// and finishes the public stat row.  The payoff and reward sums of every mode come from exact integer
// counts: sum of P over a class = ((rc SigmaN / 5 - 5 cost C n) - lo n) / span (spgg.py:256-257,373-377).
template <class Md>
__device__ __forceinline__ void step_epilogue(const KArgs &a, int rep, int cta, const RepConst &rc,
                                              const StepSums &t, double *sm_red, int *s_is_last, bool upd, bool sel) {
  typedef typename Md::Val Val;
  constexpr bool kI8 = (sizeof(typename Md::R) == 1);
  const Geom &g = a.g;
  double v[NSTAT];
#pragma unroll
  for (int z = 0; z < NSTAT; ++z) v[z] = 0.0;
  v[ST_NC_OLD] = (double)(t.cls_n[2] + t.cls_n[3]);
  v[ST_N_CD] = (double)t.cls_n[2];
  v[ST_N_DC] = (double)t.cls_n[1];
  v[ST_NC_NEW] = (double)(t.cls_n[1] + t.cls_n[3]);
#pragma unroll
  for (int z = 0; z < 4; ++z) v[ST_X_SN0 + z] = (double)t.cls_sn[z];
  // raw class counts ride in these four slots until the fold below
  v[ST_SUM_P] = (double)t.cls_n[0]; v[ST_SUM_P_C] = (double)t.cls_n[1];
  v[ST_SUM_P_D] = (double)t.cls_n[2]; v[ST_SUM_WP_P] = (double)t.cls_n[3];
  v[ST_SUM_RATIO] = t.sumRatio;
#pragma unroll
  for (int z = 0; z < 6; ++z) v[ST_GROUP0 + z] = (double)t.grp[z];
  v[ST_SUM_R] = t.sumR;
#pragma unroll
  for (int z = 0; z < 4; ++z) {
    v[ST_SUM_Q + z] = t.sumQ[z];
    v[ST_SUM_Q_C + z] = t.sumQC[z];
  }
  v[ST_SUM_NI] = t.sumNI;
  v[ST_N_BEST_POS] = (double)t.n_best;
  v[ST_N_BEST_2ND] = (double)t.n_best2;
  v[ST_X_NSEL] = (double)t.n_sel_coop;
  __syncthreads();
  block_reduce<NSTAT>(v, sm_red);
  double *part = a.partials + ((long long)rep * g.ctas_per_rep + cta) * NSTAT;
  if (threadIdx.x < NSTAT) part[threadIdx.x] = sm_red[threadIdx.x];
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned tk = atomicInc(a.tickets + rep, (unsigned)g.ctas_per_rep - 1u);
    *s_is_last = (tk == (unsigned)g.ctas_per_rep - 1u);
  }
  __syncthreads();
  if (!*s_is_last) return;
  __threadfence();
  fold_partials(a.partials + (long long)rep * g.ctas_per_rep * NSTAT, g.ctas_per_rep, sm_red);
  if (threadIdx.x == 0) {
    double *row = a.stats + ((long long)rep * a.cap + a.rel) * NSTAT;
    double *s = sm_red;
    if constexpr (kI8) s[ST_SUM_R] *= rc.rq;
    if (upd) {
      double Pc[4];
      const double nc[4] = {s[ST_SUM_P], s[ST_SUM_P_C], s[ST_SUM_P_D], s[ST_SUM_WP_P]};
      for (int z = 0; z < 4; ++z) {
        const double C = (z >> 1) ? 1.0 : 0.0;
        Pc[z] = ((rc.rc * s[ST_X_SN0 + z] / 5.0 - 5.0 * rc.cost * C * nc[z]) - rc.lo * nc[z]) /
                rc.span;
      }
      s[ST_SUM_P] = Pc[0] + Pc[1] + Pc[2] + Pc[3];
      s[ST_SUM_P_C] = Pc[2] + Pc[3];
      s[ST_SUM_P_D] = Pc[0] + Pc[1];
      s[ST_SUM_WP_P] = rc.wP * s[ST_SUM_P];
      s[ST_SUM_REW_C] = rc.wP * (Pc[1] + Pc[3]) + rc.wR * 0.5 * (nc[1] + nc[3]);
      s[ST_SUM_REW_D] = rc.wP * (Pc[0] + Pc[2]);
      for (int z = 0; z < 4; ++z) s[ST_SUM_Q_D + z] = s[ST_SUM_Q + z] - s[ST_SUM_Q_C + z];
      s[ST_GMAX] = (double)reinterpret_cast<const Val *>(a.gmax)[(long long)rep * a.cap + a.rel];
      for (int z = 0; z < ST_X_SN0; ++z) row[z] = s[z];  // scratch columns stay zero
    } else {
      row[ST_SUM_R] = s[ST_SUM_R];
    }
    // uniform lattice after the action just chosen -> the next iteration breaks (spgg.py:405).
    // Only a handle that owns the whole lattice can tell; strips decide on the host.
    if (sel && g.wrap_rows) {
      const double nsel = s[ST_X_NSEL];
      if (nsel == 0.0 || nsel == (double)g.site_stride) a.stop_at[rep] = a.j + 1;
    }
  }
}

// ------------------------------------------------------------------ site code of k_step and k_step_lean
// k_step_lean (spgg_lean.cuh) must give k_step's results bit for bit: the pieces they share live here once.
// The statistics, the epsilon-greedy choice and the stores stay in the kernels: as helpers they reorder
// k_step_lean's machine code.  So does the group-count loop in k_step, where it adds spills (SARSA at fp32).

// the replica's constants into shared memory, then NTAB of its fp32 tables (reward, ratio statistic) into sm_tab
template <int NTAB>
__device__ __forceinline__ void load_rep_const(RepConst &s_rc, const RepConst *src, float *sm_tab) {
  for (int i = threadIdx.x; i < (int)(sizeof(RepConst) / 4); i += blockDim.x)
    reinterpret_cast<uint32_t *>(&s_rc)[i] = reinterpret_cast<const uint32_t *>(src)[i];
  __syncthreads();
  if constexpr (NTAB > 0) {
    for (int i = threadIdx.x; i < 128; i += blockDim.x) {
      sm_tab[i] = s_rc.rewtab[i];
      if constexpr (NTAB > 1) sm_tab[128 + i] = s_rc.ratiotab[i];
    }
  }
}

// denominator of lambda from the launch's global maximum (spgg.py:489): fp64 divides by den, fp32 multiplies by inv_den
template <class Md>
__device__ __forceinline__ void lambda_den(const KArgs &a, int rep, const RepConst &rc, typename Md::Val &den,
                                           typename Md::Val &inv_den) {
  const typename Md::Val gm = reinterpret_cast<const typename Md::Val *>(a.gmax)[(long long)rep * a.cap + a.rel];
  if constexpr (Md::kFp64) den = __dadd_rn(gm, rc.leps);
  else inv_den = __fdiv_rn(1.0f, __fadd_rn(gm, rc.leps_f));
}

// Philox words of the four sites a lane owns in the 128-site row segment at column c0 (c0 + 32*k4 + lane):
// counter = (column / 4, global row, ctr2, ctr3), one call serves 4 consecutive sites.  This lane computes the
// words of columns c0+4*lane..+3; its own sites fetch theirs from lane 8*k4 + lane/4, word lane%4.
__device__ __forceinline__ void philox_row(int c0, int row, uint32_t ctr2, uint32_t ctr3, const RepConst &rc, int lane,
                                           uint32_t w4[4]) {
  uint32_t wc[4];
  philox4x32_10((uint32_t)((c0 >> 2) + lane), (uint32_t)row, ctr2, ctr3, rc.seed_lo, rc.seed_hi, wc);
#pragma unroll
  for (int k4 = 0; k4 < 4; ++k4) {
    const int src = 8 * k4 + (lane >> 2);
    const uint32_t x0 = __shfl_sync(0xffffffffu, wc[0], src), x1 = __shfl_sync(0xffffffffu, wc[1], src);
    const uint32_t x2 = __shfl_sync(0xffffffffu, wc[2], src), x3 = __shfl_sync(0xffffffffu, wc[3], src);
    w4[k4] = sel4<uint32_t>(lane & 3, x0, x1, x2, x3);
  }
}

// neighbour-aware term inputs (spgg.py:486-494): the largest neighbour reward difference d (first arg-max wins),
// that neighbour's shared-memory index and its offset number k
template <class Val>
struct BestNeighbour {
  Val d;
  int idx, k;
};
template <class Md, int M>
__device__ __forceinline__ BestNeighbour<typename Md::Val> best_neighbour(const typename Md::Val *sm_val, int sr, int sc,
                                                                          typename Md::Val vx) {
  typedef typename Md::Val Val;
  constexpr int NK = (M == 2) ? 12 : 4;
  Val best = Val(0);
  int bidx = sr * SMW + sc, kstar = 0;
#pragma unroll
  for (int k = 0; k < NK; ++k) {
    const int nidx = (sr - c_off[k][0]) * SMW + (sc - c_off[k][1]);
    const Val vk = sm_val[nidx];
    Val d;
    if constexpr (Md::kFp64) d = __dsub_rn(vk, vx);
    else d = __fsub_rn(vk, vx);
    if (k == 0 || d > best) { best = d; bidx = nidx; kstar = k; }
  }
  return {best, bidx, kstar};
}

// fp32 TD update of Q[s][act] (algorithms.py:122-131) plus the neighbour-aware term (spgg.py:478-509); returns the
// new entry and adds the site's NI statistic (spgg.py:512) to tni.  next(x0, x1, after) is the value of the next
// state's row (x0, x1) before (after = false) and after (true) the TD write; na, nb is that row before it.
template <class NextF>
__device__ __forceinline__ float td_update_f32(const RepConst &rc, float vx, float qe, float na, float nb, int s,
                                               int s_new, int act, float best, bool same, float inv_den, NextF next,
                                               float &tni) {
  const float mx = next(na, nb, false);
  const float td = __fsub_rn(__fmaf_rn(rc.gamma_f, mx, vx), qe);
  const float qtd = __fmaf_rn(rc.alpha_f, td, qe);
  const float lam = __fmul_rn(__fmul_rn(rc.kappa_f, fmaxf(0.0f, best)), inv_den);
  const float nu = same ? lam : -lam;
  const float na2 = (s_new == s && act == 0) ? qtd : na;
  const float nb2 = (s_new == s && act == 1) ? qtd : nb;
  const float td2 = __fsub_rn(__fmaf_rn(rc.gamma_f, next(na2, nb2, true), vx), qtd);
  const float qfin = __fadd_rn(qtd, nu);
  const float an = fabsf(nu);
  tni = __fmaf_rn(__fdividef(an, __fadd_rn(__fadd_rn(fabsf(__fmul_rn(rc.alpha_f, td2)), an), 1e-8f)), 100.0f, tni);
  return qfin;
}


// The general kernel is latency-bound (one site per thread and row, dependent shared-memory stencils):
// what it needs is resident warps, not registers.  Measured at L=4000 (fp32, int8 R), us per iteration:
// 1 CTA/SM (190 registers) 1604, 2 CTAs/SM 891, 3 CTAs/SM (80 registers, a few hundred bytes of spills) 718.
#ifndef SPGG_GEN_MINBLOCKS
#define SPGG_GEN_MINBLOCKS 3
#endif
template <class Md, int M, bool ACTION, bool REPLAY>
__global__ void __launch_bounds__(MAX_THREADS, SPGG_GEN_MINBLOCKS) k_step(KArgs a) {
  typedef typename Md::Q QT;
  typedef typename Md::R RT;
  typedef typename Md::Code Code;
  typedef typename Md::Val Val;
  constexpr bool kI8 = (sizeof(RT) == 1);
  const Geom &g = a.g;
  const int rep = blockIdx.x / g.ctas_per_rep, cta = blockIdx.x % g.ctas_per_rep;
  pdl_launch_dependents();  // launched with programmatic stream serialization only when a launch is short (spgg_capi.cu)
  pdl_wait();  // the planes, the stop flags and gmax come from the kernels before this one
  const int stop = a.stop_at[rep];
  if (stop >= 0 && a.j > stop) return;
  const bool upd = a.do_update != 0;
  const bool sel = (a.do_select != 0) && !(stop >= 0 && a.j == stop);

  extern __shared__ __align__(16) unsigned char smem[];
  const SmemLayout<Md> lay(g.TR);
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
  const bool dq = (a.algo == 3);  // Double Q-learning keeps two tables per site: [site][table][s][a]
  QT *Qp = reinterpret_cast<QT *>(a.Q) + (long long)rep * g.site_stride * (dq ? 8 : 4);
  const RT *R_in = reinterpret_cast<const RT *>(a.R_in) + (long long)rep * g.plane_stride;
  RT *R_out = reinterpret_cast<RT *>(a.R_out) + (long long)rep * g.plane_stride;
  const Code *code_in = reinterpret_cast<const Code *>(a.code_in) + (long long)rep * g.plane_stride;
  Code *code_out = reinterpret_cast<Code *>(a.code_out) + (long long)rep * g.plane_stride;
  const uint32_t *S_in = a.S_in + (long long)rep * g.bits_stride;
  uint32_t *S_out = a.S_out + (long long)rep * g.bits_stride;
  // contraction-free arithmetic in the table's precision (reference operation order in fp64)
  auto q_add = [](QT x, QT y) -> QT { if constexpr (Md::kFp64) return __dadd_rn(x, y); else return __fadd_rn(x, y); };
  auto q_sub = [](QT x, QT y) -> QT { if constexpr (Md::kFp64) return __dsub_rn(x, y); else return __fsub_rn(x, y); };
  auto q_mul = [](QT x, QT y) -> QT { if constexpr (Md::kFp64) return __dmul_rn(x, y); else return __fmul_rn(x, y); };
  auto q_div = [](QT x, QT y) -> QT { if constexpr (Md::kFp64) return __ddiv_rn(x, y); else return __fdiv_rn(x, y); };
  auto q_max = [](QT x, QT y) -> QT { return x > y ? x : (y > x ? y : x); };
  auto q_mean = [&](QT x, QT y) -> QT { return q_div(q_add(x, y), QT(2)); };

  // scalars of this launch
  Val inv_den = Val(0), den = Val(1);
  if (upd) lambda_den<Md>(a, rep, rc, den, inv_den);
  const long long tab_idx = (long long)(a.rel + 1) * g.n_rep + rep;
  // SARSA / Expected SARSA evaluate the policy of the iteration being finished (epsilon_j)
  const double eps_u = (upd && a.algo != 0) ? a.eps_tab[(long long)a.rel * g.n_rep + rep] : 0.0;
  const uint32_t thr_u = (upd && a.algo == 1) ? a.thr_tab[(long long)a.rel * g.n_rep + rep] : 0u;
  const uint32_t thr = sel ? a.thr_tab[tab_idx] : 0u;
  const double eps = (sel && REPLAY) ? a.eps_tab[tab_idx] : 0.0;

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;

  // per-thread statistics (exact integers, doubles folded once per tile)
  unsigned long long cls_n[4] = {0, 0, 0, 0};   // by class = C_old*2 + coop
  unsigned long long cls_sn[4] = {0, 0, 0, 0};  // fp32 mode: sum of SigmaN per class
  unsigned long long grp[6] = {0, 0, 0, 0, 0, 0};
  unsigned long long n_best = 0, n_best2 = 0, n_sel_coop = 0;
  double sumQ[4] = {0, 0, 0, 0}, sumQC[4] = {0, 0, 0, 0};
  double sumNI = 0.0, sumR = 0.0, sumRatio = 0.0;

  const int n_tiles = g.n_tx * g.n_ty;
  for (int tile = cta; tile < n_tiles; tile += g.ctas_per_rep) {
    const int r0 = (tile / g.n_tx) * g.TR, c0 = (tile % g.n_tx) * TC;
    __syncthreads();
    // ---- stage tiles + halos: all loads of a thread in flight at once (stage_tile; the codes and their rewards are
    // staged for a select-only launch too - they are not read then)
    stage_tile<Md, M, true>(g, r0, c0, code_in, R_in, S_in, rc, sm_tab, vtab, sm_val, sm_code, sm_R, sm_C);
    __syncthreads();
    {
      // N = cooperators in the 5-site group centred on each site (spgg.py:23-36) of S_j,
      // for the tile and a one-site ring
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

    // per-tile packed counters (flushed below): 8-bit class counts, 16-bit SigmaN sums,
    // 10-bit group histogram; a thread sees at most 4*TR/nw <= 64 sites per tile
    unsigned pk_n = 0;
    unsigned long long pk_sn = 0, pk_grp = 0;
    float tq[4] = {0.f, 0.f, 0.f, 0.f}, tqc[4] = {0.f, 0.f, 0.f, 0.f};
    float tni = 0.f, tratio = 0.f, trf = 0.f;
    int tri = 0;

    // ---- per-site work: warp = one 128-site row segment, lane = 4 sites strided by 32
    for (int rr = warp; rr < g.TR; rr += nw) {
      const int i = r0 + rr;
      if (i >= g.rows) break;
      const int sr = rr + HR;
      uint32_t w4[4] = {0, 0, 0, 0};
      if (sel && !REPLAY) philox_row(c0, g.row0 + i, (uint32_t)(a.j + 1), 0u, rc, lane, w4);
      uint32_t wS1[4] = {0, 0, 0, 0}, wS2[4] = {0, 0, 0, 0};
      if (upd && (a.algo == 1 || a.algo == 3) && a.u2 == nullptr) {
        // SARSA's two further draws of iteration j: Philox streams 1 and 2 (counter word 3)
        philox_row(c0, g.row0 + i, (uint32_t)a.j, 1u, rc, lane, wS1);
        philox_row(c0, g.row0 + i, (uint32_t)a.j, 2u, rc, lane, wS2);
      }
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) {
        const int cc = k4 * 32 + lane;
        const int col = c0 + cc;
        const bool valid = col < g.L;
        const int sc = cc + HP;
        const int sidx = sr * SMW + sc;
        int a_new = 0;
        if (valid) {
          const long long site = (long long)i * g.L + col;
          QT q0_, q1_, q2_, q3_;
          QT t1[4], t2[4];  // Double Q-learning: the two tables (algorithms.py:245-247); q*_ = their mean
          if (dq) {
#pragma unroll
            for (int z = 0; z < 4; ++z) { t1[z] = Qp[site * 8 + z]; t2[z] = Qp[site * 8 + 4 + z]; }
            q0_ = q_mean(t1[0], t2[0]); q1_ = q_mean(t1[1], t2[1]);   // get_combined_q_table, algorithms.py:263
            q2_ = q_mean(t1[2], t2[2]); q3_ = q_mean(t1[3], t2[3]);
          } else if constexpr (Md::kFp64) {
            const double2 lo2 = reinterpret_cast<const double2 *>(Qp)[site * 2];
            const double2 hi2 = reinterpret_cast<const double2 *>(Qp)[site * 2 + 1];
            q0_ = lo2.x; q1_ = lo2.y; q2_ = hi2.x; q3_ = hi2.y;
          } else {
            const float4 v = reinterpret_cast<const float4 *>(Qp)[site];
            q0_ = v.x; q1_ = v.y; q2_ = v.z; q3_ = v.w;
          }
          const RT r_old = sm_R[sidx];
          const int Ccur = sm_C[sidx];
          // post-action state of iteration j == pre-action state of iteration j+1
          const int s_new = ACTION ? Ccur : rep_state<RT, M>(sm_R, sr, sc);
          if constexpr (kI8) tri += (int)r_old;
          else if constexpr (sizeof(RT) == 4) trf += r_old;
          else sumR += r_old;

          if (upd) {
            const Code code = sm_code[sidx];
            const int s = code & 1u, coop = (code >> 1) & 1u, wasC = (code >> 2) & 1u;
            const int act = coop ^ 1;
            const Val vx = sm_val[sidx];
            const auto bn = best_neighbour<Md, M>(sm_val, sr, sc, vx);
            const Val best = bn.d;
            const bool same = (((sm_code[bn.idx] >> 1) & 1u) == (unsigned)coop);
            const int e = 2 * s + act;
            const QT qe = sel4<QT>(e, q0_, q1_, q2_, q3_);
            const QT na = s_new ? q2_ : q0_, nb = s_new ? q3_ : q1_;  // pre-update row of s'
            QT qtd, qfin;
            // SARSA: the eps-greedy draws that pick the next action (update, then NI statistic)
            bool ex1 = false, ex2 = false;
            int rn1 = 0, rn2 = 0;
            if (a.algo == 1) {
              if (a.u2 != nullptr) {
                ex1 = a.u2[site] < eps_u; rn1 = a.b2[site];
                ex2 = a.u3[site] < eps_u; rn2 = a.b3[site];
              } else {
                ex1 = (wS1[k4] >> 8) < thr_u; rn1 = (int)(wS1[k4] & 1u);
                ex2 = (wS2[k4] >> 8) < thr_u; rn2 = (int)(wS2[k4] & 1u);
              }
            }
            bool dq_done = false;
            if (dq) {
              // Double Q-learning (algorithms.py:292-341): a fair draw picks the table to update;
              // its TD target is the max of the OTHER table's row of s' (as the reference codes
              // it: next_q_1 = Q2[s', argmax Q2[s']], :320-325)
              const bool upd1 = (a.u2 != nullptr) ? (a.u2[site] < 0.5) : ((wS1[k4] >> 8) < (1u << 23));
              const int r0i = 2 * s_new;
              const QT nx1 = q_max(t2[r0i], t2[r0i + 1]), nx2 = q_max(t1[r0i], t1[r0i + 1]);
              const QT g_ = Md::kFp64 ? (QT)rc.gamma : (QT)rc.gamma_f, al_ = Md::kFp64 ? (QT)rc.alpha : (QT)rc.alpha_f;
              if (upd1) t1[e] = q_add(t1[e], q_mul(al_, q_sub(q_add(vx, q_mul(g_, nx1)), t1[e])));
              else t2[e] = q_add(t2[e], q_mul(al_, q_sub(q_add(vx, q_mul(g_, nx2)), t2[e])));
              // TD error of the combined table after the write (spgg.py:464-468)
              QT cq[4];
#pragma unroll
              for (int z = 0; z < 4; ++z) cq[z] = q_mean(t1[z], t2[z]);
              qtd = cq[e];
              const QT td2 = q_sub(q_add(vx, q_mul(g_, q_max(cq[r0i], cq[r0i + 1]))), qtd);
              QT lam;
              if constexpr (Md::kFp64) lam = ddiv_zero_safe(__dmul_rn(rc.kappa, fmax(0.0, best)), den);
              else lam = __fmul_rn(__fmul_rn(rc.kappa_f, fmaxf(0.0f, best)), inv_den);
              const QT nu = same ? lam : -lam;
              t1[e] = q_add(t1[e], nu);                      // spgg.py:499-505: both tables
              t2[e] = q_add(t2[e], nu);
              q0_ = q_mean(t1[0], t2[0]); q1_ = q_mean(t1[1], t2[1]);
              q2_ = q_mean(t1[2], t2[2]); q3_ = q_mean(t1[3], t2[3]);
              qfin = sel4<QT>(e, q0_, q1_, q2_, q3_);
              const QT an = nu < QT(0) ? -nu : nu;
              const QT atd = q_mul(al_, td2);
              const QT pct = q_mul(q_div(an, q_add(q_add(atd < QT(0) ? -atd : atd, an), (QT)1e-8)), (QT)100.0);
              if constexpr (Md::kFp64) {
                sumNI += pct;
                pk_sn += (unsigned long long)sigma_n_of_code(code) << (16 * (wasC * 2 + coop));
                if (coop)
                  sumRatio += __dmul_rn(
                      __ddiv_rn(fabs(__dmul_rn(rc.wR, 0.5)), __dadd_rn(fabs(vx), 1e-9)), 100.0);
              } else {
                tni += pct;
                pk_sn += (unsigned long long)(code >> 3) << (16 * (wasC * 2 + coop));
                if (rc.has_ratio && coop) tratio += sm_ratio[code >> 1];
              }
              dq_done = true;
            }
            if (dq_done) {
            } else if constexpr (Md::kFp64) {
              // value of the next state: max (algorithms.py:125), Q[s'][a'] (:169) or the
              // eps-greedy expectation p0*Q[s'][0] + p1*Q[s'][1] (:212-224)
              auto next_value = [&](double x0, double x1, bool ex, int rn) -> double {
                if (a.algo == 0) return fmax(x0, x1);
                const int greedy = (x1 > x0) ? 1 : 0;
                if (a.algo == 1) return (ex ? rn : greedy) ? x1 : x0;
                const double po = __ddiv_rn(eps_u, 2.0);
                const double pg = __dadd_rn(__dsub_rn(1.0, eps_u), po);
                return __dadd_rn(__dmul_rn(greedy ? po : pg, x0), __dmul_rn(greedy ? pg : po, x1));
              };
              const double mx = next_value(na, nb, ex1, rn1);
              const double td = __dsub_rn(__dadd_rn(vx, __dmul_rn(rc.gamma, mx)), qe);  // algorithms.py:128
              qtd = __dadd_rn(qe, __dmul_rn(rc.alpha, td));                              // algorithms.py:131
              const double lam = ddiv_zero_safe(__dmul_rn(rc.kappa, fmax(0.0, best)), den);  // spgg.py:489
              const double nu = same ? lam : -lam;                                       // spgg.py:494-495
              // TD error on the table after the TD write (spgg.py:446-473)
              const double na2 = (s_new == s && act == 0) ? qtd : na;
              const double nb2 = (s_new == s && act == 1) ? qtd : nb;
              const double td2 = __dsub_rn(__dadd_rn(vx, __dmul_rn(rc.gamma, next_value(na2, nb2, ex2, rn2))), qtd);
              qfin = __dadd_rn(qtd, nu);                                                 // spgg.py:509
              const double an = fabs(nu);
              sumNI += __dmul_rn(
                  ddiv_zero_safe(an, __dadd_rn(__dadd_rn(fabs(__dmul_rn(rc.alpha, td2)), an), 1e-8)),
                  100.0);                                                                // spgg.py:512
              // payoff / reward sums (spgg.py:381-392,419-426) come from exact integer counts at the fold,
              // as in the fp32 modes: sum P = ((rc SigmaN / 5 - 5 cost C n) - lo n) / span per class
              pk_sn += (unsigned long long)sigma_n_of_code(code) << (16 * (wasC * 2 + coop));
              if (coop)
                sumRatio += __dmul_rn(
                    __ddiv_rn(fabs(__dmul_rn(rc.wR, 0.5)), __dadd_rn(fabs(vx), 1e-9)), 100.0);
            } else {
              auto next_value = [&](float x0, float x1, bool after) -> float {
                if (a.algo == 0) return fmaxf(x0, x1);
                const int greedy = (x1 > x0) ? 1 : 0;
                if (a.algo == 1) return ((after ? ex2 : ex1) ? (after ? rn2 : rn1) : greedy) ? x1 : x0;
                const float e = (float)eps_u, po = __fmul_rn(e, 0.5f), pg = __fadd_rn(__fsub_rn(1.0f, e), po);
                return __fmaf_rn(greedy ? pg : po, x1, __fmul_rn(greedy ? po : pg, x0));
              };
              qfin = td_update_f32(rc, vx, qe, na, nb, s, s_new, act, best, same, inv_den, next_value, tni);
              pk_sn += (unsigned long long)(code >> 3) << (16 * (wasC * 2 + coop));
              if (rc.has_ratio && coop) tratio += sm_ratio[code >> 1];
            }
            if (!dq) {
              q0_ = (e == 0) ? qfin : q0_;
              q1_ = (e == 1) ? qfin : q1_;
              q2_ = (e == 2) ? qfin : q2_;
              q3_ = (e == 3) ? qfin : q3_;
            }
            pk_n += 1u << (8 * (wasC * 2 + coop));
            if (best > Val(0)) { n_best += 1u; n_best2 += (bn.k >= 4); }
            pk_grp += 1ull << (10 * (5 - (int)sm_N[sidx]));                              // spgg.py:586-592
            if constexpr (Md::kFp64) {
              sumQ[0] += q0_; sumQ[1] += q1_; sumQ[2] += q2_; sumQ[3] += q3_;
              if (wasC) { sumQC[0] += q0_; sumQC[1] += q1_; sumQC[2] += q2_; sumQC[3] += q3_; }
            } else {
              const float m = wasC ? 1.0f : 0.0f;
              tq[0] += q0_; tq[1] += q1_; tq[2] += q2_; tq[3] += q3_;
              tqc[0] = fmaf(m, q0_, tqc[0]); tqc[1] = fmaf(m, q1_, tqc[1]);
              tqc[2] = fmaf(m, q2_, tqc[2]); tqc[3] = fmaf(m, q3_, tqc[3]);
            }
          }

          if (sel) {
            int explore, rnd;
            if constexpr (REPLAY) {
              explore = a.u[site] < eps;  // algorithms.py:105
              rnd = a.b[site];            // algorithms.py:108
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
            const int n5[5] = {sm_N[sidx], sm_N[sidx - SMW], sm_N[sidx + SMW], sm_N[sidx - 1],
                               sm_N[sidx + 1]};
            const Code cnew = pack_code<Md>(n5, Ccur, a_new ^ 1, s_new);
            store_cell<Code>(code_out, g, i, col, cnew);
            store_cell<RT>(R_out, g, i, col, r_new);
          }
          if (upd) {
            if (dq) {
#pragma unroll
              for (int z = 0; z < 4; ++z) { Qp[site * 8 + z] = t1[z]; Qp[site * 8 + 4 + z] = t2[z]; }
            } else if constexpr (Md::kFp64) {
              reinterpret_cast<double2 *>(Qp)[site * 2] = make_double2(q0_, q1_);
              reinterpret_cast<double2 *>(Qp)[site * 2 + 1] = make_double2(q2_, q3_);
            } else {
              reinterpret_cast<float4 *>(Qp)[site] = make_float4(q0_, q1_, q2_, q3_);
            }
          }
        }
        if (sel) {
          const uint32_t word = __ballot_sync(0xffffffffu, valid && a_new);
          const int wi = (c0 >> 5) + k4;
          if (lane == 0 && wi * 32 < g.L) store_bits_word(S_out, g, i, wi, word);
        }
      }
    }
    // flush the per-tile packed counters
#pragma unroll
    for (int z = 0; z < 4; ++z) {
      cls_n[z] += (pk_n >> (8 * z)) & 0xffu;
      cls_sn[z] += (pk_sn >> (16 * z)) & 0xffffull;
      sumQ[z] += (double)tq[z];
      sumQC[z] += (double)tqc[z];
    }
#pragma unroll
    for (int z = 0; z < 6; ++z) grp[z] += (pk_grp >> (10 * z)) & 0x3ffull;
    sumNI += (double)tni;
    sumRatio += (double)tratio;
    sumR += (double)tri + (double)trf;
  }

  // ---- per-CTA partial row, then the last CTA of the replica folds them in a fixed order
  StepSums sums;
#pragma unroll
  for (int z = 0; z < 4; ++z) { sums.cls_n[z] = cls_n[z]; sums.cls_sn[z] = cls_sn[z]; sums.sumQ[z] = sumQ[z]; sums.sumQC[z] = sumQC[z]; }
#pragma unroll
  for (int z = 0; z < 6; ++z) sums.grp[z] = grp[z];
  sums.n_best = n_best; sums.n_best2 = n_best2; sums.n_sel_coop = n_sel_coop;
  sums.sumNI = sumNI; sums.sumR = sumR; sums.sumRatio = sumRatio;
  step_epilogue<Md>(a, rep, cta, rc, sums, sm_red, &s_is_last, upd, sel);
}

// strip decomposition: boundary rows <-> contiguous halo buffers --------------------
// buffer layout per replica: [GH rows of code][GH rows of R][GH rows of S bits]
template <class Md>
__global__ void k_halo_pack(Geom g, const void *code, const void *R, const uint32_t *S,
                            unsigned char *to_up, unsigned char *to_down, long long rep_bytes) {
  typedef typename Md::Code Code;
  typedef typename Md::R RT;
  const int rep = blockIdx.y;
  const long long nB = (long long)GH * g.pitchB, nW = (long long)GH * g.pitchW;
  const Code *cp = reinterpret_cast<const Code *>(code) + (long long)rep * g.plane_stride;
  const RT *rp = reinterpret_cast<const RT *>(R) + (long long)rep * g.plane_stride;
  const uint32_t *sp = S + (long long)rep * g.bits_stride;
  unsigned char *up = to_up + rep * rep_bytes, *dn = to_down + rep * rep_bytes;
  Code *upc = reinterpret_cast<Code *>(up), *dnc = reinterpret_cast<Code *>(dn);
  RT *upr = reinterpret_cast<RT *>(up + sizeof(Code) * nB), *dnr = reinterpret_cast<RT *>(dn + sizeof(Code) * nB);
  uint32_t *ups = reinterpret_cast<uint32_t *>(up + (sizeof(Code) + sizeof(RT)) * nB);
  uint32_t *dns = reinterpret_cast<uint32_t *>(dn + (sizeof(Code) + sizeof(RT)) * nB);
  const long long top = (long long)GH * g.pitchB, bot = (long long)g.rows * g.pitchB;  // first / last GH owned rows
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < nB;
       e += (long long)gridDim.x * blockDim.x) {
    upc[e] = cp[top + e]; upr[e] = rp[top + e];
    dnc[e] = cp[bot + e]; dnr[e] = rp[bot + e];
  }
  const long long topw = (long long)GH * g.pitchW, botw = (long long)g.rows * g.pitchW;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < nW;
       e += (long long)gridDim.x * blockDim.x) {
    ups[e] = sp[topw + e];
    dns[e] = sp[botw + e];
  }
}

template <class Md>
__global__ void k_halo_unpack(Geom g, void *code, void *R, uint32_t *S, const unsigned char *from_up,
                              const unsigned char *from_down, long long rep_bytes) {
  typedef typename Md::Code Code;
  typedef typename Md::R RT;
  const int rep = blockIdx.y;
  const long long nB = (long long)GH * g.pitchB, nW = (long long)GH * g.pitchW;
  Code *cp = reinterpret_cast<Code *>(code) + (long long)rep * g.plane_stride;
  RT *rp = reinterpret_cast<RT *>(R) + (long long)rep * g.plane_stride;
  uint32_t *sp = S + (long long)rep * g.bits_stride;
  const unsigned char *up = from_up + rep * rep_bytes, *dn = from_down + rep * rep_bytes;
  const Code *upc = reinterpret_cast<const Code *>(up), *dnc = reinterpret_cast<const Code *>(dn);
  const RT *upr = reinterpret_cast<const RT *>(up + sizeof(Code) * nB);
  const RT *dnr = reinterpret_cast<const RT *>(dn + sizeof(Code) * nB);
  const uint32_t *ups = reinterpret_cast<const uint32_t *>(up + (sizeof(Code) + sizeof(RT)) * nB);
  const uint32_t *dns = reinterpret_cast<const uint32_t *>(dn + (sizeof(Code) + sizeof(RT)) * nB);
  // the upper neighbour's *last* rows become our top ghosts; the lower neighbour's first rows our bottom ghosts
  const long long botg = (long long)(g.rows + GH) * g.pitchB;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < nB;
       e += (long long)gridDim.x * blockDim.x) {
    cp[e] = upc[e]; rp[e] = upr[e];
    cp[botg + e] = dnc[e]; rp[botg + e] = dnr[e];
  }
  const long long botgw = (long long)(g.rows + GH) * g.pitchW;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < nW;
       e += (long long)gridDim.x * blockDim.x) {
    sp[e] = ups[e];
    sp[botgw + e] = dns[e];
  }
}

// device-side initial state with the reference ctor's distributions (spgg.py:121,129,162):
// Q ~ U(-0.01, 0.01), R = 0, S ~ Bernoulli(1/2).  Philox counters use stream ids 1 (Q) and
// 2 (S) in word 3 so they never collide with the per-iteration draws (stream 0).
template <class Md>
__global__ void k_init_random(Geom g, int rep, void *Q, void *R, uint32_t *S, uint32_t seed_lo,
                              uint32_t seed_hi, int nq) {
  typedef typename Md::Q QT;
  typedef typename Md::R RT;
  QT *Qp = reinterpret_cast<QT *>(Q) + (long long)rep * g.site_stride * nq;
  RT *Rp = reinterpret_cast<RT *>(R) + (long long)rep * g.plane_stride;
  uint32_t *Sp = S + (long long)rep * g.bits_stride;
  const long long n_sites = g.site_stride;
  for (long long x = blockIdx.x * (long long)blockDim.x + threadIdx.x; x < n_sites;
       x += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(x / g.L), j = (int)(x % g.L);
    for (int t = 0; t < nq / 4; ++t) {  // one table, or the two of Double Q-learning
      uint32_t w[4];
      philox4x32_10((uint32_t)j, (uint32_t)(g.row0 + i), (uint32_t)t, 1u, seed_lo, seed_hi, w);
#pragma unroll
      for (int z = 0; z < 4; ++z) {
        // 24-bit uniform in [0,1) -> [-0.01, 0.01)
        const double uu = (double)(w[z] >> 8) * (1.0 / 16777216.0);
        Qp[x * nq + 4 * t + z] = (QT)(-0.01 + 0.02 * uu);
      }
    }
  }
  // strategy bits from stream 2, written through the ghost-aware store; R planes are zero
  const int nW = (g.L + 31) >> 5;
  const long long n_words = (long long)g.rows * nW;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n_words;
       e += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(e / nW), wi = (int)(e % nW);
    uint32_t w[4];
    philox4x32_10((uint32_t)(wi >> 2), (uint32_t)(g.row0 + i), 0u, 2u, seed_lo, seed_hi, w);
    uint32_t word = w[wi & 3];
    const int rem = g.L - wi * 32;
    if (rem < 32) word &= (1u << rem) - 1u;
    store_bits_word(Sp, g, i, wi, word);
  }
  const long long n_plane = (long long)(g.rows + 2 * GH) * g.pitchB;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n_plane;
       e += (long long)gridDim.x * blockDim.x)
    Rp[e] = RT(0);
}

// host layout (reference arrays: _Sn bytes 0/1, R float64, q_table float64 (rows,L,2,2))
// <-> device planes, `nrows` rows starting at local row i0.  One warp per 32-site word.
// info[0] = error flag (1: S not 0/1, 2: R not representable in int8 units), info[1] = #cooperators,
// info[2] = 1 if an int8 R lies outside [-16, 15] units (beyond k_step_fast's biased bytes)
template <class Md>
__global__ void k_import_rows(Geom g, int rep, int i0, int nrows, const uint8_t *S, const double *R,
                              const double *Q, void *Qd, void *Rd, uint32_t *Sd, double rq,
                              unsigned long long *info, int nq) {
  typedef typename Md::Q QT;
  typedef typename Md::R RT;
  QT *Qp = reinterpret_cast<QT *>(Qd) + (long long)rep * g.site_stride * nq;
  RT *Rp = reinterpret_cast<RT *>(Rd) + (long long)rep * g.plane_stride;
  uint32_t *Sp = Sd + (long long)rep * g.bits_stride;
  const int lane = threadIdx.x & 31;
  const int words = (g.L + 31) / 32;
  const long long n_items = (long long)nrows * words;
  const long long warp0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  unsigned long long coop = 0;
  bool wide = false;
  for (long long it = warp0; it < n_items; it += n_warps) {
    const int ii = (int)(it / words), w = (int)(it % words);
    const int i = i0 + ii, col = w * 32 + lane;
    const bool valid = col < g.L;
    int bit = 0;
    RT rv = RT(0);
    if (valid) {
      const long long src = (long long)ii * g.L + col;
      const uint8_t sv = S[src];
      if (sv > 1) atomicExch(info, 1ull);
      bit = sv & 1;
      const double r = R[src];
      if constexpr (sizeof(RT) == 1) {
        const double q = r / rq;
        if (q != floor(q) || q < -128.0 || q > 127.0) atomicExch(info, 2ull);
        wide = wide || q < -16.0 || q > 15.0;
        rv = (RT)(int)q;
      } else {
        rv = (RT)r;
      }
      const long long site = (long long)i * g.L + col;
      for (int z = 0; z < nq; ++z) Qp[site * nq + z] = (QT)Q[src * nq + z];
    }
    const uint32_t word = __ballot_sync(0xffffffffu, valid && bit);
    const uint32_t vmask = __ballot_sync(0xffffffffu, valid);
    if (lane == 0) coop += __popc(vmask & ~word);
    if (valid) store_cell<RT>(Rp, g, i, col, rv);
    if (lane == 0) store_bits_word(Sp, g, i, w, word);
  }
  if (lane == 0 && coop) atomicAdd(info + 1, coop);
  if (wide) atomicExch(info + 2, 1ull);
}

template <class Md>
__global__ void k_export_rows(Geom g, int rep, int i0, int nrows, uint8_t *S, double *R, double *Q,
                              const void *Qd, const void *Rd, const uint32_t *Sd, double rq, int nq) {
  typedef typename Md::Q QT;
  typedef typename Md::R RT;
  const QT *Qp = reinterpret_cast<const QT *>(Qd) + (long long)rep * g.site_stride * nq;
  const RT *Rp = reinterpret_cast<const RT *>(Rd) + (long long)rep * g.plane_stride;
  const uint32_t *Sp = Sd + (long long)rep * g.bits_stride;
  const long long n = (long long)nrows * g.L;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n;
       e += (long long)gridDim.x * blockDim.x) {
    const int ii = (int)(e / g.L), col = (int)(e % g.L);
    const int i = i0 + ii;
    if (S) S[e] = (uint8_t)((Sp[(long long)(i + GH) * g.pitchW + WPAD + (col >> 5)] >> (col & 31)) & 1u);
    if (R) {
      const RT rv = Rp[(long long)(i + GH) * g.pitchB + CPAD + col];
      R[e] = (sizeof(RT) == 1) ? (double)rv * rq : (double)rv;
    }
    if (Q) {
      const long long site = (long long)i * g.L + col;
      for (int z = 0; z < nq; ++z) Q[e * nq + z] = (double)Qp[site * nq + z];
    }
  }
}

// Position-keyed digests of one replica's owned rows: out[0] strategies, out[1] reputations,
// out[2] Q.  Every site contributes (hash(global row, column[, entry]) | 1) * (value bits + 1)
// modulo 2^64, so the digests of the strips of a lattice ADD UP to the digest of the whole lattice:
// an N-strip run is compared with a single-handle run without moving either state to the host.
// The multiplier is odd, hence invertible mod 2^64: any change of one value changes its term.  (An
// even one would miss a sign flip, which moves the bits by 2^63.)  oracle_state_digest restates this.
__device__ __forceinline__ unsigned long long digest_mix(unsigned long long x) {
  x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
  return x;
}
template <class Md>
__global__ void k_state_digest(Geom g, int rep, const void *Qd, const void *Rd, const uint32_t *Sd, int nq,
                               double rq, unsigned long long *out) {
  typedef typename Md::Q QT;
  typedef typename Md::R RT;
  const QT *Qp = reinterpret_cast<const QT *>(Qd) + (long long)rep * g.site_stride * nq;
  const RT *Rp = reinterpret_cast<const RT *>(Rd) + (long long)rep * g.plane_stride;
  const uint32_t *Sp = Sd + (long long)rep * g.bits_stride;
  unsigned long long dS = 0, dR = 0, dQ = 0;
  const long long n = g.site_stride;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n;
       e += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(e / g.L), col = (int)(e % g.L);
    const unsigned long long key = ((unsigned long long)(unsigned)(g.row0 + i) << 32) | (unsigned)col;
    const unsigned long long hS = digest_mix(key * 3 + 1) | 1ull, hR = digest_mix(key * 3 + 2) | 1ull;
    const unsigned bit = (Sp[(long long)(i + GH) * g.pitchW + WPAD + (col >> 5)] >> (col & 31)) & 1u;
    dS += hS * (unsigned long long)(bit + 1u);
    double rv = (double)Rp[(long long)(i + GH) * g.pitchB + CPAD + col];
    if (sizeof(RT) == 1) rv *= rq;  // int8 units -> the reference's value
    dR += hR * ((unsigned long long)__double_as_longlong(rv) + 1ull);
    for (int z = 0; z < nq; ++z) {
      const double qv = (double)Qp[e * nq + z];
      dQ += (digest_mix(key * 3 + 3 + ((unsigned long long)(z + 1) << 58)) | 1ull) *
            ((unsigned long long)__double_as_longlong(qv) + 1ull);
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    dS += __shfl_down_sync(0xffffffffu, dS, o);
    dR += __shfl_down_sync(0xffffffffu, dR, o);
    dQ += __shfl_down_sync(0xffffffffu, dQ, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(out + 0, dS);
    atomicAdd(out + 1, dR);
    atomicAdd(out + 2, dQ);
  }
}

// Strips: the per-iteration vector {max, any D, any C, -} has been max-reduced over the ranks.  One thread.
static __global__ void k_strip_verify(float *gvec, int rel, int j, int was_upd, int was_spec, int was_sel, float *gcarry,
                               float *gmax_tab, int *bad_at, int *stop_at) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (*bad_at < rel) return;                        // a failed guess earlier in the chunk: nothing after it ran
  // the lattice is uniform (spgg.py:405): the launch returned at once - or, at the stopping iteration itself,
  // only finished the update and had nothing to do if it was a select-only launch
  if (stop_at[0] >= 0 && (j > stop_at[0] || (j == stop_at[0] && !was_upd))) return;
  if (was_upd) {
    const float g_exact = gvec[4 * rel + 0];
    const float guess = gcarry[0];
    gmax_tab[rel] = g_exact;
    gcarry[0] = g_exact;
    // (was_spec == 2: the test hook made the launch use a value that is certainly not the maximum)
    if (was_spec == 2 || (was_spec && g_exact != guess)) { atomicMin(bad_at, rel); return; }
  }
  // every action of the lattice is the same: the next iteration breaks (spgg.py:405)
  if (was_sel && (gvec[4 * rel + 1] == 0.0f || gvec[4 * rel + 2] == 0.0f) && stop_at[0] < 0) stop_at[0] = j + 1;
}

// np.histogram(R, bins=nb, range=(edges[0], edges[nb])) of one replica's reputations (spgg.py:399-401,
// 626-628) without moving the lattice to the host: uniform bins, the last one closed on the right, the
// float index corrected against the edges exactly as NumPy's uniform-bin path does.  nb <= 64.
template <class Md>
__global__ void k_r_histogram(Geom g, int rep, const void *Rd, double rq, int nb, const double *edges,
                              unsigned long long *counts) {
  typedef typename Md::R RT;
  __shared__ unsigned int s_cnt[64];
  __shared__ double s_edge[65];
  const RT *Rp = reinterpret_cast<const RT *>(Rd) + (long long)rep * g.plane_stride;
  if (threadIdx.x < 64) s_cnt[threadIdx.x] = 0u;
  if (threadIdx.x <= nb) s_edge[threadIdx.x] = edges[threadIdx.x];
  __syncthreads();
  const double lo = s_edge[0], hi = s_edge[nb];
  const double norm = (double)nb / (hi - lo);
  const long long n = g.site_stride;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n;
       e += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(e / g.L), col = (int)(e % g.L);
    double v = (double)Rp[(long long)(i + GH) * g.pitchB + CPAD + col];
    if (sizeof(RT) == 1) v *= rq;
    if (!(v >= lo && v <= hi)) continue;
    int idx = (int)((v - lo) * norm);
    if (idx == nb) idx -= 1;
    if (v < s_edge[idx]) idx -= 1;
    else if (v >= s_edge[idx + 1] && idx != nb - 1) idx += 1;
    atomicAdd(&s_cnt[idx], 1u);
  }
  __syncthreads();
  if (threadIdx.x < nb && s_cnt[threadIdx.x]) atomicAdd(counts + threadIdx.x, (unsigned long long)s_cnt[threadIdx.x]);
}

// Strips, ring mode: wait until every rank has combined its report of launch `gen` into this rank's ring slot,
// publish it as gvec[rel] and take the verdict (k_strip_verify's logic).  One thread; spins on its own memory.
static __global__ void k_ring_verify(unsigned *ring, int gen, int world, float *gvec, int rel, int j, int was_upd, int was_spec,
                              int was_sel, float *gcarry, float *gmax_tab, int *bad_at, int *stop_at) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (*bad_at < rel) return;                        // nothing after a failed guess ran - and nothing was pushed
  // uniform lattice: the launch returned at once on every rank (or was a select-only launch at the stop)
  if (stop_at[0] >= 0 && (j > stop_at[0] || (j == stop_at[0] && !was_upd))) return;
  volatile unsigned *slot = ring + (gen & (RING_SLOTS - 1)) * RING_WORDS;
  const long long t0 = clock64();
  while (slot[3] < (unsigned)world) {
    if (clock64() - t0 > 20000000000ll) __trap();   // ~10 s: a rank is missing - fail loudly instead of hanging
    __nanosleep(200);
  }
  __threadfence_system();
  const float g_exact = __uint_as_float(slot[0]);
  const float anyD = slot[1] ? 1.0f : 0.0f, anyC = slot[2] ? 1.0f : 0.0f;
  gvec[4 * rel + 0] = g_exact; gvec[4 * rel + 1] = anyD; gvec[4 * rel + 2] = anyC;
  // slot gen+2 (= gen-2) was consumed two launches ago and no rank can push into it before it has seen this
  // rank's arrival for gen+1, which is enqueued after this kernel
  unsigned *nxt = ring + ((gen + 2) & (RING_SLOTS - 1)) * RING_WORDS;
  nxt[0] = 0u; nxt[1] = 0u; nxt[2] = 0u; nxt[3] = 0u;
  __threadfence_system();
  if (was_upd) {
    const float guess = gcarry[0];
    gmax_tab[rel] = g_exact;
    gcarry[0] = g_exact;
    if (was_spec == 2 || (was_spec && g_exact != guess)) { atomicMin(bad_at, rel); return; }
  }
  if (was_sel && (anyD == 0.0f || anyC == 0.0f) && stop_at[0] < 0) stop_at[0] = j + 1;
}

}  // namespace spgg
