// Value distributions (spgg_hist.cuh has the scheme; include/spgg.h the contract).  The only unit that holds these
// kernels: spgg_capi.cu reaches them through launch_value_ranges / launch_histograms.
#include "spgg_hist.cuh"
#include "spgg_kernels.cuh"   // ModeF32I8 / ModeF32F / ModeF64

#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

namespace spgg {

constexpr int HIST_BS = 512;   // threads per CTA
constexpr unsigned HIST_FULL = 0xffffffffu;
constexpr unsigned long long HIST_EMPTY_MIN = ~0ull, HIST_EMPTY_MAX = 0ull;   // keys no finite value maps to

// The device scratch of one call, all in 8-byte words: n_rep replicas, m channels, nb bins
struct HistBufs {
  unsigned long long *counts;   // [n_rep][m][2][nb]
  unsigned long long *codes;    // [n_rep][2][256]: int8 R per code + 128
  unsigned long long *policy;   // [n_rep][2][2]
  unsigned long long *mn, *mx;  // [n_rep][m][2]: hist_key of the extremes
  double *edges;                // [n_rep][m][nb + 1]
  double *rq;                   // [n_rep]
};

static HistBufs hist_bufs(void *scratch, int n_rep, int m, int nb, size_t *bytes) {
  HistBufs b;
  unsigned long long *w = reinterpret_cast<unsigned long long *>(scratch);
  b.counts = w; w += (size_t)n_rep * m * 2 * nb;
  b.codes = w; w += (size_t)n_rep * 512;
  b.policy = w; w += (size_t)n_rep * 4;
  b.mn = w; w += (size_t)n_rep * m * 2;
  b.mx = w; w += (size_t)n_rep * m * 2;
  b.edges = reinterpret_cast<double *>(w); w += (size_t)n_rep * m * (nb + 1);
  b.rq = reinterpret_cast<double *>(w); w += n_rep;
  *bytes = (size_t)(w - reinterpret_cast<unsigned long long *>(scratch)) * 8;
  return b;
}

size_t hist_scratch_bytes(int n_rep, int m, int n_bins) {
  size_t bytes;
  hist_bufs(nullptr, n_rep, m, std::max(n_bins, 1), &bytes);
  return bytes;
}

// Order-preserving map of an fp64 value to a 64-bit key (a < b  <=>  key(a) < key(b), -0.0 below +0.0)
__device__ __forceinline__ unsigned long long hist_key(double v) {
  const unsigned long long u = (unsigned long long)__double_as_longlong(v);
  return (u >> 63) ? ~u : u | 0x8000000000000000ull;
}
static double hist_unkey(unsigned long long k) {
  const unsigned long long u = (k >> 63) ? k & 0x7fffffffffffffffull : ~k;
  double v;
  memcpy(&v, &u, 8);
  return v;
}

// np.histogram's uniform-bin rule (the one k_r_histogram restates): -1 outside [lo, hi], else the float index
// (v - lo) * nb / (hi - lo) corrected by one against the edges e[0 .. nb], the last bin closed on the right.
// Explicit round-to-nearest operations: no FMA contraction.  The clamp only matters for ranges so narrow that
// nb / (hi - lo) overflows, where it keeps the edge reads in bounds.
__device__ __forceinline__ int hist_bin(double v, const double *e, int nb, double lo, double hi, double norm) {
  if (!(v >= lo && v <= hi)) return -1;
  int idx = (int)__dmul_rn(__dsub_rn(v, lo), norm);
  idx = min(max(idx, 0), nb - 1);
  if (v < __ldg(e + idx)) idx -= 1;
  else if (idx != nb - 1 && v >= __ldg(e + idx + 1)) idx += 1;
  return idx;
}

// One site's values: its class and the R and Q entries the kernel reads
template <class Md, bool RR, int NQ>
struct HistSite {
  typedef typename Md::Q QT;
  typedef typename Md::R RT;
  static constexpr int NV = NQ * (int)sizeof(QT) / 16;   // 16-byte loads per site of Q
  bool ok, coop;
  RT r;
  uint4 raw[NV > 0 ? NV : 1];
  __device__ __forceinline__ void load(const HistPlanes &p, const uint32_t *S, const RT *R, const QT *Q, bool ok_, int i,
                                       int col) {
    ok = ok_;
    coop = false;
    r = RT(0);
    if (!ok) return;
    coop = !((__ldg(S + (long long)i * p.pitchW + (col >> 5)) >> (col & 31)) & 1u);
    if constexpr (RR) r = __ldcs(R + (long long)i * p.pitchB + col);
    if constexpr (NQ > 0) {
      const uint4 *qp = reinterpret_cast<const uint4 *>(Q + ((long long)i * p.L + col) * NQ);
#pragma unroll
      for (int k = 0; k < NV; ++k) raw[k] = __ldcs(qp + k);
    }
  }
  __device__ __forceinline__ double q(int z) const { return (double)reinterpret_cast<const QT *>(raw)[z]; }
};

// The rows [ra, rb) of replica blockIdx.y that CTA blockIdx.x covers, walked HIST_BS sites at a time in row-major
// order; every lane of a warp takes the same number of steps (ok false past the end), so warp collectives see
// the whole warp.
struct HistWalk {
  long long n, e0;
  int L, i, col;
  __device__ __forceinline__ HistWalk(const HistPlanes &p, int rpc) {
    const int ra = blockIdx.x * rpc, rb = min(ra + rpc, p.rows);
    n = ra < rb ? (long long)(rb - ra) * p.L : 0;
    e0 = 0;
    L = p.L;
    i = ra + (int)threadIdx.x / L;
    col = (int)threadIdx.x % L;
  }
  __device__ __forceinline__ bool ok() const { return e0 + threadIdx.x < n; }
  __device__ __forceinline__ void next() {
    e0 += HIST_BS;
    col += HIST_BS;
    while (col >= L) { col -= L; ++i; }
  }
};

// Min and max of every (channel, class) of each replica.  Channels: R (if WR) as get_state returns it, then the NQ
// Q entries (if HQ).
template <class Md, bool WR, bool HQ, int NQ>
__global__ void __launch_bounds__(HIST_BS) k_hist_range(HistPlanes p, int rpc, int m, HistBufs b) {
  typedef typename Md::Q QT;
  typedef typename Md::R RT;
  constexpr int NQR = HQ ? NQ : 0, M = (WR ? 1 : 0) + NQR, C = 2 * M;
  __shared__ unsigned long long s_mm[2 * C];
  const int t = threadIdx.x, lane = t & 31, rl = blockIdx.y;
  if (t < C) { s_mm[t] = HIST_EMPTY_MIN; s_mm[C + t] = HIST_EMPTY_MAX; }
  __syncthreads();
  const double rq = b.rq[rl];
  const uint32_t *S = p.S + rl * p.bits_stride;
  const RT *R = reinterpret_cast<const RT *>(p.R) + rl * p.plane_stride;
  const QT *Q = reinterpret_cast<const QT *>(p.Q) + rl * p.q_stride;
  double mn[C], mx[C];
#pragma unroll
  for (int c = 0; c < C; ++c) { mn[c] = __longlong_as_double(0x7ff0000000000000ll); mx[c] = -mn[c]; }
  HistWalk w(p, rpc);
  HistSite<Md, WR, NQR> cur;
  cur.load(p, S, R, Q, w.ok(), w.i, w.col);
  while (w.e0 < w.n) {
    w.next();
    HistSite<Md, WR, NQR> nxt;   // the next site's loads are in flight while this one is reduced
    nxt.load(p, S, R, Q, w.ok(), w.i, w.col);
    if (cur.ok) {
#pragma unroll
      for (int ch = 0; ch < M; ++ch) {
        double v;
        if (WR && ch == 0) v = sizeof(RT) == 1 ? __dmul_rn((double)cur.r, rq) : (double)cur.r;
        else v = cur.q(ch - (WR ? 1 : 0));
        mn[ch] = fmin(mn[ch], v);
        mx[ch] = fmax(mx[ch], v);
        if (cur.coop) { mn[M + ch] = fmin(mn[M + ch], v); mx[M + ch] = fmax(mx[M + ch], v); }
      }
    }
    cur = nxt;
  }
#pragma unroll
  for (int c = 0; c < C; ++c) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mn[c] = fmin(mn[c], __shfl_xor_sync(HIST_FULL, mn[c], o));
      mx[c] = fmax(mx[c], __shfl_xor_sync(HIST_FULL, mx[c], o));
    }
    if (lane == 0) { atomicMin(&s_mm[c], hist_key(mn[c])); atomicMax(&s_mm[C + c], hist_key(mx[c])); }
  }
  __syncthreads();
  if (t < C) {
    // shared [k][ch] -> global [replica][ch][k]
    const int k = t / M, ch = t % M;
    const long long g = ((long long)rl * m + ch) * 2 + k;
    atomicMin(b.mn + g, s_mm[t]);
    atomicMax(b.mx + g, s_mm[C + t]);
  }
}

// Histograms of every (channel, class) and the greedy-policy counts of each replica.  Shared channels cb are the
// channels binned against edges: R (if WR and not int8-stored), then the NQ Q entries (if HQ); int8 R goes to
// the per-code counts instead.  POL: count the sites whose greedy action in state s is C, reading Q even
// without HQ.
template <class Md, bool WR, bool HQ, bool POL, int NQ>
__global__ void __launch_bounds__(HIST_BS) k_hist(HistPlanes p, int rpc, int nb, int m, HistBufs b) {
  typedef typename Md::Q QT;
  typedef typename Md::R RT;
  constexpr bool CODES = WR && sizeof(RT) == 1;
  constexpr int NBR = WR && !CODES ? 1 : 0, NCH = NBR + (HQ ? NQ : 0);
  constexpr int NQR = HQ || POL ? NQ : 0;
  extern __shared__ unsigned s_cnt[];   // [NCH][2][nb], then with CODES [2][256]
  __shared__ double s_par[NCH > 0 ? NCH : 1][3];   // lo, hi, nb / (hi - lo) of each shared channel
  __shared__ unsigned s_pol[4];
  unsigned *s_code = s_cnt + NCH * 2 * nb;
  const int t = threadIdx.x, lane = t & 31, rl = blockIdx.y;
  const double *E = b.edges + ((long long)rl * m + (CODES ? 1 : 0)) * (nb + 1);   // edge row of shared channel 0
  for (int k = t; k < NCH * 2 * nb + (CODES ? 512 : 0); k += HIST_BS) s_cnt[k] = 0u;
  if (t < NCH) {
    const double lo = E[t * (nb + 1)], hi = E[t * (nb + 1) + nb];
    s_par[t][0] = lo;
    s_par[t][1] = hi;
    s_par[t][2] = (double)nb / (hi - lo);
  }
  if (t < 4) s_pol[t] = 0u;
  __syncthreads();
  const uint32_t *S = p.S + rl * p.bits_stride;
  const RT *R = reinterpret_cast<const RT *>(p.R) + rl * p.plane_stride;
  const QT *Q = reinterpret_cast<const QT *>(p.Q) + rl * p.q_stride;
  // one (bin, class) group of the warp: its leader adds the group's size
  auto count = [&](int cb, double v, bool ok, bool coop) {
    const int bin = ok ? hist_bin(v, E + cb * (nb + 1), nb, s_par[cb][0], s_par[cb][1], s_par[cb][2]) : -1;
    const unsigned grp = __match_any_sync(HIST_FULL, bin * 2 + (int)coop);
    if (bin >= 0 && lane == __ffs(grp) - 1) {
      const unsigned c = __popc(grp);
      atomicAdd(&s_cnt[cb * 2 * nb + bin], c);
      if (coop) atomicAdd(&s_cnt[(cb * 2 + 1) * nb + bin], c);
    }
  };
  unsigned pol[4] = {0u, 0u, 0u, 0u};   // [class][state]
  HistWalk w(p, rpc);
  HistSite<Md, WR, NQR> cur;
  cur.load(p, S, R, Q, w.ok(), w.i, w.col);
  while (w.e0 < w.n) {
    w.next();
    HistSite<Md, WR, NQR> nxt;   // the next site's loads are in flight while this one is counted
    nxt.load(p, S, R, Q, w.ok(), w.i, w.col);
    if constexpr (CODES) {
      const int code = (int)cur.r + 128;
      const unsigned grp = __match_any_sync(HIST_FULL, cur.ok ? code * 2 + (int)cur.coop : -1);
      if (cur.ok && lane == __ffs(grp) - 1) {
        const unsigned c = __popc(grp);
        atomicAdd(&s_code[code], c);
        if (cur.coop) atomicAdd(&s_code[256 + code], c);
      }
    }
    if constexpr (NBR > 0) count(0, (double)cur.r, cur.ok, cur.coop);
    if constexpr (HQ) {
#pragma unroll
      for (int z = 0; z < NQ; ++z) count(NBR + z, cur.q(z), cur.ok, cur.coop);
    }
    if constexpr (POL) {
      if (cur.ok) {
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          // Q-bar[s, a]: Q, or (QA + QB) / 2 of Double Q-learning, in fp64; argmax's first maximum: C on a tie
          double a0 = cur.q(2 * s), a1 = cur.q(2 * s + 1);
          if (NQ == 8) {
            a0 = __dmul_rn(__dadd_rn(a0, cur.q(4 + 2 * s)), 0.5);
            a1 = __dmul_rn(__dadd_rn(a1, cur.q(5 + 2 * s)), 0.5);
          }
          const unsigned g = a0 >= a1;
          pol[s] += g;
          pol[2 + s] += g & (unsigned)cur.coop;
        }
      }
    }
    cur = nxt;
  }
  if constexpr (POL) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const unsigned v = __reduce_add_sync(HIST_FULL, pol[k]);
      if (lane == 0 && v) atomicAdd(&s_pol[k], v);
    }
  }
  __syncthreads();
  unsigned long long *G = b.counts + ((long long)rl * m + (CODES ? 1 : 0)) * 2 * nb;   // [cb][k][bin] is contiguous
  for (int k = t; k < NCH * 2 * nb; k += HIST_BS)
    if (s_cnt[k]) atomicAdd(G + k, (unsigned long long)s_cnt[k]);
  if constexpr (CODES) {
    for (int k = t; k < 512; k += HIST_BS)
      if (s_code[k]) atomicAdd(b.codes + (long long)rl * 512 + k, (unsigned long long)s_code[k]);
  }
  if (POL && t < 4 && s_pol[t]) atomicAdd(b.policy + rl * 4 + t, (unsigned long long)s_pol[t]);
}

// int8 R: each code's count goes to the bin of code * rq, by the same rule.  One thread per (replica, class, code).
__global__ void k_hist_codes(int n_rep, int nb, int m, HistBufs b) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= n_rep * 512) return;
  const int rl = x / 512, k = (x / 256) % 2, code = x % 256;
  const unsigned long long c = b.codes[x];
  if (!c) return;
  const double *E = b.edges + (long long)rl * m * (nb + 1);
  const double lo = E[0], hi = E[nb];
  const double v = __dmul_rn((double)(code - 128), b.rq[rl]);
  const int bin = hist_bin(v, E, nb, lo, hi, (double)nb / (hi - lo));
  if (bin >= 0) atomicAdd(b.counts + (((long long)rl * m) * 2 + k) * nb + bin, c);
}

// CTAs per replica: enough for `occ` resident CTAs on every SM over all replicas, at most one per row, and at
// most 2^31 sites per CTA (its shared counts are 32-bit)
template <class K>
static cudaError_t hist_grid(K kern, size_t smem, const HistPlanes &p, dim3 *grid, int *rpc) {
  int dev = 0, sms = 0, occ = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (e == cudaSuccess && smem > 48 * 1024)
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, HIST_BS, smem);
  if (e != cudaSuccess) return e;
  long long x = ((long long)std::max(occ, 1) * sms + p.n_rep - 1) / p.n_rep;
  x = std::max(x, ((long long)p.rows * p.L + (1ll << 31) - 1) >> 31);
  x = std::min(x, (long long)p.rows);
  *rpc = (int)((p.rows + x - 1) / x);
  *grid = dim3((unsigned)((p.rows + *rpc - 1) / *rpc), (unsigned)p.n_rep);
  return cudaSuccess;
}

template <class Md, bool WR, bool HQ, int NQ>
static cudaError_t launch_range(const HistPlanes &p, int m, const HistBufs &b) {
  auto kern = k_hist_range<Md, WR, HQ, NQ>;
  dim3 grid;
  int rpc;
  const cudaError_t e = hist_grid(kern, 0, p, &grid, &rpc);
  if (e != cudaSuccess) return e;
  kern<<<grid, HIST_BS>>>(p, rpc, m, b);
  return cudaGetLastError();
}

template <class Md>
cudaError_t launch_value_ranges(const HistPlanes &p, bool want_r, bool want_q, const double *rq, void *scratch,
                                double *minmax) {
  const int m = (want_r ? 1 : 0) + (want_q ? p.nq : 0);
  if (m == 0) return cudaSuccess;
  size_t bytes;
  const HistBufs b = hist_bufs(scratch, p.n_rep, m, 1, &bytes);
  const size_t nmm = (size_t)p.n_rep * m * 2;
  cudaError_t e = cudaMemset(b.mn, 0xff, nmm * 8);
  if (e == cudaSuccess) e = cudaMemset(b.mx, 0, nmm * 8);
  if (e == cudaSuccess) e = cudaMemcpy(b.rq, rq, p.n_rep * sizeof(double), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return e;
  if (!want_q) e = launch_range<Md, true, false, 4>(p, m, b);
  else if (p.nq == 4) e = want_r ? launch_range<Md, true, true, 4>(p, m, b) : launch_range<Md, false, true, 4>(p, m, b);
  else e = want_r ? launch_range<Md, true, true, 8>(p, m, b) : launch_range<Md, false, true, 8>(p, m, b);
  if (e != cudaSuccess) return e;
  std::vector<unsigned long long> k(2 * nmm);
  e = cudaMemcpy(k.data(), b.mn, 2 * nmm * 8, cudaMemcpyDeviceToHost);   // mn and mx are adjacent
  if (e != cudaSuccess) return e;
  for (size_t i = 0; i < nmm; ++i) {
    const unsigned long long a = k[i], z = k[nmm + i];
    minmax[2 * i] = a == HIST_EMPTY_MIN ? INFINITY : hist_unkey(a);
    minmax[2 * i + 1] = z == HIST_EMPTY_MAX ? -INFINITY : hist_unkey(z);
  }
  return cudaSuccess;
}

template <class Md, bool WR, bool HQ, bool POL, int NQ>
static cudaError_t launch_hist(const HistPlanes &p, int nb, int m, const HistBufs &b) {
  auto kern = k_hist<Md, WR, HQ, POL, NQ>;
  constexpr int nch = (WR && sizeof(typename Md::R) != 1 ? 1 : 0) + (HQ ? NQ : 0);
  const size_t smem = ((size_t)nch * 2 * nb + (WR && sizeof(typename Md::R) == 1 ? 512 : 0)) * sizeof(unsigned);
  dim3 grid;
  int rpc;
  const cudaError_t e = hist_grid(kern, smem, p, &grid, &rpc);
  if (e != cudaSuccess) return e;
  kern<<<grid, HIST_BS, smem>>>(p, rpc, nb, m, b);
  return cudaGetLastError();
}

template <class Md, bool POL, int NQ>
static cudaError_t launch_hist_fields(const HistPlanes &p, bool want_r, bool want_q, int nb, int m,
                                      const HistBufs &b) {
  if (want_r) return want_q ? launch_hist<Md, true, true, POL, NQ>(p, nb, m, b) : launch_hist<Md, true, false, POL, NQ>(p, nb, m, b);
  return want_q ? launch_hist<Md, false, true, POL, NQ>(p, nb, m, b) : launch_hist<Md, false, false, POL, NQ>(p, nb, m, b);
}

template <class Md>
cudaError_t launch_histograms(const HistPlanes &p, bool want_r, bool want_q, int n_bins, const double *edges,
                              const double *rq, void *scratch, int64_t *counts, int64_t *policy) {
  const int m = (want_r ? 1 : 0) + (want_q ? p.nq : 0);
  if (m == 0 && !policy) return cudaSuccess;
  size_t bytes;
  const HistBufs b = hist_bufs(scratch, p.n_rep, m, n_bins, &bytes);
  // counts, codes and policy are adjacent
  cudaError_t e = cudaMemset(b.counts, 0, ((size_t)p.n_rep * (m * 2 * n_bins + 512 + 4)) * 8);
  if (e == cudaSuccess && m > 0)
    e = cudaMemcpy(b.edges, edges, (size_t)p.n_rep * m * (n_bins + 1) * sizeof(double), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(b.rq, rq, p.n_rep * sizeof(double), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return e;
  if (policy) e = p.nq == 4 ? launch_hist_fields<Md, true, 4>(p, want_r, want_q, n_bins, m, b)
                            : launch_hist_fields<Md, true, 8>(p, want_r, want_q, n_bins, m, b);
  else e = p.nq == 4 ? launch_hist_fields<Md, false, 4>(p, want_r, want_q, n_bins, m, b)
                     : launch_hist_fields<Md, false, 8>(p, want_r, want_q, n_bins, m, b);
  if (e == cudaSuccess && want_r && sizeof(typename Md::R) == 1) {
    k_hist_codes<<<(p.n_rep * 512 + 255) / 256, 256>>>(p.n_rep, n_bins, m, b);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess && m > 0)
    e = cudaMemcpy(counts, b.counts, (size_t)p.n_rep * m * 2 * n_bins * 8, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && policy) e = cudaMemcpy(policy, b.policy, (size_t)p.n_rep * 4 * 8, cudaMemcpyDeviceToHost);
  return e;
}

#define SPGG_HIST_INST(Md)                                                                                             \
  template cudaError_t launch_value_ranges<Md>(const HistPlanes &, bool, bool, const double *, void *, double *);   \
  template cudaError_t launch_histograms<Md>(const HistPlanes &, bool, bool, int, const double *, const double *,    \
                                             void *, int64_t *, int64_t *);
SPGG_HIST_INST(ModeF32I8)
SPGG_HIST_INST(ModeF32F)
SPGG_HIST_INST(ModeF64)

}  // namespace spgg
