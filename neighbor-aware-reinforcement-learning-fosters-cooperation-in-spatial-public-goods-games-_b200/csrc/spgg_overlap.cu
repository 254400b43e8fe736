// State overlaps (spgg_overlap.cuh has the scheme; include/spgg.h the contract).  The only unit that holds these
// kernels: spgg_capi.cu reaches them through launch_overlap.
#include "spgg_overlap.cuh"
#include "spgg_kernels.cuh"   // ModeF32I8 / ModeF32F / ModeF64

#include <algorithm>
#include <cstring>
#include <vector>

namespace spgg {

constexpr int OV_BS = 256, OV_NW = OV_BS / 32;   // threads and warps per CTA
constexpr unsigned OV_FULL = 0xffffffffu;
constexpr int OV_MAX_TILES = 4096;        // tiles per replica at most ...
constexpr int OV_MIN_TILE_SITES = 4096;   // ... and at least this many sites per tile (unless the lattice is smaller)

// The device scratch of one call, all in 8-byte words: n_rep replicas, m channels, T tiles per replica
struct OvBufs {
  unsigned long long *counts;    // [n_rep][2][2]: strategy then, strategy now
  unsigned long long *changed;   // [n_rep][m]
  unsigned long long *mx;        // [n_rep][m]: bits of max |d| (>= +0.0, so integer order is numeric order)
  double *sums;                  // [n_rep][m][2]: sum |d|, sum d^2
  double *part;                  // [n_rep][m][2][T]: the tiles' partials of sums
  double *rq;                    // [2][n_rep]: int8 quanta, live then snapshot
};

static OvBufs ov_bufs(void *scratch, int T, int n_rep, int m, size_t *bytes) {
  OvBufs b;
  unsigned long long *w = reinterpret_cast<unsigned long long *>(scratch);
  b.counts = w; w += (size_t)n_rep * 4;
  b.changed = w; w += (size_t)n_rep * m;
  b.mx = w; w += (size_t)n_rep * m;
  b.sums = reinterpret_cast<double *>(w); w += (size_t)n_rep * m * 2;
  b.part = reinterpret_cast<double *>(w); w += (size_t)n_rep * m * 2 * T;
  b.rq = reinterpret_cast<double *>(w); w += (size_t)n_rep * 2;
  *bytes = (size_t)(w - reinterpret_cast<unsigned long long *>(scratch)) * 8;
  return b;
}

int overlap_rows_per_tile(int L, int rows) {
  const int rpc = std::max((rows + OV_MAX_TILES - 1) / OV_MAX_TILES, (OV_MIN_TILE_SITES + L - 1) / L);
  return std::min(rpc, rows);
}

size_t overlap_scratch_bytes(int L, int rows, int n_rep, int m) {
  const int rpc = overlap_rows_per_tile(L, rows);
  size_t bytes;
  ov_bufs(nullptr, (rows + rpc - 1) / rpc, n_rep, m, &bytes);
  return bytes;
}

// One channel's running results over a thread's values: changed count, max |d|, sum |d|, sum d^2, d = now - then
// in fp64 with explicit round-to-nearest operations (no FMA contraction)
struct OvAcc {
  unsigned n;
  double mx, s1, s2;
  __device__ __forceinline__ void init() { n = 0u; mx = 0.0; s1 = 0.0; s2 = 0.0; }
  __device__ __forceinline__ void add(double now, double then) {
    n += now != then ? 1u : 0u;
    const double d = __dsub_rn(now, then), a = fabs(d);
    mx = fmax(mx, a);
    s1 = __dadd_rn(s1, a);
    s2 = __dadd_rn(s2, __dmul_rn(d, d));
  }
};

// R as spgg_get_state returns it: int8 units x quantum, or the stored float / double
template <class RT>
__device__ __forceinline__ double ov_r(RT x, double rq) {
  if constexpr (sizeof(RT) == 1) return __dmul_rn((double)x, rq);
  else return (double)x;
}

// Joint strategy counts and, per channel (R if WR, then the NQR Q entries), the changed counts, the max |d| and
// the tile's partial sums of |d| and d^2 of replica blockIdx.y over the rows of tile blockIdx.x
template <class Md, bool WR, int NQR>
__global__ void __launch_bounds__(OV_BS) k_overlap(OvPlanes p, int rpc, int T, OvBufs b) {
  typedef typename Md::Q QT;
  typedef typename Md::R RT;
  constexpr int M = (WR ? 1 : 0) + NQR, MS = M > 0 ? M : 1;
  __shared__ unsigned long long s_cnt[4], s_chg[MS], s_mx[MS];
  __shared__ double s_sum[OV_NW][MS][2];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5, rl = blockIdx.y, tile = blockIdx.x;
  if (t < 4) s_cnt[t] = 0ull;
  if (t < M) { s_chg[t] = 0ull; s_mx[t] = 0ull; }
  __syncthreads();
  const int ra = tile * rpc, nr = min(rpc, p.rows - ra);

  // strategies: the tile's bit words, spare bits past column L - 1 masked off
  {
    const uint32_t *Sn = p.S[0] + rl * p.bits_stride + (long long)ra * p.pitchW;
    const uint32_t *St = p.S[1] + rl * p.bits_stride + (long long)ra * p.pitchW;
    const int nW = (p.L + 31) >> 5, nk = nr * nW;
    const uint32_t last = (p.L & 31) ? (1u << (p.L & 31)) - 1u : ~0u;
    unsigned c[4] = {0u, 0u, 0u, 0u};   // [then][now], 0 = C, 1 = D
    for (int k = t; k < nk; k += OV_BS) {
      const int i = k / nW, w = k - i * nW;
      const uint32_t msk = w == nW - 1 ? last : ~0u;
      const uint32_t a = __ldcs(St + (long long)i * p.pitchW + w), z = __ldcs(Sn + (long long)i * p.pitchW + w);
      c[0] += __popc(~a & ~z & msk);
      c[1] += __popc(~a & z & msk);
      c[2] += __popc(a & ~z & msk);
      c[3] += __popc(a & z & msk);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const unsigned v = __reduce_add_sync(OV_FULL, c[k]);
      if (lane == 0 && v) atomicAdd(&s_cnt[k], (unsigned long long)v);
    }
  }

  OvAcc acc[MS];
#pragma unroll
  for (int ch = 0; ch < MS; ++ch) acc[ch].init();

  // R: the tile's rows in 16-byte chunks (rows start 16-byte aligned; a chunk past column L - 1 stays inside the
  // row's padding and its extra elements are not counted)
  if constexpr (WR) {
    constexpr int VR = 16 / (int)sizeof(RT);
    const RT *Rn = reinterpret_cast<const RT *>(p.R[0]) + rl * p.plane_stride + (long long)ra * p.pitchB;
    const RT *Rt = reinterpret_cast<const RT *>(p.R[1]) + rl * p.plane_stride + (long long)ra * p.pitchB;
    const double qn = b.rq[rl], qt = b.rq[p.n_rep + rl];
    const int nc = (p.L + VR - 1) / VR, nk = nr * nc;
    for (int k = t; k < nk; k += OV_BS) {
      const int i = k / nc, c0 = (k - i * nc) * VR;
      const uint4 un = __ldcs(reinterpret_cast<const uint4 *>(Rn + (long long)i * p.pitchB + c0));
      const uint4 ut = __ldcs(reinterpret_cast<const uint4 *>(Rt + (long long)i * p.pitchB + c0));
      const RT *vn = reinterpret_cast<const RT *>(&un), *vt = reinterpret_cast<const RT *>(&ut);
#pragma unroll
      for (int v = 0; v < VR; ++v)
        if (c0 + v < p.L) acc[0].add(ov_r(vn[v], qn), ov_r(vt[v], qt));
    }
  }

  // Q: the tile's sites as one flat run, U sites per thread per step, all their 16-byte loads issued first
  if constexpr (NQR > 0) {
    constexpr int NV = NQR * (int)sizeof(QT) / 16;   // 16-byte loads per site
    constexpr int U = NV >= 4 ? 1 : 4 / NV;
    constexpr int C0 = WR ? 1 : 0;
    const uint4 *Qn = reinterpret_cast<const uint4 *>(reinterpret_cast<const QT *>(p.Q[0]) + rl * p.q_stride);
    const uint4 *Qt = reinterpret_cast<const uint4 *>(reinterpret_cast<const QT *>(p.Q[1]) + rl * p.q_stride);
    const long long s0 = (long long)ra * p.L, s1 = s0 + (long long)nr * p.L;
    for (long long e = s0 + t; e < s1; e += (long long)OV_BS * U) {
      uint4 rn[U][NV], rt[U][NV];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long s = e + (long long)u * OV_BS;
        if (s < s1) {
#pragma unroll
          for (int k = 0; k < NV; ++k) {
            rn[u][k] = __ldcs(Qn + s * NV + k);
            rt[u][k] = __ldcs(Qt + s * NV + k);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (e + (long long)u * OV_BS < s1) {
          const QT *vn = reinterpret_cast<const QT *>(rn[u]), *vt = reinterpret_cast<const QT *>(rt[u]);
#pragma unroll
          for (int z = 0; z < NQR; ++z) acc[C0 + z].add((double)vn[z], (double)vt[z]);
        }
      }
    }
  }

  // per channel: counts and maxima by integer atomics, sums by a fixed butterfly, then the warps in order
#pragma unroll
  for (int ch = 0; ch < M; ++ch) {
    const unsigned n = __reduce_add_sync(OV_FULL, acc[ch].n);
    double mx = acc[ch].mx, s1 = acc[ch].s1, s2 = acc[ch].s2;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mx = fmax(mx, __shfl_xor_sync(OV_FULL, mx, o));
      s1 = __dadd_rn(s1, __shfl_xor_sync(OV_FULL, s1, o));
      s2 = __dadd_rn(s2, __shfl_xor_sync(OV_FULL, s2, o));
    }
    if (lane == 0) {
      if (n) atomicAdd(&s_chg[ch], (unsigned long long)n);
      atomicMax(&s_mx[ch], (unsigned long long)__double_as_longlong(mx));
      s_sum[warp][ch][0] = s1;
      s_sum[warp][ch][1] = s2;
    }
  }
  __syncthreads();
  if (t < 4 && s_cnt[t]) atomicAdd(b.counts + rl * 4 + t, s_cnt[t]);
  if (t < M) {
    if (s_chg[t]) atomicAdd(b.changed + rl * M + t, s_chg[t]);
    atomicMax(b.mx + rl * M + t, s_mx[t]);
  }
  if (t < 2 * M) {
    const int ch = t >> 1, k = t & 1;
    double s = s_sum[0][ch][k];
#pragma unroll
    for (int w = 1; w < OV_NW; ++w) s = __dadd_rn(s, s_sum[w][ch][k]);
    b.part[(((long long)rl * M + ch) * 2 + k) * T + tile] = s;
  }
}

// sums[row] = the T partials of row added in a fixed order: lane l the tiles l, l + 32, ..., then a butterfly.
// One warp per row.
__global__ void k_overlap_fold(int n_rows, int T, const double *part, double *sums) {
  const int row = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (row >= n_rows) return;   // whole warps: blockDim is a multiple of 32
  double s = 0.0;
  for (int k = lane; k < T; k += 32) s = __dadd_rn(s, part[(long long)row * T + k]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s = __dadd_rn(s, __shfl_xor_sync(OV_FULL, s, o));
  if (lane == 0) sums[row] = s;
}

template <class Md, bool WR, int NQR>
static cudaError_t launch_ov(const OvPlanes &p, int rpc, int T, const OvBufs &b) {
  k_overlap<Md, WR, NQR><<<dim3((unsigned)T, (unsigned)p.n_rep), OV_BS>>>(p, rpc, T, b);
  return cudaGetLastError();
}

template <class Md, int NQR>
static cudaError_t launch_ov_r(const OvPlanes &p, bool want_r, int rpc, int T, const OvBufs &b) {
  return want_r ? launch_ov<Md, true, NQR>(p, rpc, T, b) : launch_ov<Md, false, NQR>(p, rpc, T, b);
}

template <class Md>
cudaError_t launch_overlap(const OvPlanes &p, bool want_r, bool want_q, const double *rq, void *scratch,
                           int64_t *counts, int64_t *changed, double *diffs) {
  const int m = (want_r ? 1 : 0) + (want_q ? p.nq : 0);
  const int rpc = overlap_rows_per_tile(p.L, p.rows), T = (p.rows + rpc - 1) / rpc;
  size_t bytes;
  const OvBufs b = ov_bufs(scratch, T, p.n_rep, m, &bytes);
  // counts, changed and mx are adjacent, and sums follows them
  const size_t n_int = (size_t)p.n_rep * (4 + 2 * m), n_out = n_int + (size_t)p.n_rep * m * 2;
  cudaError_t e = cudaMemset(b.counts, 0, n_int * 8);
  if (e == cudaSuccess) e = cudaMemcpy(b.rq, rq, 2 * p.n_rep * sizeof(double), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return e;
  if (!want_q) e = launch_ov_r<Md, 0>(p, want_r, rpc, T, b);
  else if (p.nq == 4) e = launch_ov_r<Md, 4>(p, want_r, rpc, T, b);
  else e = launch_ov_r<Md, 8>(p, want_r, rpc, T, b);
  if (e == cudaSuccess && m > 0) {
    const int n_rows = p.n_rep * m * 2;
    k_overlap_fold<<<(n_rows * 32 + 255) / 256, 256>>>(n_rows, T, b.part, b.sums);
    e = cudaGetLastError();
  }
  std::vector<unsigned long long> w(n_out);
  if (e == cudaSuccess) e = cudaMemcpy(w.data(), b.counts, n_out * 8, cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) return e;
  const unsigned long long *cnt = w.data(), *chg = cnt + (size_t)p.n_rep * 4, *mx = chg + (size_t)p.n_rep * m;
  const unsigned long long *sums = mx + (size_t)p.n_rep * m;
  for (size_t i = 0; i < (size_t)p.n_rep * 4; ++i) counts[i] = (int64_t)cnt[i];
  for (size_t i = 0; i < (size_t)p.n_rep * m; ++i) {
    changed[i] = (int64_t)chg[i];
    memcpy(diffs + 3 * i, mx + i, 8);
    memcpy(diffs + 3 * i + 1, sums + 2 * i, 16);
  }
  return cudaSuccess;
}

#define SPGG_OVERLAP_INST(Md)                                                                                      \
  template cudaError_t launch_overlap<Md>(const OvPlanes &, bool, bool, const double *, void *, int64_t *,         \
                                          int64_t *, double *);
SPGG_OVERLAP_INST(ModeF32I8)
SPGG_OVERLAP_INST(ModeF32F)
SPGG_OVERLAP_INST(ModeF64)

}  // namespace spgg
