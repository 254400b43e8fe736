// Strategy pair counts of a bit plane (spgg_pairs.cuh has the scheme; include/spgg.h the contract).  The only
// unit that holds these kernels: spgg_capi.cu reaches them through the launchers in spgg_pairs.cuh.
#include "spgg_pairs.cuh"
#include "spgg_clusters.cuh"   // ccl_word

#include <algorithm>

namespace spgg {

constexpr int PAIR_THREADS = 256;   // 8 warps
constexpr int PAIR_WARPS = PAIR_THREADS / 32;
constexpr int PR_RB = 32;           // k_pairs_rows: rows per staged band
constexpr int PR_DPT = 8;           // k_pairs_rows: offsets per thread
constexpr long long PAIR_CTAS = 148ll * 8;   // grid size the launches aim for: 8 CTAs for each of a B200's 148 SMs

static int pow2ceil(int x) {
  int p = 1;
  while (p < x) p <<= 1;
  return p;
}

__device__ __forceinline__ uint32_t pair_last_mask(int L) { return (L & 31) ? (1u << (L & 31)) - 1u : ~0u; }

// Axis 0: partner (i + d, j).  CTA = (32-word column band wb, offsets [d0, d0 + wd*PR_DPT), row segment); warp =
// (offset group wdi, row phase rs), lane = word column.  Shared memory: A = PR_RB rows of the band, B = the
// PR_RB + wd*PR_DPT - 1 rows that follow row r0 + d0, both with spare bits cleared.  Row r >= rows is read from
// the tail (row r - rows), which for a whole lattice is the plane itself.
__global__ void __launch_bounds__(PAIR_THREADS) k_pairs_rows(const uint32_t *S, int pitchW, int rows, int L,
                                                             const uint32_t *T, int tpitch, int max_d, int wd, int n_wb,
                                                             int n_dc, int n_seg, unsigned long long *out) {
  extern __shared__ uint32_t pair_sm[];
  __shared__ unsigned long long acc[PAIR_WARPS * PR_DPT][2];
  const int nW = (L + 31) >> 5, rsn = PAIR_WARPS / wd, dcn = wd * PR_DPT, nB = PR_RB + dcn - 1;
  const int wb = blockIdx.x % n_wb, dc = (blockIdx.x / n_wb) % n_dc, seg = blockIdx.x / (n_wb * n_dc);
  const int r_beg = (int)((long long)rows * seg / n_seg), r_end = (int)((long long)rows * (seg + 1) / n_seg);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wdi = warp % wd, rs = warp / wd;
  const int w = wb * 32 + lane, d0 = dc * dcn;
  const uint32_t m = w < nW ? (w == nW - 1 ? pair_last_mask(L) : ~0u) : 0u;
  const uint32_t *A = pair_sm, *B = pair_sm + PR_RB * 32;
  for (int t = threadIdx.x; t < PAIR_WARPS * PR_DPT * 2; t += PAIR_THREADS) acc[t >> 1][t & 1] = 0;
  unsigned cc[PR_DPT], df[PR_DPT];   // per lane at most 32 a row: exact for rows < 2^27
#pragma unroll
  for (int k = 0; k < PR_DPT; ++k) cc[k] = df[k] = 0;
  for (int r0 = r_beg; r0 < r_end; r0 += PR_RB) {
    __syncthreads();
    for (int e = threadIdx.x; e < (PR_RB + nB) * 32; e += PAIR_THREADS) {
      const int k = e >> 5, c = wb * 32 + (e & 31);
      uint32_t v = 0;
      if (c < nW) {
        if (k < PR_RB) {
          if (r0 + k < r_end) v = ccl_word(S, pitchW, L, nW, r0 + k, c, 1);
        } else {
          const long long r = (long long)r0 + d0 + (k - PR_RB);   // rows past rows + max_d serve no offset <= max_d
          if (r < rows) v = ccl_word(S, pitchW, L, nW, (int)r, c, 1);
          else if (r < (long long)rows + max_d) v = ccl_word(T, tpitch, L, nW, (int)(r - rows), c, 1);
        }
      }
      pair_sm[e] = v;
    }
    __syncthreads();
    const int nr = min(PR_RB, r_end - r0);
    for (int i = rs; i < nr; i += rsn) {
      const uint32_t a = A[i * 32 + lane], na = ~a & m;
      const uint32_t *b = B + (i + wdi * PR_DPT) * 32 + lane;
#pragma unroll
      for (int k = 0; k < PR_DPT; ++k) {
        const uint32_t bk = b[k * 32];
        cc[k] += __popc(na & ~bk);
        df[k] += __popc(a ^ bk);   // spare bits and columns past nW are 0 in both
      }
    }
  }
#pragma unroll
  for (int k = 0; k < PR_DPT; ++k) {
    const unsigned sc = __reduce_add_sync(0xffffffffu, cc[k]), sd = __reduce_add_sync(0xffffffffu, df[k]);
    if (lane == 0) {
      atomicAdd(&acc[wdi * PR_DPT + k][0], (unsigned long long)sc);
      atomicAdd(&acc[wdi * PR_DPT + k][1], (unsigned long long)sd);
    }
  }
  __syncthreads();
  for (int t = threadIdx.x; t < dcn * 2; t += PAIR_THREADS) {
    const int d = d0 + (t >> 1);
    if (d <= max_d && acc[t >> 1][t & 1]) atomicAdd(out + 2 * d + (t & 1), acc[t >> 1][t & 1]);
  }
}

// bits [s, s + 32) of the periodic bit stream of one row (column c in bit c & 31 of word c >> 5; bits past
// column L-1 are not part of it), 0 <= s < L; a lattice narrower than 32 columns repeats within one word
__device__ __forceinline__ uint32_t pair_stream_word(const uint32_t *row, int L, int nW, int s) {
  uint32_t v = 0;
  for (int got = 0; got < 32; s = 0) {   // after a piece that ends short of 32 bits the stream wraps to column 0
    const int w = s >> 5, n = min(32 - got, L - s);
    uint32_t bits = __funnelshift_r(row[w], w + 1 < nW ? row[w + 1] : 0u, s & 31);
    if (n < 32) bits &= (1u << n) - 1u;
    v |= bits << got;
    got += n;
  }
  return v;
}

// Axis 1: partner (i, j + d).  CTA = (gc groups of 32 offsets, row segment); warp = (offset group gw, row phase
// rs); lane = (offset dl of the group, word phase ws): a group of dw < 32 offsets (max_d < 31) spreads its
// words over 32 / dw lanes.  Shared memory: per row phase the row's periodic stream, imgW words.
__global__ void __launch_bounds__(PAIR_THREADS) k_pairs_cols(const uint32_t *S, int pitchW, int rows, int L, int max_d,
                                                             int gc, int dw, int n_dc, int n_seg,
                                                             unsigned long long *out) {
  extern __shared__ uint32_t pair_sm[];
  __shared__ unsigned long long acc[PAIR_THREADS][2];
  const int nW = (L + 31) >> 5, imgW = nW + (max_d >> 5) + 2, rsn = PAIR_WARPS / gc, ns = 32 / dw;
  const int dc = blockIdx.x % n_dc, seg = blockIdx.x / n_dc;
  const int r_beg = (int)((long long)rows * seg / n_seg), r_end = (int)((long long)rows * (seg + 1) / n_seg);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, gw = warp % gc, rs = warp / gc;
  const int dl = lane % dw, ws = lane / dw;
  const int d = (dc * gc + gw) * 32 + dl, q = d >> 5, sh = d & 31;
  const bool active = d <= max_d;
  const uint32_t lastm = pair_last_mask(L);
  for (int t = threadIdx.x; t < PAIR_THREADS * 2; t += PAIR_THREADS) acc[t >> 1][t & 1] = 0;
  unsigned long long ncc = 0, ndf = 0;
  for (int r0 = r_beg; r0 < r_end; r0 += rsn) {
    __syncthreads();
    for (int e = threadIdx.x; e < rsn * imgW; e += PAIR_THREADS) {
      const int k = e / imgW, j = e - k * imgW;
      pair_sm[e] = r0 + k < r_end ? pair_stream_word(S + (long long)(r0 + k) * pitchW, L, nW, (32 * j) % L) : 0u;
    }
    __syncthreads();
    if (active && r0 + rs < r_end) {
      const uint32_t *img = pair_sm + rs * imgW;
      unsigned cc = 0, df = 0;
      for (int w = ws; w < nW; w += ns) {
        const uint32_t a = img[w], b = __funnelshift_r(img[w + q], img[w + q + 1], sh);
        const uint32_t m = w == nW - 1 ? lastm : ~0u;
        cc += __popc(~(a | b) & m);
        df += __popc((a ^ b) & m);
      }
      ncc += cc;
      ndf += df;
    }
  }
  for (int o = dw; o < 32; o <<= 1) {
    ncc += __shfl_xor_sync(0xffffffffu, ncc, o);
    ndf += __shfl_xor_sync(0xffffffffu, ndf, o);
  }
  if (ws == 0 && active) {
    atomicAdd(&acc[gw * 32 + dl][0], ncc);
    atomicAdd(&acc[gw * 32 + dl][1], ndf);
  }
  __syncthreads();
  for (int t = threadIdx.x; t < gc * 32 * 2; t += PAIR_THREADS) {
    const int dd = dc * gc * 32 + (t >> 1);
    if (dd <= max_d && acc[t >> 1][t & 1]) atomicAdd(out + 2 * dd + (t & 1), acc[t >> 1][t & 1]);
  }
}

__global__ void k_pair_record(const uint32_t *S, int pitchW, int row0, int rows, int L, int max_d, int max_rows,
                              uint32_t *rec) {
  const int nW = (L + 31) >> 5, n = min(max_d, rows);
  const long long tot = (long long)max_rows * nW;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < tot; e += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(e / nW), c = (int)(e - (long long)r * nW);
    rec[PAIR_REC_HDR + e] = r < n ? ccl_word(S, pitchW, L, nW, r, c, 1) : 0u;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    rec[PAIR_H_MAGIC] = PAIR_REC_MAGIC; rec[PAIR_H_L] = L; rec[PAIR_H_ROW0] = row0; rec[PAIR_H_ROWS] = rows;
    rec[PAIR_H_MAXD] = max_d; rec[PAIR_H_MAXROWS] = max_rows; rec[PAIR_H_NROWS] = n; rec[PAIR_REC_HDR - 1] = 0;
  }
}

// ---------------------------------------------------------------- host side
static cudaError_t pair_smem(const void *k, size_t bytes) {
  return bytes > 48 * 1024 ? cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) : cudaSuccess;
}

static long long pair_segments(long long base, int rows, int per) {
  return std::max(1ll, std::min((PAIR_CTAS + base - 1) / base, (long long)(rows + per - 1) / per));
}

cudaError_t launch_pair_counts(const uint32_t *S, int pitchW, int rows, int L, const uint32_t *tail, int tail_pitch,
                               int max_d, unsigned long long *counts, int64_t *out) {
  const int nW = (L + 31) / 32, nd = max_d + 1;
  const size_t n_out = 2 * (size_t)nd * 2;
  cudaError_t e = cudaMemset(counts, 0, n_out * sizeof(unsigned long long));
  if (e != cudaSuccess) return e;
  {  // axis 0
    const int wd = std::min(PAIR_WARPS, pow2ceil((nd + PR_DPT - 1) / PR_DPT)), dcn = wd * PR_DPT;
    const int n_wb = (nW + 31) / 32, n_dc = (nd + dcn - 1) / dcn;
    const long long n_seg = pair_segments((long long)n_wb * n_dc, rows, PR_RB);
    const size_t smem = sizeof(uint32_t) * 32 * (2 * PR_RB + dcn - 1);
    k_pairs_rows<<<(unsigned)(n_wb * n_dc * n_seg), PAIR_THREADS, smem>>>(S, pitchW, rows, L, tail, tail_pitch, max_d,
                                                                          wd, n_wb, n_dc, (int)n_seg, counts);
  }
  {  // axis 1
    const int G = (max_d >> 5) + 1, dw = max_d < 32 ? pow2ceil(nd) : 32;
    const int gc = std::min(PAIR_WARPS, pow2ceil(G)), n_dc = (G + gc - 1) / gc, rsn = PAIR_WARPS / gc;
    const long long n_seg = pair_segments(n_dc, rows, rsn);
    const size_t smem = sizeof(uint32_t) * rsn * (size_t)(nW + (max_d >> 5) + 2);
    e = pair_smem((const void *)k_pairs_cols, smem);
    if (e != cudaSuccess) return e;
    k_pairs_cols<<<(unsigned)(n_dc * n_seg), PAIR_THREADS, smem>>>(S, pitchW, rows, L, max_d, gc, dw, n_dc, (int)n_seg,
                                                                    counts + 2 * nd);
  }
  e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpy(out, counts, n_out * sizeof(int64_t), cudaMemcpyDeviceToHost);
  return e;
}

cudaError_t launch_pair_record(const uint32_t *S, int pitchW, int row0, int rows, int L, int max_d, int max_rows,
                               void *dev_record) {
  const long long n = (long long)max_rows * ((L + 31) / 32);
  k_pair_record<<<(unsigned)std::max(1ll, std::min(148ll * 8, (n + 255) / 256)), 256>>>(S, pitchW, row0, rows, L, max_d,
                                                                                       max_rows, (uint32_t *)dev_record);
  return cudaGetLastError();
}

}  // namespace spgg
