// Block-averaged fields of one replica (spgg_blocks.cuh has the scheme; include/spgg.h the contract).  The only
// unit that holds these kernels: spgg_capi.cu reaches them through launch_block_fields.
#include "spgg_blocks.cuh"
#include "spgg_kernels.cuh"    // ModeF32I8 / ModeF32F / ModeF64
#include "spgg_clusters.cuh"   // ccl_word

#include <algorithm>
#include <vector>

namespace spgg {

constexpr int BLK_CT = 256;   // k_block_count: threads per CTA, one bit word each
constexpr unsigned BLK_FULL = 0xffffffffu;

// Row tile y: block rows [Ib, Ie) of the output, and for b >= BLK_TH the chunk rc of each
struct BlkRowTile {
  int Ib, Ie, rc;
};
__device__ __forceinline__ BlkRowTile blk_row_tile(const BlockGeom &q, int y) {
  BlkRowTile r;
  r.rc = y % q.nrc;
  r.Ib = q.I0 + (y / q.nrc) * q.kr;
  r.Ie = min(r.Ib + q.kr, q.I0 + q.nI);
  return r;
}

// the strip's rows [lo, hi) (local indices) of chunk rc of block row I
__device__ __forceinline__ void blk_rows(const BlockGeom &q, int I, int rc, int &lo, int &hi) {
  const int g0 = I * q.b + rc * BLK_TH;
  const int g1 = min(I * q.b + min((rc + 1) * BLK_TH, q.b), q.L);
  lo = max(g0, q.row0) - q.row0;
  hi = min(g1, q.row0 + q.rows) - q.row0;
}

// n_C per output block.  Thread = bit word w of the rows of one row tile; the word's columns fall in blocks
// J0 .. J0 + nseg - 1 (nseg <= MAXSEG), whose column masks are fixed per thread.  Per block row the lanes of a
// warp that share a block add their counts (__reduce_add_sync) and one of them does the 64-bit atomicAdd.
template <int MAXSEG>
__global__ void __launch_bounds__(BLK_CT) k_block_count(BlockGeom q, const uint32_t *S, int pitchW,
                                                        unsigned long long *nc) {
  const int nW = (q.L + 31) >> 5;
  const int w = blockIdx.x * BLK_CT + threadIdx.x;
  const bool ok = w < nW;
  const int c0 = w * 32, c1 = ok ? min(c0 + 32, q.L) : c0 + 1;
  const int J0 = c0 / q.b, nseg = ok ? (c1 - 1) / q.b - J0 + 1 : 0;
  uint32_t mk[MAXSEG];
#pragma unroll
  for (int s = 0; s < MAXSEG; ++s) {
    mk[s] = 0u;
    if (s < nseg) {   // columns [a, e) of the word lie in block J0 + s
      const int a = max((J0 + s) * q.b, c0) - c0, e = min((J0 + s + 1) * q.b, c1) - c0;
      mk[s] = (e >= 32 ? ~0u : (1u << e) - 1u) & ~((1u << a) - 1u);
    }
  }
  const BlkRowTile rt = blk_row_tile(q, blockIdx.y);
  for (int I = rt.Ib; I < rt.Ie; ++I) {
    int lo, hi;
    blk_rows(q, I, rt.rc, lo, hi);
    unsigned acc[MAXSEG];
#pragma unroll
    for (int s = 0; s < MAXSEG; ++s) acc[s] = 0u;
    if (ok) {
#pragma unroll 4
      for (int r = lo; r < hi; ++r) {
        const uint32_t c = ccl_word(S, pitchW, q.L, nW, r, w, 0);   // bit 1 = cooperator, spare bits cleared
#pragma unroll
        for (int s = 0; s < MAXSEG; ++s) acc[s] += __popc(c & mk[s]);
      }
    }
#pragma unroll
    for (int s = 0; s < MAXSEG; ++s) {
      const long long key = s < nseg ? (long long)(I - q.I0) * q.B + J0 + s : -1;
      const unsigned grp = __match_any_sync(BLK_FULL, key);
      const unsigned sum = __reduce_add_sync(grp, acc[s]);
      if (key >= 0 && sum && (threadIdx.x & 31) == __ffs(grp) - 1) atomicAdd(nc + key, (unsigned long long)sum);
    }
  }
}

// fp64 sums of one tile (spgg_blocks.cuh).  Channels c = k * M + ch: k 0 all sites, k 1 cooperators; ch 0 R (if
// WR), then the NQ Q entries.  out: [block][piece][C] with npc pieces per block (npc == 1: the result itself).
template <class Md, bool WR, int NQ>
__global__ void __launch_bounds__(BLK_TW) k_block_sums(BlockGeom q, const uint32_t *S, int pitchW, const void *Rd,
                                                       int pitchB, const void *Qd, double rq, double *out) {
  typedef typename Md::Q QT;
  typedef typename Md::R RT;
  constexpr int M = (WR ? 1 : 0) + NQ, C = 2 * M;
  constexpr int NV = NQ * (int)sizeof(QT) / 16;   // 16-byte loads per site of Q
  __shared__ double sh[C * BLK_TW];
  const RT *R = reinterpret_cast<const RT *>(Rd);
  const QT *Q = reinterpret_cast<const QT *>(Qd);
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int cs = blockIdx.x % q.ncs, Jb = (int)(blockIdx.x / q.ncs) * q.kc;
  const int c0 = Jb * q.b + cs * BLK_TW, c1 = min(Jb * q.b + min((cs + 1) * BLK_TW, q.kc * q.b), q.L);
  if (c0 >= c1) return;   // a column piece past column L-1 of the last block (its piece stays zero)
  const int col = c0 + t;
  const bool ok = col < c1;
  const BlkRowTile rt = blk_row_tile(q, blockIdx.y);
  const int npc = q.nrc * q.ncs, p = rt.rc * q.ncs + cs;
  // the segmented tree: lanes [lane, send) of this warp hold columns of the lane's block; a head lane starts a
  // block within its warp and holds the warp's partial of that block afterwards
  const int send = ok ? min(min((col / q.b + 1) * q.b, c1) - (c0 + warp * 32), 32) : 32;
  const bool head = ok && (lane == 0 || col % q.b == 0);
  const int Jf = c0 / q.b, nseg = (c1 - 1) / q.b - Jf + 1;
  const uint32_t *Sc = S + (col >> 5);
  const RT *Rc = R + col;
  const uint4 *Qc = reinterpret_cast<const uint4 *>(Q + (long long)col * NQ);
  const long long qpitch = (long long)q.L * NQ * (long long)sizeof(QT) / 16;   // uint4 per Q row
  for (int I = rt.Ib; I < rt.Ie; ++I) {
    int lo, hi;
    blk_rows(q, I, rt.rc, lo, hi);
    double acc[C];
#pragma unroll
    for (int c = 0; c < C; ++c) acc[c] = 0.0;
    if (ok) {
#pragma unroll 4
      for (int r = lo; r < hi; ++r) {
        const bool coop = !((__ldg(Sc + (long long)r * pitchW) >> (col & 31)) & 1u);
        if constexpr (WR) {
          const double v = (double)__ldcs(Rc + (long long)r * pitchB);
          acc[0] += v;
          if (coop) acc[M] += v;
        }
        if constexpr (NQ > 0) {
          uint4 raw[NV];
#pragma unroll
          for (int k = 0; k < NV; ++k) raw[k] = __ldcs(Qc + r * qpitch + k);
          const QT *qv = reinterpret_cast<const QT *>(raw);
#pragma unroll
          for (int z = 0; z < NQ; ++z) {
            const double v = (double)qv[z];
            acc[M - NQ + z] += v;
            if (coop) acc[2 * M - NQ + z] += v;
          }
        }
      }
    }
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const double v = __shfl_down_sync(BLK_FULL, acc[c], o);
        if (lane + o < send) acc[c] += v;
      }
    }
    if (head) {
#pragma unroll
      for (int c = 0; c < C; ++c) sh[c * BLK_TW + t] = acc[c];
    }
    __syncthreads();
    // per (block, channel): the head partials of the warps the block covers, in column order
    for (int i = t; i < nseg * C; i += BLK_TW) {
      const int s = i / C, c = i % C, J = Jf + s;
      const int a = max(J * q.b, c0) - c0, e = min((J + 1) * q.b, c1) - c0;
      double v = sh[c * BLK_TW + a];
      for (int u = (a & ~31) + 32; u < e; u += 32) v += sh[c * BLK_TW + u];
      if (WR && sizeof(RT) == 1 && c % M == 0) v *= rq;   // int8 units -> the reference's value (exact: rq = 2^-k)
      out[(((long long)(I - q.I0) * q.B + J) * npc + p) * C + c] = v;
    }
    __syncthreads();
  }
}

// the pieces of every block in piece order: out[blk][c] = sum over p of pieces[blk][p][c]
__global__ void k_block_pieces(const double *pieces, long long n, int npc, int C, double *out) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long blk = i / C;
    const int c = (int)(i % C);
    const double *pp = pieces + blk * npc * C + c;
    double v = pp[0];
    for (int k = 1; k < npc; ++k) v += pp[(long long)k * C];
    out[i] = v;
  }
}

static long long blk_n(const BlockGeom &q) { return (long long)q.nI * q.B; }

size_t block_scratch_bytes(const BlockGeom &q, int m) {
  const int npc = q.nrc * q.ncs;
  size_t n = (size_t)blk_n(q) * sizeof(unsigned long long);
  if (m > 0) n += (size_t)blk_n(q) * 2 * m * sizeof(double) * (npc > 1 ? 1 + npc : 1);
  return n;
}

template <class Md, bool WR, int NQ>
static void launch_sums(const BlockGeom &q, const uint32_t *S, int pitchW, const void *R, int pitchB, const void *Q,
                        double rq, double *out) {
  k_block_sums<Md, WR, NQ><<<dim3((unsigned)q.n_ct, (unsigned)q.n_rt), BLK_TW>>>(q, S, pitchW, R, pitchB, Q, rq, out);
}

template <class Md>
cudaError_t launch_block_fields(const BlockGeom &q, int pitchW, int pitchB, const uint32_t *S, const void *R,
                                const void *Q, double rq, int nq, bool want_r, bool want_q, void *scratch,
                                int64_t *counts, double *sums) {
  const long long nb = blk_n(q);
  const int m = (want_r ? 1 : 0) + (want_q ? nq : 0), C = 2 * m, npc = q.nrc * q.ncs;
  unsigned long long *nc = reinterpret_cast<unsigned long long *>(scratch);
  double *res = reinterpret_cast<double *>(nc + nb);
  double *pieces = res + (npc > 1 ? nb * C : 0);   // npc == 1: the tiles write the result itself
  cudaError_t e = cudaMemset(nc, 0, nb * sizeof(unsigned long long));
  if (e == cudaSuccess && m > 0 && npc > 1) e = cudaMemset(pieces, 0, (size_t)nb * npc * C * sizeof(double));
  if (e != cudaSuccess) return e;
  const dim3 gc((unsigned)(((q.L + 31) / 32 + BLK_CT - 1) / BLK_CT), (unsigned)q.n_rt);
  if (q.b >= 32) k_block_count<2><<<gc, BLK_CT>>>(q, S, pitchW, nc);
  else if (q.b >= 5) k_block_count<8><<<gc, BLK_CT>>>(q, S, pitchW, nc);   // <= floor(30 / b) + 2 blocks per word
  else k_block_count<32><<<gc, BLK_CT>>>(q, S, pitchW, nc);
  if (m > 0) {
    if (!want_q) launch_sums<Md, true, 0>(q, S, pitchW, R, pitchB, Q, rq, pieces);
    else if (nq == 4) want_r ? launch_sums<Md, true, 4>(q, S, pitchW, R, pitchB, Q, rq, pieces)
                             : launch_sums<Md, false, 4>(q, S, pitchW, R, pitchB, Q, rq, pieces);
    else want_r ? launch_sums<Md, true, 8>(q, S, pitchW, R, pitchB, Q, rq, pieces)
                : launch_sums<Md, false, 8>(q, S, pitchW, R, pitchB, Q, rq, pieces);
    if (npc > 1)
      k_block_pieces<<<(unsigned)std::max(1ll, std::min(148ll * 8, (nb * C + 255) / 256)), 256>>>(pieces, nb * C, npc, C,
                                                                                                  res);
  }
  e = cudaGetLastError();
  std::vector<unsigned long long> hc((size_t)nb);
  if (e == cudaSuccess) e = cudaMemcpy(hc.data(), nc, nb * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && m > 0) e = cudaMemcpy(sums, res, (size_t)nb * C * sizeof(double), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) return e;
  // n of every block: its rows within the strip times its columns
  for (int i = 0; i < q.nI; ++i) {
    const int I = q.I0 + i;
    const long long nr = std::min({(I + 1) * q.b, q.L, q.row0 + q.rows}) - std::max(I * q.b, q.row0);
    for (int J = 0; J < q.B; ++J) {
      const long long k = (long long)i * q.B + J;
      counts[2 * k] = nr * (std::min((J + 1) * q.b, q.L) - J * q.b);
      counts[2 * k + 1] = (int64_t)hc[(size_t)k];
    }
  }
  return cudaSuccess;
}

template cudaError_t launch_block_fields<ModeF32I8>(const BlockGeom &, int, int, const uint32_t *, const void *,
                                                    const void *, double, int, bool, bool, void *, int64_t *, double *);
template cudaError_t launch_block_fields<ModeF32F>(const BlockGeom &, int, int, const uint32_t *, const void *,
                                                   const void *, double, int, bool, bool, void *, int64_t *, double *);
template cudaError_t launch_block_fields<ModeF64>(const BlockGeom &, int, int, const uint32_t *, const void *,
                                                  const void *, double, int, bool, bool, void *, int64_t *, double *);

}  // namespace spgg
