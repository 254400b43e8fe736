// Cluster labelling of a strategy bit plane (spgg_clusters.cuh has the pipeline; include/spgg.h the
// contract).  The only unit that holds these kernels: spgg_capi.cu reaches them through the launchers
// declared in spgg_clusters.cuh (included by spgg_dispatch.h).
#include "spgg_clusters.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>

#include <algorithm>
#include <climits>

namespace spgg {

// Union-find with parent[x] <= x: every root is the smallest index of its set.  A link is an atomicMin on
// a root; if the root was linked meanwhile the loop goes on with the value it found (Playne & Hawick).
__device__ __forceinline__ int ccl_find(const int *P, int x) {
  const volatile int *V = P;
  int p;
  while ((p = V[x]) != x) x = p;
  return x;
}

// global version with path halving; the halving store is an atomicMin, so it never undoes a link
__device__ __forceinline__ int ccl_find_halve(int *P, int x) {
  volatile int *V = P;
  for (;;) {
    const int p = V[x];
    if (p == x) return x;
    const int gp = V[p];
    if (gp == p) return p;
    atomicMin(P + x, gp);
    x = gp;
  }
}

template <bool HALVE>
__device__ __forceinline__ void ccl_unite(int *P, int a, int b) {
  for (;;) {
    a = HALVE ? ccl_find_halve(P, a) : ccl_find(P, a);
    b = HALVE ? ccl_find_halve(P, b) : ccl_find(P, b);
    if (a == b) return;
    if (a > b) { const int t = a; a = b; b = t; }
    const int old = atomicMin(P + b, a);
    if (old == b) return;
    b = old;
  }
}

// one CTA per CCL_TR x CCL_TW tile; dynamic shared memory: lab[CCL_TR*CCL_TW] and cnt[CCL_TR*CCL_TW]
__global__ void __launch_bounds__(CCL_THREADS) k_ccl_local(const uint32_t *S, int pitchW, int rows, int L, int which,
                                                           int *parent, int *total, uint32_t *mask) {
  __shared__ uint32_t fs[CCL_TR][CCL_TWW];
  extern __shared__ int ccl_sm[];
  int *lab = ccl_sm, *cnt = ccl_sm + CCL_TR * CCL_TW;
  const int nW = (L + 31) >> 5;
  const int r = threadIdx.x / CCL_TWW, w = threadIdx.x % CCL_TWW;
  const int R = blockIdx.y * CCL_TR + r, W = blockIdx.x * CCL_TWW + w;
  const bool inside = R < rows && W < nW;
  const uint32_t f = inside ? ccl_word(S, pitchW, L, nW, R, W, which) : 0u;
  fs[r][w] = f;
  __syncthreads();
  // every selected site starts in the set of the first site of its run within the word
  for (int li = threadIdx.x; li < CCL_TR * CCL_TW; li += CCL_THREADS) {
    const uint32_t fw = fs[li / CCL_TW][(li % CCL_TW) >> 5];
    const int b = li & 31;
    int v = -1;
    if ((fw >> b) & 1u) {
      const uint32_t z = ~fw & ((1u << b) - 1u);   // clear bits below b: the run starts after the highest
      v = li - b + (z ? 32 - __clz(z) : 0);
    }
    lab[li] = v;
    cnt[li] = 0;
  }
  __syncthreads();
  const int base = r * CCL_TW + w * 32;
  if (w > 0 && (f & 1u) && (fs[r][w - 1] >> 31)) ccl_unite<false>(lab, base, base - 1);   // run across the word edge
  if (r > 0) {   // one union per overlapping stretch of this row's and the row above's runs
    const uint32_t o = f & fs[r - 1][w];
    for (uint32_t s = o & ~(o << 1); s; s &= s - 1) {
      const int b = __ffs(s) - 1;
      ccl_unite<false>(lab, base + b, base + b - CCL_TW);
    }
  }
  __syncthreads();
  for (int li = threadIdx.x; li < CCL_TR * CCL_TW; li += CCL_THREADS)
    if (lab[li] >= 0) lab[li] = ccl_find(lab, li);
  __syncthreads();
  // tile-local sizes (one shared atomic per run of a word) and the tile-local roots, which start runs
  uint32_t roots = 0;
  for (uint32_t s = f & ~(f << 1); s; s &= s - 1) {
    const int b = __ffs(s) - 1;
    const uint32_t rest = ~(f >> b);
    const int root = lab[base + b];
    atomicAdd(cnt + root, rest ? __ffs(rest) - 1 : 32);
    if (root == base + b) roots |= 1u << b;
  }
  if (inside) mask[(long long)R * nW + W] = roots;
  __syncthreads();
  const int r0 = blockIdx.y * CCL_TR, c0 = blockIdx.x * CCL_TW;
  for (int li = threadIdx.x; li < CCL_TR * CCL_TW; li += CCL_THREADS) {
    const int rr = r0 + li / CCL_TW, cc = c0 + li % CCL_TW;
    if (rr >= rows || cc >= L) continue;
    const int v = lab[li];
    parent[rr * L + cc] = v < 0 ? -1 : (r0 + v / CCL_TW) * L + c0 + v % CCL_TW;
    if (v == li) total[rr * L + cc] = cnt[li];
  }
}

// unions across the tile borders, with `row_seam` across row rows-1 | 0 and with `periodic` across
// column L-1 | 0
__global__ void k_ccl_merge(const uint32_t *S, int pitchW, int rows, int L, int which, int periodic, int row_seam,
                            int *parent) {
  const int nW = (L + 31) >> 5;
  const int nTR = (rows + CCL_TR - 1) / CCL_TR, nTC = (L + CCL_TW - 1) / CCL_TW;
  const long long nA = (long long)(nTR - 1) * nW;            // words along the borders between tile rows
  const long long nB = nA + (long long)(nTC - 1) * rows;     // + rows along the borders between tile columns
  const long long nC = nB + (row_seam ? nW : 0);             // + words of the row seam
  const long long nD = nC + (periodic ? rows : 0);           // + rows of the column seam
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < nD; e += (long long)gridDim.x * blockDim.x) {
    if (e < nA || (e >= nB && e < nC)) {   // vertical pairs (ru, c) - (rd, c)
      int ru, rd, w;
      if (e < nA) { rd = (int)(e / nW + 1) * CCL_TR; ru = rd - 1; w = (int)(e % nW); }
      else { ru = rows - 1; rd = 0; w = (int)(e - nB); }
      const uint32_t o = ccl_word(S, pitchW, L, nW, ru, w, which) & ccl_word(S, pitchW, L, nW, rd, w, which);
      for (uint32_t s = o & ~(o << 1); s; s &= s - 1) {   // a run of a word lies in one tile: one union per stretch
        const int c = w * 32 + __ffs(s) - 1;
        ccl_unite<true>(parent, rd * L + c, ru * L + c);
      }
    } else {                               // horizontal pairs (row, cl) - (row, cr)
      int row, cl, cr;
      if (e < nB) { const long long k = e - nA; row = (int)(k % rows); cr = (int)(k / rows + 1) * CCL_TW; cl = cr - 1; }
      else { row = (int)(e - nC); cl = L - 1; cr = 0; }
      const uint32_t fl = ccl_word(S, pitchW, L, nW, row, cl >> 5, which), fr = ccl_word(S, pitchW, L, nW, row, cr >> 5, which);
      if (((fl >> (cl & 31)) & 1u) && ((fr >> (cr & 31)) & 1u)) ccl_unite<true>(parent, row * L + cr, row * L + cl);
    }
  }
}

template <int NT>
__device__ __forceinline__ int ccl_block_exclusive_scan(int v, int *total_out) {
  __shared__ int ws[NT / 32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int incl = v;
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) ws[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    int x = lane < NT / 32 ? ws[lane] : 0;
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += t;
    }
    if (lane < NT / 32) ws[lane] = x;
  }
  __syncthreads();
  if (total_out) *total_out = ws[NT / 32 - 1];
  return incl - v + (wid ? ws[wid - 1] : 0);
}

// tile-local roots that are no longer global roots hand their size to their global root and point at it
__global__ void __launch_bounds__(CCL_WPB) k_ccl_count(int rows, int L, int *parent, int *total, uint32_t *mask, int *blk) {
  const int nW = (L + 31) >> 5;
  const long long w = (long long)blockIdx.x * CCL_WPB + threadIdx.x;
  int n = 0;
  if (w < (long long)rows * nW) {
    uint32_t m = mask[w], keep = m;
    const int row = (int)(w / nW), col0 = (int)(w % nW) * 32;
    for (; m; m &= m - 1) {
      const int b = __ffs(m) - 1, x = row * L + col0 + b;
      const int g = ccl_find(parent, x);
      if (g != x) {
        atomicAdd(total + g, total[x]);
        parent[x] = g;
        keep &= ~(1u << b);
      }
    }
    mask[w] = keep;
    n = __popc(keep);
  }
  int tot;
  ccl_block_exclusive_scan<CCL_WPB>(n, &tot);
  if (threadIdx.x == 0) blk[blockIdx.x] = tot;
}

// exclusive scan of the per-block root counts in place; blk[nb] = number of clusters
__global__ void __launch_bounds__(CCL_SCAN_THREADS) k_ccl_scan(int *blk, int nb) {
  const int per = (nb + CCL_SCAN_THREADS - 1) / CCL_SCAN_THREADS;
  const int lo = min(nb, threadIdx.x * per), hi = min(nb, lo + per);
  int s = 0;
  for (int i = lo; i < hi; ++i) s += blk[i];
  int tot;
  int run = ccl_block_exclusive_scan<CCL_SCAN_THREADS>(s, &tot);
  for (int i = lo; i < hi; ++i) {
    const int v = blk[i];
    blk[i] = run;
    run += v;
  }
  if (threadIdx.x == 0) blk[nb] = tot;
}

// ranks in raster order: sizes[rank] = total[root]
__global__ void __launch_bounds__(CCL_WPB) k_ccl_compact(int rows, int L, const int *total, const uint32_t *mask, const int *blk,
                                                         int *wordoff, long long *sizes) {
  const int nW = (L + 31) >> 5;
  const long long w = (long long)blockIdx.x * CCL_WPB + threadIdx.x;
  const bool in = w < (long long)rows * nW;
  uint32_t m = in ? mask[w] : 0u;
  int k = blk[blockIdx.x] + ccl_block_exclusive_scan<CCL_WPB>(__popc(m), nullptr);
  if (!in) return;
  wordoff[w] = k;
  const int row = (int)(w / nW), col0 = (int)(w % nW) * 32;
  for (; m; m &= m - 1) sizes[k++] = total[row * L + col0 + __ffs(m) - 1];
}

// labels[site] = base + rank of its root + 1, 0 where the site is not selected.  After k_ccl_count a site's
// parent is a tile-local root, whose parent is the root.  A strip root that lost to another strip's root
// (k_res_apply) has left the mask and holds -2 - its global label as its parent.
__global__ void k_ccl_labels(int rows, int L, int base, const int *parent, const uint32_t *mask, const int *wordoff,
                             int *labels) {
  const int nW = (L + 31) >> 5;
  const long long n = (long long)rows * L;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    const int p = parent[e];
    int v = 0;
    if (p <= -2) {
      v = -2 - p;                             // the site is a lost root
    } else if (p >= 0) {
      const int g = parent[p], row = g / L, col = g % L;
      if (g <= -2) {
        v = -2 - g;                           // its tile-local root is a lost root
      } else {
        const long long wi = (long long)row * nW + (col >> 5);
        const uint32_t m = mask[wi];
        v = (m >> (col & 31)) & 1u ? base + wordoff[wi] + __popc(m & ((1u << (col & 31)) - 1u)) + 1 : -2 - parent[g];
      }
    }
    labels[e] = v;
  }
}

// ---------------------------------------------------------------- row strips: the boundary record
// the strip root of boundary slot e (first row, then last row), or -1 when the site is not selected
__device__ __forceinline__ int ccl_slot_root(const int *parent, int rows, int L, int e) {
  const int x = (e < L ? 0 : rows - 1) * L + (e < L ? e : e - L);
  const int p = parent[x];
  return p < 0 ? -1 : parent[p];
}

__global__ void k_ccl_bnd(const int *parent, int rows, int L, int *keys) {
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < 2 * L; e += gridDim.x * blockDim.x) {
    const int g = ccl_slot_root(parent, rows, L, e);
    keys[e] = g < 0 ? INT_MAX : g;
  }
}

// uniq: the distinct boundary roots in increasing order (their part indices), then INT_MAX if a site was
// not selected; n_sel: how many
__global__ void k_ccl_record(const int *parent, const int *total, const uint32_t *mask, const int *wordoff,
                             const int *n_local, int rows, int L, int row0, int which, int flags, const int *uniq,
                             const int *n_sel, int *rec) {
  const int nW = (L + 31) >> 5;
  const int ns = *n_sel, np = ns - (ns > 0 && uniq[ns - 1] == INT_MAX);
  int *part = rec + CCL_REC_HDR, *root = part + 2 * L, *rank = root + 2 * L, *size = rank + 2 * L;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < 2 * L; e += gridDim.x * blockDim.x) {
    const int g = ccl_slot_root(parent, rows, L, e);
    int k = -1;
    if (g >= 0) {   // lower bound of g in uniq[0, np)
      int lo = 0, hi = np;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (uniq[mid] < g) lo = mid + 1; else hi = mid;
      }
      k = lo;
    }
    part[e] = k;
    if (e < np) {
      const int r = uniq[e], col = r % L;
      const long long wi = (long long)(r / L) * nW + (col >> 5);
      root[e] = row0 * L + r;
      rank[e] = wordoff[wi] + __popc(mask[wi] & ((1u << (col & 31)) - 1u));
      size[e] = total[r];
    } else {
      root[e] = -1; rank[e] = -1; size[e] = 0;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    rec[CCL_H_MAGIC] = CCL_REC_MAGIC; rec[CCL_H_L] = L; rec[CCL_H_ROW0] = row0; rec[CCL_H_ROWS] = rows;
    rec[CCL_H_WHICH] = which; rec[CCL_H_FLAGS] = flags; rec[CCL_H_NLOCAL] = *n_local; rec[CCL_H_NPARTS] = np;
  }
}

// ---------------------------------------------------------------- row strips: resolution of the records
// part id = strip * 2L + index in the strip's record; ids increase with the global linear index of the root
__device__ __forceinline__ const int *ccl_rec(const int *recs, int L, int k) { return recs + (long long)k * (CCL_REC_HDR + 8 * L); }

__global__ void k_res_init(const int *recs, int world, int L, int *uf, int *msize) {
  for (int id = blockIdx.x * blockDim.x + threadIdx.x; id < world * 2 * L; id += gridDim.x * blockDim.x) {
    const int k = id / (2 * L);
    uf[id] = id - k * 2 * L < ccl_rec(recs, L, k)[CCL_H_NPARTS] ? id : -1;
    msize[id] = 0;
  }
}

// strip k's last row | strip k+1's first row, and strip world-1 | strip 0 when periodic
__global__ void k_res_seams(const int *recs, int world, int L, int periodic, int *uf) {
  const int n = (world - 1 + periodic) * L;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
    const int k = e / L, c = e - k * L, k2 = k + 1 == world ? 0 : k + 1;
    const int *up = ccl_rec(recs, L, k) + CCL_REC_HDR + L, *dn = ccl_rec(recs, L, k2) + CCL_REC_HDR;
    const int a = up[c], b = dn[c];
    if (a < 0 || b < 0 || (c > 0 && up[c - 1] == a && dn[c - 1] == b)) continue;   // one union per stretch
    ccl_unite<true>(uf, k * 2 * L + a, k2 * 2 * L + b);
  }
}

// uf[id] = root of the merged set; msize[root] = sum of its parts' sizes
__global__ void k_res_sizes(const int *recs, int world, int L, int *uf, int *msize) {
  for (int id = blockIdx.x * blockDim.x + threadIdx.x; id < world * 2 * L; id += gridDim.x * blockDim.x) {
    if (uf[id] < 0) continue;
    const int k = id / (2 * L), r = ccl_find(uf, id);
    uf[id] = r;
    atomicAdd(msize + r, ccl_rec(recs, L, k)[CCL_REC_HDR + 6 * L + id - k * 2 * L]);
  }
}

// one CTA per strip: lost[id] = parts of the strip below id that are not their set's root; strip[k] = all
__global__ void __launch_bounds__(CCL_SCAN_THREADS) k_res_lost(const int *recs, int L, const int *uf, int *lost,
                                                               int *strip) {
  const int k = blockIdx.x, np = ccl_rec(recs, L, k)[CCL_H_NPARTS];
  int carry = 0;
  for (int j0 = 0; j0 < np; j0 += CCL_SCAN_THREADS) {
    const int j = j0 + threadIdx.x, id = k * 2 * L + j;
    int tot;
    const int x = ccl_block_exclusive_scan<CCL_SCAN_THREADS>(j < np && uf[id] != id, &tot);
    if (j < np) lost[id] = carry + x;
    carry += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) strip[k] = carry;
}

// strip[world + k] = clusters owned by strip k, strip[2 world + k] = their first label - 1, strip[3 world] = all
__global__ void k_res_first(const int *recs, int world, int L, int *strip) {
  int acc = 0;
  for (int k = 0; k < world; ++k) {
    const int owned = ccl_rec(recs, L, k)[CCL_H_NLOCAL] - strip[k];
    strip[world + k] = owned;
    strip[2 * world + k] = acc;
    acc += owned;
  }
  strip[3 * world] = acc;
}

// global label of every merged set, at its root part: first label of the owner + rank among its owned roots
__global__ void k_res_label(const int *recs, int world, int L, const int *uf, const int *lost, const int *strip, int *lab) {
  for (int id = blockIdx.x * blockDim.x + threadIdx.x; id < world * 2 * L; id += gridDim.x * blockDim.x) {
    if (uf[id] != id) continue;
    const int k = id / (2 * L);
    lab[id] = strip[2 * world + k] + ccl_rec(recs, L, k)[CCL_REC_HDR + 4 * L + id - k * 2 * L] - lost[id] + 1;
  }
}

// this strip's parts: an owner takes the merged size, a lost root leaves the mask and keeps its label
__global__ void k_res_apply(const int *recs, int rank, int L, const int *uf, const int *msize, const int *lab,
                            int *parent, int *total, uint32_t *mask) {
  const int nW = (L + 31) >> 5;
  const int *rec = ccl_rec(recs, L, rank), np = rec[CCL_H_NPARTS], row0 = rec[CCL_H_ROW0];
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < np; j += gridDim.x * blockDim.x) {
    const int id = rank * 2 * L + j, r = uf[id], g = rec[CCL_REC_HDR + 2 * L + j] - row0 * L, col = g % L;
    if (r == id) {
      total[g] = msize[id];
    } else {
      atomicAnd(mask + (long long)(g / L) * nW + (col >> 5), ~(1u << (col & 31)));
      parent[g] = -2 - lab[r];
    }
  }
}

// ---------------------------------------------------------------- host side
static size_t ccl_smem() { return sizeof(int) * 2 * CCL_TR * CCL_TW; }
static long long ccl_blocks(int rows, int L) { return ((long long)rows * ((L + 31) / 32) + CCL_WPB - 1) / CCL_WPB; }
static unsigned ccl_grid(long long n) { return (unsigned)std::max(1ll, std::min(148ll * 8, (n + 255) / 256)); }

void ccl_free(CclScratch *s) {
  cudaFree(s->parent); cudaFree(s->total); cudaFree(s->mask); cudaFree(s->wordoff); cudaFree(s->blk); cudaFree(s->sizes);
  *s = CclScratch();
}

cudaError_t ccl_alloc(CclScratch *s, int rows, int L) {
  if (s->rows == rows && s->L == L) return cudaSuccess;
  ccl_free(s);
  const size_t n = (size_t)rows * L, nw = (size_t)rows * ((L + 31) / 32);
  cudaError_t e = cudaFuncSetAttribute(k_ccl_local, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ccl_smem());
  if (e == cudaSuccess) e = cudaMalloc((void **)&s->parent, n * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc((void **)&s->total, n * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc((void **)&s->mask, nw * sizeof(uint32_t));
  if (e == cudaSuccess) e = cudaMalloc((void **)&s->wordoff, nw * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc((void **)&s->blk, (size_t)(ccl_blocks(rows, L) + 1) * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc((void **)&s->sizes, (n + 1) / 2 * sizeof(long long));
  if (e != cudaSuccess) {
    ccl_free(s);
    return e;
  }
  s->rows = rows;
  s->L = L;
  return cudaSuccess;
}

// strip-local labelling: with row_seam = periodic it is the whole-lattice labelling
static void ccl_pass(const CclScratch &s, const uint32_t *S, int pitchW, int which, int periodic, int row_seam) {
  const int rows = s.rows, L = s.L, nW = (L + 31) / 32;
  const dim3 tiles((unsigned)((nW + CCL_TWW - 1) / CCL_TWW), (unsigned)((rows + CCL_TR - 1) / CCL_TR));
  k_ccl_local<<<tiles, CCL_THREADS, ccl_smem()>>>(S, pitchW, rows, L, which, s.parent, s.total, s.mask);
  const long long border = (long long)(tiles.y - 1) * nW + (long long)((L + CCL_TW - 1) / CCL_TW - 1) * rows +
                           (row_seam ? nW : 0) + (periodic ? rows : 0);
  k_ccl_merge<<<ccl_grid(border), 256>>>(S, pitchW, rows, L, which, periodic, row_seam, s.parent);
}

// ranks of the roots in the mask: per-word offsets, sizes by rank, blk[nb] = number of roots
static void ccl_rank(const CclScratch &s) {
  const long long nb = ccl_blocks(s.rows, s.L);
  k_ccl_count<<<(unsigned)nb, CCL_WPB>>>(s.rows, s.L, s.parent, s.total, s.mask, s.blk);
  k_ccl_scan<<<1, CCL_SCAN_THREADS>>>(s.blk, (int)nb);
  k_ccl_compact<<<(unsigned)nb, CCL_WPB>>>(s.rows, s.L, s.total, s.mask, s.blk, s.wordoff, s.sizes);
}

static cudaError_t ccl_count_out(const CclScratch &s, int64_t *n_out) {
  cudaError_t e = cudaGetLastError();
  int n = 0;
  if (e == cudaSuccess) e = cudaMemcpy(&n, s.blk + ccl_blocks(s.rows, s.L), sizeof(int), cudaMemcpyDeviceToHost);
  *n_out = n;
  return e;
}

cudaError_t launch_clusters(const CclScratch &s, const uint32_t *S, int pitchW, int which, int periodic, int64_t *n_clusters) {
  ccl_pass(s, S, pitchW, which, periodic, periodic);
  ccl_rank(s);
  return ccl_count_out(s, n_clusters);
}

cudaError_t launch_cluster_labels(const CclScratch &s) {
  const long long n = (long long)s.rows * s.L;
  k_ccl_labels<<<(unsigned)std::max(1ll, std::min(148ll * 16, (n + 255) / 256)), 256>>>(s.rows, s.L, s.base, s.parent,
                                                                                       s.mask, s.wordoff, s.total);
  return cudaGetLastError();
}

void ccl_strip_free(CclStripScratch *t) {
  cudaFree(t->keys); cudaFree(t->uniq); cudaFree(t->cub);
  cudaFree(t->uf); cudaFree(t->msize); cudaFree(t->lost); cudaFree(t->lab); cudaFree(t->strip);
  *t = CclStripScratch();
}

cudaError_t ccl_strip_alloc(CclStripScratch *t, int L, int world) {
  cudaError_t e = cudaSuccess;
  if (t->L != L) {
    ccl_strip_free(t);
    const int n = 2 * L;
    size_t b1 = 0, b2 = 0;
    e = cub::DeviceRadixSort::SortKeys(nullptr, b1, (const int *)nullptr, (int *)nullptr, n);
    if (e == cudaSuccess) e = cub::DeviceSelect::Unique(nullptr, b2, (const int *)nullptr, (int *)nullptr, (int *)nullptr, n);
    t->cub_bytes = std::max(b1, b2);
    if (e == cudaSuccess) e = cudaMalloc(&t->cub, t->cub_bytes);
    if (e == cudaSuccess) e = cudaMalloc((void **)&t->keys, n * sizeof(int));
    if (e == cudaSuccess) e = cudaMalloc((void **)&t->uniq, (n + 1) * sizeof(int));
    if (e != cudaSuccess) {
      ccl_strip_free(t);
      return e;
    }
    t->L = L;
  }
  if (world > 0 && t->world != world) {
    cudaFree(t->uf); cudaFree(t->msize); cudaFree(t->lost); cudaFree(t->lab); cudaFree(t->strip);
    t->uf = t->msize = t->lost = t->lab = t->strip = nullptr;
    t->world = 0;
    const size_t n = (size_t)world * 2 * L;
    e = cudaMalloc((void **)&t->uf, n * sizeof(int));
    if (e == cudaSuccess) e = cudaMalloc((void **)&t->msize, n * sizeof(int));
    if (e == cudaSuccess) e = cudaMalloc((void **)&t->lost, n * sizeof(int));
    if (e == cudaSuccess) e = cudaMalloc((void **)&t->lab, n * sizeof(int));
    if (e == cudaSuccess) e = cudaMalloc((void **)&t->strip, (3 * (size_t)world + 1) * sizeof(int));
    if (e != cudaSuccess) {
      ccl_strip_free(t);
      return e;
    }
    t->world = world;
  }
  return e;
}

cudaError_t launch_strip_clusters(const CclScratch &s, CclStripScratch &t, const uint32_t *S, int pitchW, int row0,
                                  int which, int periodic, void *dev_record, int64_t *n_local) {
  const int L = s.L, n = 2 * L;
  ccl_pass(s, S, pitchW, which, periodic, 0);
  ccl_rank(s);
  k_ccl_bnd<<<ccl_grid(n), 256>>>(s.parent, s.rows, L, t.keys);
  size_t bytes = t.cub_bytes;
  cudaError_t e = cub::DeviceRadixSort::SortKeys(t.cub, bytes, t.keys, t.uniq, n);
  bytes = t.cub_bytes;
  if (e == cudaSuccess) e = cub::DeviceSelect::Unique(t.cub, bytes, t.uniq, t.keys, t.uniq + n, n);
  if (e != cudaSuccess) return e;
  k_ccl_record<<<ccl_grid(n), 256>>>(s.parent, s.total, s.mask, s.wordoff, s.blk + ccl_blocks(s.rows, L), s.rows, L,
                                     row0, which, periodic, t.keys, t.uniq + n, (int *)dev_record);
  return ccl_count_out(s, n_local);
}

cudaError_t launch_strip_resolve(CclScratch &s, CclStripScratch &t, const void *dev_records, int world, int rank,
                                 int periodic, int64_t *n_owned, int64_t *first_label, int64_t *n_total) {
  const int L = s.L, n = world * 2 * L;
  const int *recs = (const int *)dev_records;
  k_res_init<<<ccl_grid(n), 256>>>(recs, world, L, t.uf, t.msize);
  if (world - 1 + periodic > 0) k_res_seams<<<ccl_grid((long long)(world - 1 + periodic) * L), 256>>>(recs, world, L, periodic, t.uf);
  k_res_sizes<<<ccl_grid(n), 256>>>(recs, world, L, t.uf, t.msize);
  k_res_lost<<<world, CCL_SCAN_THREADS>>>(recs, L, t.uf, t.lost, t.strip);
  k_res_first<<<1, 1>>>(recs, world, L, t.strip);
  k_res_label<<<ccl_grid(n), 256>>>(recs, world, L, t.uf, t.lost, t.strip, t.lab);
  k_res_apply<<<ccl_grid(2 * L), 256>>>(recs, rank, L, t.uf, t.msize, t.lab, s.parent, s.total, s.mask);
  ccl_rank(s);
  int st[2] = {0, 0};
  cudaError_t e = ccl_count_out(s, n_owned);
  if (e == cudaSuccess) e = cudaMemcpy(&st[0], t.strip + 2 * world + rank, sizeof(int), cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(&st[1], t.strip + 3 * world, sizeof(int), cudaMemcpyDeviceToHost);
  s.base = st[0];
  *first_label = st[0];
  *n_total = st[1];
  return e;
}

}  // namespace spgg
