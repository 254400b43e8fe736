// Cluster labelling of a strategy bit plane (spgg_clusters.cuh has the pipeline; include/spgg.h the
// contract).  The only unit that holds these kernels: spgg_capi.cu reaches them through the launchers
// declared in spgg_clusters.cuh (included by spgg_dispatch.h).
#include "spgg_clusters.cuh"

#include <algorithm>

namespace spgg {

// the selected sites of word w of a row: S bit 1 = defect; bits beyond column L-1 are never selected
__device__ __forceinline__ uint32_t ccl_word(const uint32_t *S, int pitchW, int L, int nW, int row, int w, int which) {
  uint32_t v = S[(long long)row * pitchW + w];
  v = which ? v : ~v;
  if (w == nW - 1 && (L & 31)) v &= (1u << (L & 31)) - 1u;
  return v;
}

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
__global__ void __launch_bounds__(CCL_THREADS) k_ccl_local(const uint32_t *S, int pitchW, int L, int which,
                                                           int *parent, int *total, uint32_t *mask) {
  __shared__ uint32_t fs[CCL_TR][CCL_TWW];
  extern __shared__ int ccl_sm[];
  int *lab = ccl_sm, *cnt = ccl_sm + CCL_TR * CCL_TW;
  const int nW = (L + 31) >> 5;
  const int r = threadIdx.x / CCL_TWW, w = threadIdx.x % CCL_TWW;
  const int R = blockIdx.y * CCL_TR + r, W = blockIdx.x * CCL_TWW + w;
  const bool inside = R < L && W < nW;
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
    if (rr >= L || cc >= L) continue;
    const int v = lab[li];
    parent[rr * L + cc] = v < 0 ? -1 : (r0 + v / CCL_TW) * L + c0 + v % CCL_TW;
    if (v == li) total[rr * L + cc] = cnt[li];
  }
}

// unions across the tile borders and, with `periodic`, across row L-1 | 0 and column L-1 | 0
__global__ void k_ccl_merge(const uint32_t *S, int pitchW, int L, int which, int periodic, int *parent) {
  const int nW = (L + 31) >> 5;
  const int nTR = (L + CCL_TR - 1) / CCL_TR, nTC = (L + CCL_TW - 1) / CCL_TW;
  const long long nA = (long long)(nTR - 1) * nW;            // words along the borders between tile rows
  const long long nB = nA + (long long)(nTC - 1) * L;        // + rows along the borders between tile columns
  const long long nC = nB + (periodic ? nW : 0);             // + words of the row seam
  const long long nD = nC + (periodic ? L : 0);              // + rows of the column seam
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < nD; e += (long long)gridDim.x * blockDim.x) {
    if (e < nA || (e >= nB && e < nC)) {   // vertical pairs (ru, c) - (rd, c)
      int ru, rd, w;
      if (e < nA) { rd = (int)(e / nW + 1) * CCL_TR; ru = rd - 1; w = (int)(e % nW); }
      else { ru = L - 1; rd = 0; w = (int)(e - nB); }
      const uint32_t o = ccl_word(S, pitchW, L, nW, ru, w, which) & ccl_word(S, pitchW, L, nW, rd, w, which);
      for (uint32_t s = o & ~(o << 1); s; s &= s - 1) {   // a run of a word lies in one tile: one union per stretch
        const int c = w * 32 + __ffs(s) - 1;
        ccl_unite<true>(parent, rd * L + c, ru * L + c);
      }
    } else {                               // horizontal pairs (row, cl) - (row, cr)
      int row, cl, cr;
      if (e < nB) { const long long k = e - nA; row = (int)(k % L); cr = (int)(k / L + 1) * CCL_TW; cl = cr - 1; }
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
__global__ void __launch_bounds__(CCL_WPB) k_ccl_count(int L, int *parent, int *total, uint32_t *mask, int *blk) {
  const int nW = (L + 31) >> 5;
  const long long w = (long long)blockIdx.x * CCL_WPB + threadIdx.x;
  int n = 0;
  if (w < (long long)L * nW) {
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
__global__ void __launch_bounds__(CCL_WPB) k_ccl_compact(int L, const int *total, const uint32_t *mask, const int *blk,
                                                         int *wordoff, long long *sizes) {
  const int nW = (L + 31) >> 5;
  const long long w = (long long)blockIdx.x * CCL_WPB + threadIdx.x;
  const bool in = w < (long long)L * nW;
  uint32_t m = in ? mask[w] : 0u;
  int k = blk[blockIdx.x] + ccl_block_exclusive_scan<CCL_WPB>(__popc(m), nullptr);
  if (!in) return;
  wordoff[w] = k;
  const int row = (int)(w / nW), col0 = (int)(w % nW) * 32;
  for (; m; m &= m - 1) sizes[k++] = total[row * L + col0 + __ffs(m) - 1];
}

// labels[site] = rank of its root + 1, 0 where the site is not selected.  After k_ccl_count a site's parent
// is a tile-local root, whose parent is the global root.
__global__ void k_ccl_labels(int L, const int *parent, const uint32_t *mask, const int *wordoff, int *labels) {
  const int nW = (L + 31) >> 5;
  const long long n = (long long)L * L;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    const int p = parent[e];
    int v = 0;
    if (p >= 0) {
      const int g = parent[p], row = g / L, col = g % L;
      const long long wi = (long long)row * nW + (col >> 5);
      v = wordoff[wi] + __popc(mask[wi] & ((1u << (col & 31)) - 1u)) + 1;
    }
    labels[e] = v;
  }
}

// ---------------------------------------------------------------- host side
static size_t ccl_smem() { return sizeof(int) * 2 * CCL_TR * CCL_TW; }
static long long ccl_blocks(int L) { return ((long long)L * ((L + 31) / 32) + CCL_WPB - 1) / CCL_WPB; }

void ccl_free(CclScratch *s) {
  cudaFree(s->parent); cudaFree(s->total); cudaFree(s->mask); cudaFree(s->wordoff); cudaFree(s->blk); cudaFree(s->sizes);
  *s = CclScratch();
}

cudaError_t ccl_alloc(CclScratch *s, int L) {
  if (s->L == L) return cudaSuccess;
  ccl_free(s);
  const size_t n = (size_t)L * L, nw = (size_t)L * ((L + 31) / 32);
  cudaError_t e = cudaFuncSetAttribute(k_ccl_local, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ccl_smem());
  if (e == cudaSuccess) e = cudaMalloc((void **)&s->parent, n * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc((void **)&s->total, n * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc((void **)&s->mask, nw * sizeof(uint32_t));
  if (e == cudaSuccess) e = cudaMalloc((void **)&s->wordoff, nw * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc((void **)&s->blk, (size_t)(ccl_blocks(L) + 1) * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc((void **)&s->sizes, (n + 1) / 2 * sizeof(long long));
  if (e != cudaSuccess) {
    ccl_free(s);
    return e;
  }
  s->L = L;
  return cudaSuccess;
}

cudaError_t launch_clusters(const CclScratch &s, const uint32_t *S, int pitchW, int which, int periodic, int64_t *n_clusters) {
  const int L = s.L, nW = (L + 31) / 32;
  const dim3 tiles((unsigned)((nW + CCL_TWW - 1) / CCL_TWW), (unsigned)((L + CCL_TR - 1) / CCL_TR));
  k_ccl_local<<<tiles, CCL_THREADS, ccl_smem()>>>(S, pitchW, L, which, s.parent, s.total, s.mask);
  const long long border = (long long)(tiles.y - 1) * nW + (long long)((L + CCL_TW - 1) / CCL_TW - 1) * L +
                           (periodic ? nW + L : 0);
  k_ccl_merge<<<(unsigned)std::max(1ll, std::min(148ll * 8, (border + 255) / 256)), 256>>>(S, pitchW, L, which, periodic, s.parent);
  const long long nb = ccl_blocks(L);
  k_ccl_count<<<(unsigned)nb, CCL_WPB>>>(L, s.parent, s.total, s.mask, s.blk);
  k_ccl_scan<<<1, CCL_SCAN_THREADS>>>(s.blk, (int)nb);
  k_ccl_compact<<<(unsigned)nb, CCL_WPB>>>(L, s.total, s.mask, s.blk, s.wordoff, s.sizes);
  cudaError_t e = cudaGetLastError();
  int n = 0;
  if (e == cudaSuccess) e = cudaMemcpy(&n, s.blk + nb, sizeof(int), cudaMemcpyDeviceToHost);
  *n_clusters = n;
  return e;
}

cudaError_t launch_cluster_labels(const CclScratch &s) {
  const long long n = (long long)s.L * s.L;
  k_ccl_labels<<<(unsigned)std::max(1ll, std::min(148ll * 16, (n + 255) / 256)), 256>>>(s.L, s.parent, s.mask, s.wordoff, s.total);
  return cudaGetLastError();
}

}  // namespace spgg
