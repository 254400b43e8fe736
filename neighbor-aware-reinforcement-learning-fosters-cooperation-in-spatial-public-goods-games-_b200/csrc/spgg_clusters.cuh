// Connected-component labelling of one replica's strategy bit plane (spgg_clusters, include/spgg.h):
// scipy.ndimage.label(S == which) with 4-connectivity, optionally periodic, labels numbered in
// increasing order of each cluster's smallest linear index row*L + col.
//
// Block-based union-find (Playne & Hawick 2018, Allegretti et al. 2019), five launches:
//   k_ccl_local    one CTA per CCL_TR x CCL_TW tile: provisional labels in shared memory, horizontal
//                  runs from the bit words, vertical unions where two rows' runs overlap; writes
//                  parent[site] = linear index of the tile-local root, total[root] = tile-local size and
//                  one bit per tile-local root into a mask laid out like the bit plane (nW words a row)
//   k_ccl_merge    unions across tile borders (and the two seams of the torus) with atomicMin links,
//                  so every root is the smallest linear index of its set and the result does not
//                  depend on scheduling
//   k_ccl_count    a tile-local root that is no longer a global root adds its size to its global
//                  root (one atomic per tile a cluster touches, never one per site) and points at it;
//                  the mask keeps the global roots only, each CCL_WPB-word block counts its roots
//   k_ccl_scan     exclusive scan of the block counts (one CTA) -> n_clusters
//   k_ccl_compact  per-word ranks in raster order, sizes[rank] = total[root]
// and, on request, k_ccl_labels: labels[site] = rank(root(site)) + 1, 0 where the site is not selected.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace spgg {

constexpr int CCL_TR = 32;               // tile rows
constexpr int CCL_TWW = 8;               // tile width in 32-bit words (256 columns)
constexpr int CCL_TW = CCL_TWW * 32;
constexpr int CCL_THREADS = CCL_TR * CCL_TWW;  // k_ccl_local: one thread per (row, word) of the tile
constexpr int CCL_WPB = 512;             // mask words per block of k_ccl_count / k_ccl_compact
constexpr int CCL_SCAN_THREADS = 1024;

// Device scratch of the labelling, owned by the handle (allocated by the first spgg_clusters call):
// 8 bytes a site (parent, total), 2 bits a site (root mask, per-word rank offsets) and the sizes of
// at most ceil(L*L/2) clusters (int64).  `total` is reused for the labels that spgg_cluster_labels
// copies out.
struct CclScratch {
  int L = 0;                  // lattice side the buffers were sized for
  int *parent = nullptr;      // [L*L] union-find parent (linear index), -1: site not selected
  int *total = nullptr;       // [L*L] size of the set whose root this is; labels after k_ccl_labels
  uint32_t *mask = nullptr;   // [L*nW] roots, one bit per site
  int *wordoff = nullptr;     // [L*nW] rank of the first root of each mask word
  int *blk = nullptr;         // [n_blocks + 1] roots per CCL_WPB-word block, then their exclusive scan + total
  long long *sizes = nullptr; // [ceil(L*L/2)] cluster sizes by rank
};

// Host launchers (spgg_clusters.cu).  S points at word 0 of row 0 of one replica's bit plane, rows pitchW
// words apart.  launch_clusters runs the labelling on the legacy default stream and returns the number of
// clusters (a synchronous copy); launch_cluster_labels then writes the labels into s.total.
cudaError_t ccl_alloc(CclScratch *s, int L);
void ccl_free(CclScratch *s);
cudaError_t launch_clusters(const CclScratch &s, const uint32_t *S, int pitchW, int which, int periodic, int64_t *n_clusters);
cudaError_t launch_cluster_labels(const CclScratch &s);

}  // namespace spgg
