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

// the selected sites of word w of a row: S bit 1 = defect; bits beyond column L-1 are never selected
// (also read by the pair counts, spgg_pairs.cu)
__device__ __forceinline__ uint32_t ccl_word(const uint32_t *S, int pitchW, int L, int nW, int row, int w, int which) {
  uint32_t v = S[(long long)row * pitchW + w];
  v = which ? v : ~v;
  if (w == nW - 1 && (L & 31)) v &= (1u << (L & 31)) - 1u;
  return v;
}

// Device scratch of the labelling, owned by the handle (allocated by the first spgg_clusters /
// spgg_strip_clusters call) and sized for the handle's rows x L sites: 8 bytes a site (parent, total),
// 2 bits a site (root mask, per-word rank offsets) and the sizes of at most ceil(rows*L/2) clusters
// (int64).  `total` is reused for the labels that spgg_cluster_labels copies out.
struct CclScratch {
  int rows = 0, L = 0;        // sites the buffers were sized for
  int base = 0;               // label of the first cluster of this strip minus one (0: whole lattice)
  int *parent = nullptr;      // [rows*L] union-find parent (linear index), -1: site not selected;
                              // a strip root that lost to another strip's root: -2 - its global label
  int *total = nullptr;       // [rows*L] size of the set whose root this is; labels after k_ccl_labels
  uint32_t *mask = nullptr;   // [rows*nW] roots, one bit per site
  int *wordoff = nullptr;     // [rows*nW] rank of the first root of each mask word
  int *blk = nullptr;         // [n_blocks + 1] roots per CCL_WPB-word block, then their exclusive scan + total
  long long *sizes = nullptr; // [ceil(rows*L/2)] cluster sizes by rank
};

// Host launchers (spgg_clusters.cu).  S points at word 0 of row 0 of one replica's bit plane, rows pitchW
// words apart.  launch_clusters runs the labelling on the legacy default stream and returns the number of
// clusters (a synchronous copy); launch_cluster_labels then writes the labels into s.total.
cudaError_t ccl_alloc(CclScratch *s, int rows, int L);
void ccl_free(CclScratch *s);
cudaError_t launch_clusters(const CclScratch &s, const uint32_t *S, int pitchW, int which, int periodic, int64_t *n_clusters);
cudaError_t launch_cluster_labels(const CclScratch &s);

// ---------------------------------------------------------------- row strips (spgg_strip_clusters)
// A lattice split into row strips, one per rank.  Each strip labels its own rows with the pipeline above
// (column seam when periodic, never the row seam) and writes one boundary record (ccl_record_bytes(L),
// the same on every rank); every rank then resolves the records of all ranks on its device:
//   k_res_init / k_res_seams   union-find (ccl_unite) over the boundary roots ("parts") of all strips,
//                  linked across strip k's last row | strip k+1's first row and, periodic, strip N-1 | 0;
//                  parts are numbered in global root order, so every merged set's root is its part with
//                  the smallest global linear index, the same on every rank
//   k_res_sizes    merged sizes; a part that is not its set's root is a strip root that lost root status
//   k_res_lost     per strip: lost parts below each part (the parts are sorted by root), lost count
//   k_res_first    owned clusters per strip (strip roots - lost parts) and their exclusive scan:
//                  first label of each strip, number of clusters of the lattice
//   k_res_label    the global label of every merged set (first label of the owner + owned rank + 1)
//   k_res_apply    this strip: owner parts take the merged size, lost parts leave the root mask and hold
//                  -2 - label in parent
// then k_ccl_count / k_ccl_scan / k_ccl_compact rank this strip's owned roots again (sizes in raster
// order) and k_ccl_labels adds s.base.
//
// The record (int32 words): header CCL_REC_HDR words {magic, L, row0, rows, which, flags, strip roots,
// parts}, then part[2L] (the part index of the local root of each site of the first row, then of the
// last row; -1: site not selected), then per part, sorted by root, root[2L] (global linear index),
// rank[2L] (raster rank among the strip's roots) and size[2L] (sites in the strip).
constexpr int CCL_REC_HDR = 8;
constexpr int CCL_REC_MAGIC = 0x53434c31;  // "SCL1"
enum { CCL_H_MAGIC, CCL_H_L, CCL_H_ROW0, CCL_H_ROWS, CCL_H_WHICH, CCL_H_FLAGS, CCL_H_NLOCAL, CCL_H_NPARTS };
inline long long ccl_record_bytes(int L) { return 4ll * (CCL_REC_HDR + 8ll * L); }

// record building (2L slots) and resolution (2L parts per strip) scratch, owned by the handle
struct CclStripScratch {
  int L = 0, world = 0;        // sized for
  int *keys = nullptr;         // [2L] root of each boundary site (INT_MAX: none), then sorted
  int *uniq = nullptr;         // [2L + 1] distinct roots, [2L]: their number
  void *cub = nullptr;         // CUB temporary storage
  size_t cub_bytes = 0;
  int *uf = nullptr;           // [world*2L] union-find over the parts of all strips
  int *msize = nullptr;        // [world*2L] merged size at each set root
  int *lost = nullptr;         // [world*2L] lost parts below each part
  int *lab = nullptr;          // [world*2L] global label at each set root
  int *strip = nullptr;        // [3*world + 1] lost parts, owned clusters, first label per strip; clusters
};

void ccl_strip_free(CclStripScratch *t);
cudaError_t ccl_strip_alloc(CclStripScratch *t, int L, int world);
// strip-local pass of the rows in S (row0 = global row of S's first row) and this strip's record;
// synchronous, returns the number of strip roots
cudaError_t launch_strip_clusters(const CclScratch &s, CclStripScratch &t, const uint32_t *S, int pitchW, int row0,
                                  int which, int periodic, void *dev_record, int64_t *n_local);
// resolution of `world` validated records (dev_records, rank order) for strip `rank`: this strip's owned
// clusters (sizes in raster order in s.sizes, labels from s.base + 1 on), the label before its first one
// and the number of clusters of the lattice; synchronous
cudaError_t launch_strip_resolve(CclScratch &s, CclStripScratch &t, const void *dev_records, int world, int rank,
                                 int periodic, int64_t *n_owned, int64_t *first_label, int64_t *n_total);

}  // namespace spgg