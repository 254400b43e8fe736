// Block-averaged fields of one replica (spgg_block_fields, include/spgg.h): the lattice cut into b x b blocks
// anchored at site (0, 0), per block the number of cooperators and the fp64 sums of R and the Q entries, over
// all sites and over the cooperators.  A pure streaming reduction over the planes spgg_state_digest reads.
//
// Two passes, no floating-point atomics:
//   k_block_count   one thread per (bit word, row tile): popc of the complemented word under each block's column
//                   mask, integer sums over the tile's rows, one 64-bit atomicAdd per (warp, block): integer
//                   sums, so the counts do not depend on scheduling
//   k_block_sums    one thread per column of a tile of up to BLK_TH rows x BLK_TW columns: each thread sums its
//                   column over the rows of a block row in row order, then a segmented shuffle tree with fixed
//                   masks per warp and the warps in order per block give the tile's partial of every block it
//                   touches; when a block spans several tiles (b > BLK_TH or b > BLK_TW) the tiles write pieces
//                   and k_block_pieces adds them per block in piece order
// Tiles are cut at block edges, so the order of every fp64 sum is fixed by (L, row0, rows, b): the same state
// gives bit-identical sums whichever kernel path or chunking reached it.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace spgg {

constexpr int BLK_TH = 32;    // rows of a tile
constexpr int BLK_TW = 256;   // columns of a k_block_sums tile (one per thread)
constexpr long long BLK_MAX_BLOCKS = 1ll << 24;   // cap on B * B (include/spgg.h)

// Block rows and tiles of one call.  The strip holds global rows [row0, row0 + rows); its output covers block
// rows I0 .. I0 + nI - 1.  Rows: b >= BLK_TH cuts each block row into nrc chunks of BLK_TH rows (kr = 1), a
// smaller b puts kr = BLK_TH / b whole block rows in a tile (nrc = 1); columns alike with BLK_TW, kc and ncs.
struct BlockGeom {
  int L, rows, row0, b, B;
  int I0, nI;
  int kr, nrc, n_rt;   // row tiles: n_rt = ceil(nI / kr) * nrc
  int kc, ncs, n_ct;   // column tiles of k_block_sums: n_ct = ceil(B / kc) * ncs
};

inline BlockGeom block_geom(int L, int row0, int rows, int b) {
  BlockGeom q{};
  q.L = L; q.rows = rows; q.row0 = row0; q.b = b; q.B = (L + b - 1) / b;
  q.I0 = row0 / b;
  q.nI = (row0 + rows - 1) / b - q.I0 + 1;
  q.kr = b >= BLK_TH ? 1 : BLK_TH / b;
  q.nrc = b >= BLK_TH ? (b + BLK_TH - 1) / BLK_TH : 1;
  q.n_rt = (q.nI + q.kr - 1) / q.kr * q.nrc;
  q.kc = b >= BLK_TW ? 1 : BLK_TW / b;
  q.ncs = b >= BLK_TW ? (b + BLK_TW - 1) / BLK_TW : 1;
  q.n_ct = (q.B + q.kc - 1) / q.kc * q.ncs;
  return q;
}

// Host launcher (spgg_blocks.cu), instantiated for ModeF32I8, ModeF32F and ModeF64; synchronous on the legacy
// default stream.  S: word 0 of row 0 of the replica's bit plane (rows pitchW words apart); R: column 0 of row 0
// of its R plane (rows pitchB elements apart); Q: its site 0 (rows L * nq entries apart).  rq: the int8 quantum
// (an R value is int8 units x rq in ModeF32I8).  want_r / want_q select the sum channels, m = want_r + want_q * nq.
// scratch: device memory of block_scratch_bytes(q, m) bytes.  counts: host, nI * B * 2 int64 {n, n_C}; sums:
// host, nI * B * 2 * m doubles (unused when m == 0).
size_t block_scratch_bytes(const BlockGeom &q, int m);
template <class Md>
cudaError_t launch_block_fields(const BlockGeom &q, int pitchW, int pitchB, const uint32_t *S, const void *R,
                                const void *Q, double rq, int nq, bool want_r, bool want_q, void *scratch,
                                int64_t *counts, double *sums);

}  // namespace spgg
