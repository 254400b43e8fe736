// State overlaps of replicas rep0 .. rep0 + n_rep - 1 against a snapshot (spgg_overlap, include/spgg.h): the joint
// strategy counts {then, now}, and per channel (R, then the nq Q entries) the number of changed values, the exact
// max |now - then| and the fp64 sums of |now - then| and (now - then)^2.
//
// One streaming pass per call over the live planes and the snapshot's (the same layout), one launch for all
// replicas (grid.y), then one small launch for the sums:
//   k_overlap       CTA x of replica y covers the rows of tile x, whose height is fixed by (L, rows).  Each thread
//                   walks three independent sequences: the tile's bit words (popc of the two words under the
//                   valid-column mask, four joint counts), its R rows in 16-byte chunks, and its Q entries as one
//                   flat run of sites (Q has no row padding), a batch of sites per step with every load of the
//                   batch issued before the arithmetic.  Counts and |d| maxima go through 64-bit integer atomics
//                   (exact, free of scheduling); the fp64 sums are reduced in a fixed order per CTA (shuffle
//                   butterfly, then the warps in order) into one partial per (tile, channel, sum)
//   k_overlap_fold  one warp per (replica, channel, sum) adds the tiles' partials: lane l the tiles l, l + 32, ...
//                   in order, then a fixed butterfly
// Every fp64 sum is therefore taken in an order fixed by (L, rows) alone: the same pair of states gives
// bit-identical sums whichever kernel path, chunking, batch or replica offset produced them.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace spgg {

// The planes of replica rep0 of the live state ([0]) and of replica 0 of the snapshot ([1]); replica y of a launch
// is y strides further on both sides.  S: word 0 of row 0 of the bit plane (rows pitchW words apart); R: column 0
// of row 0 of the R plane (rows pitchB elements apart); Q: site 0 (rows L * nq entries apart).
struct OvPlanes {
  int L, rows, pitchW, pitchB, nq, n_rep;
  const uint32_t *S[2];
  const void *R[2], *Q[2];
  long long bits_stride, plane_stride, q_stride;   // words, R elements and Q entries per replica
};

// Rows per tile and tiles per replica of a lattice of `rows` x L sites
int overlap_rows_per_tile(int L, int rows);
size_t overlap_scratch_bytes(int L, int rows, int n_rep, int m);

// Host launcher (spgg_overlap.cu), instantiated for ModeF32I8, ModeF32F and ModeF64; synchronous on the legacy
// default stream.  want_r / want_q select the channels, m = want_r + want_q * nq.  rq: host, 2 * n_rep int8
// quanta, the live replicas' then the snapshot's.  scratch: device memory of overlap_scratch_bytes bytes.
// counts, changed, diffs: host arrays in the layouts of include/spgg.h (changed / diffs unread when m == 0).
template <class Md>
cudaError_t launch_overlap(const OvPlanes &p, bool want_r, bool want_q, const double *rq, void *scratch,
                           int64_t *counts, int64_t *changed, double *diffs);

}  // namespace spgg
