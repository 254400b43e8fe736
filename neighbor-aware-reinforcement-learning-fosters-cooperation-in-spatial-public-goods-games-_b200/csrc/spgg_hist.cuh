// Value distributions of replicas rep0 .. rep0 + n_rep - 1 (spgg_value_ranges / spgg_histograms, include/spgg.h):
// per channel (R, then the nq Q entries) and class (all sites, cooperators) the exact min / max, the counts of
// np.histogram over uniform bins, and per state the number of sites whose greedy action is C.
//
// One streaming pass per call over the planes spgg_state_digest reads, one launch for all replicas (grid.y):
//   k_hist_range  per thread fp64 min / max in registers, fmin / fmax across the warp, then 64-bit integer
//                 atomics on an order-preserving map of the bit patterns (shared, then global): exact
//   k_hist        per CTA privatised uint32 counts in shared memory.  Lanes that land in the same (bin, class)
//                 are grouped by __match_any_sync and their leader does one shared atomic for the group, so a
//                 uniform lattice costs one atomic per warp and channel; at the end one 64-bit global add per
//                 non-zero bin per CTA.  int8-stored R takes at most 256 values: it is counted per int8 code
//                 and k_hist_codes maps each code to its bin once per call, with the same NumPy rule on
//                 code * quantum.  The greedy-policy counts are per-thread registers, added at the end.
// All results are integer sums or exact extremes, so they do not depend on scheduling.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace spgg {

constexpr int HIST_MAX_BINS = 1024;

// The planes of replica rep0 (replica rep0 + y of a launch is y strides further on).  S: word 0 of row 0 of the
// bit plane (rows pitchW words apart); R: column 0 of row 0 of the R plane (rows pitchB elements apart); Q: site
// 0 (rows L * nq entries apart).
struct HistPlanes {
  int L, rows, pitchW, pitchB, nq, n_rep;
  const uint32_t *S;
  const void *R, *Q;
  long long bits_stride, plane_stride, q_stride;   // words, R elements and Q entries per replica
};

// Host launchers (spgg_hist.cu), instantiated for ModeF32I8, ModeF32F and ModeF64; synchronous on the legacy
// default stream.  want_r / want_q select the channels, m = want_r + want_q * nq.  rq: host, the int8 quantum of
// each replica (ModeF32I8 stores R as int8 units x rq).  scratch: device memory of hist_scratch_bytes(n_rep, m,
// n_bins) bytes.  minmax, edges, counts, policy: host arrays in the layouts of include/spgg.h.
size_t hist_scratch_bytes(int n_rep, int m, int n_bins);
template <class Md>
cudaError_t launch_value_ranges(const HistPlanes &p, bool want_r, bool want_q, const double *rq, void *scratch,
                                double *minmax);
template <class Md>
cudaError_t launch_histograms(const HistPlanes &p, bool want_r, bool want_q, int n_bins, const double *edges,
                              const double *rq, void *scratch, int64_t *counts, int64_t *policy);

}  // namespace spgg
