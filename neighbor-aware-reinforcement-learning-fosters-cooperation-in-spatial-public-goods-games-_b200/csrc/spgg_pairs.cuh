// Strategy pair counts of one replica's bit plane (spgg_pair_counts, include/spgg.h): for numpy axis ax and
// every offset d in 0..max_d, over the torus, the sites x that cooperate together with x + d e_ax, and the
// sites whose partner holds the other strategy.  Bit 1 = defector, so with a the word of x and b the word of
// the partners, the counts are popc(~(a | b)) and popc(a ^ b) over the valid columns; d = 0 gives {n_C, 0}.
//
// Two kernels, each one launch, no atomics per word:
//   k_pairs_rows   ax 0, partner (i + d, j): one CTA per 32-word column band x 64 offsets x row segment;
//                  it stages bands of 32 rows and the 95 partner rows they need in shared memory, and every
//                  thread (one word column) evaluates 8 offsets per staged row from registers
//   k_pairs_cols   ax 1, partner (i, j + d): one CTA per 256 offsets x row segment; each row is staged as
//                  its periodic bit stream (the row, then its first max_d + 64 bits again: the ghost words
//                  are whole-word copies and are not that stream when L % 32 != 0), so the 32 partners of
//                  word w at offset d are one funnel shift of two stream words; a warp holds 32 offsets
// Counts stay in registers for the CTA's whole row segment, then one warp reduction, one shared 64-bit
// atomic per warp and one global 64-bit atomicAdd per (CTA, offset, kind): integer sums, so the result does
// not depend on scheduling.
//
// Row strips: the partners of ax 0 reach max_d rows past a strip's last row.  Each strip writes a record of
// its first min(max_d, rows) rows (PAIR_REC_HDR header words, then max_rows packed rows of nW words, spare
// bits cleared); from the gathered records of all ranks the strip assembles the max_d rows that follow it
// (the "tail") and counts the pairs whose site x it owns.  The counts of the strips add up to the lattice's.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace spgg {

constexpr int PAIR_REC_HDR = 8;              // header words, keeps the packed rows 32-byte aligned
constexpr int PAIR_REC_MAGIC = 0x53505231;   // "SPR1"
enum { PAIR_H_MAGIC, PAIR_H_L, PAIR_H_ROW0, PAIR_H_ROWS, PAIR_H_MAXD, PAIR_H_MAXROWS, PAIR_H_NROWS };
inline long long pair_record_bytes(int L, int max_rows) { return 4ll * (PAIR_REC_HDR + (long long)max_rows * ((L + 31) / 32)); }

// Host launchers (spgg_pairs.cu), synchronous on the legacy default stream.  S points at word 0 of row 0 of
// one replica's bit plane, rows pitchW words apart.  tail holds the max_d rows that follow row rows-1
// (tail_pitch words apart); a whole lattice passes S and pitchW, rows == L.  counts: device scratch of
// 2*(max_d+1)*2 uint64; out: the host result in the ABI's layout.
cudaError_t launch_pair_counts(const uint32_t *S, int pitchW, int rows, int L, const uint32_t *tail, int tail_pitch,
                               int max_d, unsigned long long *counts, int64_t *out);
// this strip's record (rows from S, as above) into dev_record
cudaError_t launch_pair_record(const uint32_t *S, int pitchW, int row0, int rows, int L, int max_d, int max_rows,
                               void *dev_record);

}  // namespace spgg
