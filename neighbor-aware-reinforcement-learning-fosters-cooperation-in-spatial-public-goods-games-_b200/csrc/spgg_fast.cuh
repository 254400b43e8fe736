// Fast path of the fused SPGG step for sm_100a: throughput mode (fp32 float4 Q, int8 R,
// one-byte reward code, bit-packed strategies, Philox draws) on lattices whose side is a
// multiple of 128.  Same arithmetic, bit for bit, as k_step<ModeF32I8,...> in
// spgg_kernels.cuh (tests/test_gpu_parity.py::test_fast_path_equals_general_path); what
// differs is how the work is laid out on the SM:
//
//   * the three halo'd tiles a CTA needs (reward codes, reputations, strategy bits) are
//     staged by TMA 2-D tile loads (cp.async.bulk.tensor, one elected thread, mbarrier
//     completion), double-buffered so the next tile lands while this one is computed; the
//     lattices carry physical ghost rows/columns, so the boxes never wrap
//   * the byte-valued stencils (cooperators per group N, their 5-group sum SigmaN, the
//     reputation state) are computed 4 sites per 32-bit word with SWAR adds
//   * Q goes HBM -> registers -> HBM as coalesced 16-byte accesses, four in flight per thread
//   * statistics are exact packed integer counters plus fp32 partial sums per thread,
//     folded in a fixed order (deterministic)
//
// Reference lines are cited at the arithmetic, as in spgg_kernels.cuh.
#pragma once
#include <cuda.h>

#include "spgg_kernels.cuh"

namespace spgg {

constexpr int FTR = 16;            // tile rows
constexpr int FROWB = 160;         // staged row bytes of code / R: 16 ghost + 128 + 16 ghost
constexpr int FROWW = FROWB / 4;   // the same in 32-bit words
constexpr int FSROWB = 48;         // staged row bytes of strategy bits: 16 + 16 + 16
constexpr int FTHREADS = 256;

template <int M>
struct FastSmem {
  static constexpr int kRowsCR = FTR + 2 * M;  // staged rows of code / R
  static constexpr int kRowsS = FTR + 4;       // staged rows of strategy bits (halo 2)
  static constexpr int kStageCode = 0;
  static constexpr int kStageR = (kRowsCR * FROWB + 127) / 128 * 128;
  static constexpr int kStageS = kStageR + (kRowsCR * FROWB + 127) / 128 * 128;
  static constexpr int kStageBytes = kStageS + (kRowsS * FSROWB + 127) / 128 * 128;
  static constexpr int kTxBytes = 2 * kRowsCR * FROWB + kRowsS * FSROWB;
  // outputs of a tile, written back by TMA tile stores
  static constexpr int kOutCode = 2 * kStageBytes;               // FTR x 128 bytes
  static constexpr int kOutR = kOutCode + FTR * TC;
  static constexpr int kOutS = kOutR + FTR * TC;                 // FTR x 16 bytes
  // work planes, all with the staged row geometry (row r, word w <-> tile cols 4(w-4)..4(w-4)+3),
  // one guard row before the first so flat stencils may read one word before a plane
  static constexpr int kOffC = kOutS + 256 + FROWB;              // cooperator flags, rows -2..FTR+1
  static constexpr int kOffVal = kOffC + (FTR + 4) * FROWB + FROWB;  // reward floats, rows -M..FTR+M-1 (one guard row after C)
  static constexpr int kOffTab = kOffVal + kRowsCR * FROWB * 4;
  static constexpr int kOffBar = kOffTab + 256 * 4;            // 2 tile barriers + kQBufs Q barriers per warp (<= 40)
  static constexpr int kOffFlag = kOffBar + 40 * 8;            // "last CTA" flag
  static constexpr int kOffRc = kOffFlag + 16;                 // RepConst copy
  static constexpr int kOffRed = (kOffRc + (int)sizeof(RepConst) + 127) / 128 * 128;  // final reduction [8][NSTAT]
  // per warp: kQBufs buffers of kRowsPerWarp row segments of 128 float4 (2 KB each), landed by one
  // TMA tile load with the 128-byte swizzle (1024-byte aligned) and written back in place
  static constexpr int kRowsPerWarp = FTR / (FTHREADS / 32);
  static constexpr int kQBufs = 2;
  static constexpr int kQBufBytes = kRowsPerWarp * TC * 16;
  static constexpr int kOffQ = (kOffRed + 8 * NSTAT * 8 + 1023) / 1024 * 1024;
  static constexpr int kTotal = kOffQ + (FTHREADS / 32) * kQBufs * kQBufBytes + 1024;  // + base alignment slack
};

// ---- PTX helpers: mbarrier + TMA (Blackwell guide: TMA tile load with mbarrier signalling)
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  uint32_t done;
  uint32_t spins = 0;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (!done && ++spins > (1u << 28)) __trap();  // a lost TMA must not hang the GPU
  } while (!done);
}
__device__ __forceinline__ void tma_load_3d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0,
                                            int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// contiguous global -> shared bulk copy (16-byte aligned, size multiple of 16)
__device__ __forceinline__ void bulk_load_1d(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap *map, const void *src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(map), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
// 4-D tile load / store of the Q table (swizzled), with an L2 eviction-priority hint: Q is
// streamed once per iteration and must not push the small halo'd planes out of L2
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void tma_load_4d_hint(void *dst, const CUtensorMap *map, uint64_t *bar, int c0,
                                                 int c1, int c2, int c3, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5, %6}], [%2], %7;"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(pol)
      : "memory");
}
__device__ __forceinline__ void tma_store_4d_hint(const CUtensorMap *map, const void *src, int c0, int c1,
                                                  int c2, int c3, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.4d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3, %4, %5}], [%1], %6;"
      ::"l"(map), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(pol)
      : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_read_n() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// bytes of the column-shifted neighbours of a 4-site word
__device__ __forceinline__ uint32_t sh_l1(uint32_t prev, uint32_t cur) { return __byte_perm(prev, cur, 0x6543); }
__device__ __forceinline__ uint32_t sh_r1(uint32_t cur, uint32_t next) { return __byte_perm(cur, next, 0x4321); }
__device__ __forceinline__ uint32_t sh_2(uint32_t a, uint32_t b) { return __byte_perm(a, b, 0x5432); }

struct FastMaps {
  CUtensorMap ld_code, ld_R, ld_S;  // halo'd tile loads from the planes of iteration j
  CUtensorMap st_code, st_R, st_S;  // tile stores into the planes of iteration j+1
  // Q table as (128 B = 8 sites, L/8, rows, replicas), 128-byte swizzle: read from q_ld, written to q_st
  // (the same buffer when the handle updates Q in place, the two halves of a ping-pong pair when a
  // failed speculation of the global maximum must be able to re-run an iteration from its inputs)
  CUtensorMap q_ld, q_st;
};

// UPD / SEL are compile-time so the four sites a thread handles per row form one straight-line
// block the scheduler can interleave.
// PART: the lattice side is a multiple of 32 but not of 128 - the last tile column is partial.  Its tiles
// are loaded and computed like any other (the bytes right of the ghost columns are zero, TMA zero-fills
// beyond a row, and the store maps end at column L so nothing lands outside the lattice); the lanes whose
// four sites lie beyond L ("phantom" lanes, whole 32-bit words because L is a multiple of 4) are kept out
// of every statistic and of the global maximum.
template <int M, bool ACTION, bool UPD, bool SEL, bool PART = false>
__device__ __forceinline__ void step_fast_body(const FastMaps &tm, const KArgs &a) {
  typedef FastSmem<M> SM;
  constexpr int NK = (M == 2) ? 12 : 4;
  constexpr bool upd = UPD, sel = SEL;
  const Geom &g = a.g;
  const int rep = blockIdx.x / g.ctas_per_rep, cta = blockIdx.x % g.ctas_per_rep;

  extern __shared__ __align__(1024) unsigned char smem_fast[];
  // the swizzled Q buffers need a 1024-byte aligned base; kTotal carries the slack
  unsigned char *smem = smem_fast + ((1024u - (smem_u32(smem_fast) & 1023u)) & 1023u);
  uint32_t *wC = reinterpret_cast<uint32_t *>(smem + SM::kOffC);
  float *sm_val = reinterpret_cast<float *>(smem + SM::kOffVal);
  float *sm_tab = reinterpret_cast<float *>(smem + SM::kOffTab);
  float *sm_ratio = sm_tab + 128;
  double *sm_red = reinterpret_cast<double *>(smem + SM::kOffRed);
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + SM::kOffBar);
  uint8_t *out_code = smem + SM::kOutCode;
  int8_t *out_R = reinterpret_cast<int8_t *>(smem + SM::kOutR);
  uint32_t *out_S = reinterpret_cast<uint32_t *>(smem + SM::kOutS);
  RepConst &s_rc = *reinterpret_cast<RepConst *>(smem + SM::kOffRc);
  int &s_is_last = *reinterpret_cast<int *>(smem + SM::kOffFlag);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#ifdef SPGG_TRACE
  unsigned long long t_start = 0;
  if (tid == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_start));
#endif
  for (int i = tid; i < (int)(sizeof(RepConst) / 4); i += FTHREADS)
    reinterpret_cast<uint32_t *>(&s_rc)[i] = reinterpret_cast<const uint32_t *>(a.rc + rep)[i];
  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  for (int i = tid; i < 128; i += FTHREADS) {
    sm_tab[i] = s_rc.rewtab[i];
    sm_ratio[i] = s_rc.ratiotab[i];
  }
  const RepConst &rc = s_rc;

  float4 *Qp = reinterpret_cast<float4 *>(a.Q) + (long long)rep * g.site_stride;

  float inv_den = 0.f, gm_used = 0.f;
  if (upd) {
    // spec: last iteration's maximum stands in for this one's until the launch has computed its own
    gm_used = a.spec ? a.gcarry[rep] : reinterpret_cast<const float *>(a.gmax)[(long long)rep * a.cap + a.rel];
    if (a.spec == 2) gm_used = 123.0f;   // test hook: a guess that is certainly wrong
    inv_den = __fdiv_rn(1.0f, __fadd_rn(gm_used, rc.leps_f));  // spgg.py:489 denominator
  }
  float gbest = 0.f;  // max over this thread's sites of the best signed neighbour difference (>= 0 kept)
  const uint32_t thr = sel ? a.thr_tab[(long long)(a.rel + 1) * g.n_rep + rep] : 0u;
  const float alpha = rc.alpha_f, gamma = rc.gamma_f, kappa = rc.kappa_f;
  // byte-parallel reputation update: steps beyond the width of [R_min, R_max] saturate alike
  // (gain and loss are non-negative on this path, spgg_create checks)
  const int g31 = min(rc.gain_i, 31), l31 = min(rc.loss_i, 31);
  const uint32_t r_dsum = (uint32_t)(g31 + l31);
  const uint32_t r_k = (uint32_t)(32 - l31) * 0x01010101u;
  const uint32_t r_lo = (uint32_t)(rc.rmin_i + 48) * 0x01010101u, r_hi = (uint32_t)(rc.rmax_i + 48) * 0x01010101u;
  const bool has_ratio = rc.has_ratio != 0;

  // per-thread statistics: exact 32-bit integer counters + fp32 partial sums.
  // class = C_old*2 + coop (spgg.py:383,419-420)
  uint32_t cls_n[4] = {0, 0, 0, 0}, cls_sn[4] = {0, 0, 0, 0};  // counts and sums of SigmaN per class
  uint32_t grp[6] = {0, 0, 0, 0, 0, 0};                         // #groups with k defectors
  uint32_t pk_best = 0;   // low 16: #best>0, high 16: ... with a second-order arg-max
  uint32_t n_sel = 0;
  int sum_r = 0;
  float sq0 = 0.f, sq1 = 0.f, sq2 = 0.f, sq3 = 0.f, sc0 = 0.f, sc1 = 0.f, sc2 = 0.f, sc3 = 0.f;
  float s_ni = 0.f, s_ratio = 0.f;

  const int n_tiles = g.n_tx * g.n_ty;
  // tile walk without divisions: (ty, tx) advance by (d_ty, d_tx) with a carry
  const int d_ty = g.ctas_per_rep / g.n_tx, d_tx = g.ctas_per_rep - d_ty * g.n_tx;
  const int d_skew = (d_tx + d_ty) % g.n_tx;  // advance of the skewed column per step (one division per launch)
  auto issue = [&](int ty_, int tx_, int st) {
    const int r0 = ty_ * FTR, c0 = tx_ * TC;
    unsigned char *base = smem + st * SM::kStageBytes;
    mbar_expect_tx(&bars[st], SM::kTxBytes);
    tma_load_3d(base + SM::kStageCode, &tm.ld_code, &bars[st], c0, r0 + GH - M, rep);
    tma_load_3d(base + SM::kStageR, &tm.ld_R, &bars[st], c0, r0 + GH - M, rep);
    tma_load_3d(base + SM::kStageS, &tm.ld_S, &bars[st], c0 >> 3, r0 + GH - 2, rep);
  };
  // the column of a tile is skewed by its row ((ty, txs) -> tx = (txs + ty) mod n_tx) so that the
  // tiles of one CTA sweep all columns: the edge tiles (periodic ghost copies) spread over all CTAs
  int ty = cta / g.n_tx, txs = cta - ty * g.n_tx;
  int tx = (txs + ty) % g.n_tx;
  if (tid == 0 && cta < n_tiles) issue(ty, tx, 0);

  // per-warp Q pipeline: the 2 KB row segment (128 float4) a warp handles next is fetched by one
  // TMA tile load (128-byte swizzle) into one of the warp's kQBufs buffers while the warp works
  // on the current one; results are written back in place and leave by a TMA tile store.
  uint64_t *qbar = bars + 2 + warp * SM::kQBufs;
  unsigned char *sQ = smem + SM::kOffQ + warp * (SM::kQBufs * SM::kQBufBytes);
  const uint64_t pol = l2_evict_first_policy();
  if (lane == 0) {
#pragma unroll
    for (int b = 0; b < SM::kQBufs; ++b) mbar_init(&qbar[b], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  auto q_issue = [&](int col8, int row, int buf) {
    mbar_expect_tx(&qbar[buf], SM::kQBufBytes);
    tma_load_4d_hint(sQ + buf * SM::kQBufBytes, &tm.q_ld, &qbar[buf], 0, col8, row, rep, pol);
  };
  // lane l owns the four consecutive sites 4l..4l+3 of a row segment: site s sits in 128-byte
  // line s>>3 at 16-byte chunk (s&7) ^ (line&7) (CU_TENSOR_MAP_SWIZZLE_128B)
  int qoff[4];
#pragma unroll
  for (int k = 0; k < 4; ++k)
    qoff[k] = (lane >> 1) * 128 + ((((lane & 1) * 4 + k) ^ ((lane >> 1) & 7)) << 4);
  // a warp owns kRowsPerWarp adjacent rows of every tile: one load, one store, one wait per tile
  if (lane == 0 && cta < n_tiles) q_issue((tx * TC) >> 3, ty * FTR + warp * SM::kRowsPerWarp, 0);

  int tiles_done = 0, stage = 0;
  for (int tile = cta; tile < n_tiles; tile += g.ctas_per_rep, ++tiles_done, stage ^= 1) {
    const int r0 = ty * FTR, c0 = tx * TC;
    // coordinates of this CTA's next tile
    int nty = ty + d_ty, ntxs = txs + d_tx, ntx = tx + d_skew;
    if (ntxs >= g.n_tx) { ntxs -= g.n_tx; ++nty; ++ntx; }
    if (ntx >= g.n_tx) ntx -= g.n_tx;  // tx + d_skew + 1 < 2 n_tx, so this is (ntxs + nty) mod n_tx without a division
    const bool has_next = tile + g.ctas_per_rep < n_tiles;
    // prefetch the next tile into the other stage (its readers passed the barrier that
    // closes the previous iteration)
    if (tid == 0) {
      if (has_next) issue(nty, ntx, stage ^ 1);
      if (sel) tma_store_wait_read();  // the previous tile's stores have left out_*
    }
    mbar_wait(&bars[stage], (uint32_t)(tiles_done >> 1) & 1u);  // a stage completes once every 2 tiles
    const bool lv = !PART || (c0 + 4 * lane < g.L);            // this lane's four sites exist
    const uint32_t vm = lv ? 0x01010101u : 0u;
    const unsigned char *st_base = smem + stage * SM::kStageBytes;
    const uint32_t *st_code = reinterpret_cast<const uint32_t *>(st_base + SM::kStageCode);
    const uint32_t *st_R = reinterpret_cast<const uint32_t *>(st_base + SM::kStageR);
    const uint32_t *st_S = reinterpret_cast<const uint32_t *>(st_base + SM::kStageS);

    // ---- phase A1: cooperator flags as bytes; one thread expands one staged bit word
    // (32 sites) into 8 words of 4 flag bytes.  Rows -2..FTR+1, staged words 3..8.
    // (the upper warps take this, the group statistics below go to warps 2-3: the flat loops
    // that follow are spread over all warps, so nobody arrives late at the barrier)
    const int t1 = tid - (FTHREADS - 128);
    if (t1 >= 0 && t1 < (FTR + 4) * 6) {
      const int row = t1 / 6, bw = t1 - row * 6 + 3;
      const uint32_t bits = ~st_S[row * (FSROWB / 4) + bw];  // 1 = cooperator
      uint32_t *dst = wC + row * FROWW + (bw - 4) * 8 + 4;
      if (bw == 3) {         // columns -4..-1 only
        dst[7] = ((bits >> 28) * 0x00204081u) & 0x01010101u;
      } else if (bw == 8) {  // columns 128..131 only
        dst[0] = ((bits & 0xFu) * 0x00204081u) & 0x01010101u;
      } else {
        uint4 lo, hi;
        lo.x = (((bits >> 0) & 0xFu) * 0x00204081u) & 0x01010101u;
        lo.y = (((bits >> 4) & 0xFu) * 0x00204081u) & 0x01010101u;
        lo.z = (((bits >> 8) & 0xFu) * 0x00204081u) & 0x01010101u;
        lo.w = (((bits >> 12) & 0xFu) * 0x00204081u) & 0x01010101u;
        hi.x = (((bits >> 16) & 0xFu) * 0x00204081u) & 0x01010101u;
        hi.y = (((bits >> 20) & 0xFu) * 0x00204081u) & 0x01010101u;
        hi.z = (((bits >> 24) & 0xFu) * 0x00204081u) & 0x01010101u;
        hi.w = ((bits >> 28) * 0x00204081u) & 0x01010101u;
        *reinterpret_cast<uint4 *>(dst) = lo;
        *reinterpret_cast<uint4 *>(dst + 4) = hi;
      }
    }
    // ---- phase A2: reward of every staged code (flat over the staged plane, 4 codes per thread)
    if (upd) {
      for (int e = tid; e < SM::kRowsCR * FROWW; e += FTHREADS) {
        const uint32_t cw = st_code[e];
        float4 v;
        v.x = sm_tab[(cw >> 1) & 0x7Fu];
        v.y = sm_tab[(cw >> 9) & 0x7Fu];
        v.z = sm_tab[(cw >> 17) & 0x7Fu];
        v.w = sm_tab[(cw >> 25) & 0x7Fu];
        *reinterpret_cast<float4 *>(sm_val + e * 4) = v;
      }
    }
    // ---- phase A4: integer statistics of iteration j straight from the staged words
    if (upd) {
      // defectors per 5-site group (spgg.py:586-592), bit-sliced: one thread = 32 sites
      const int t2 = tid - 64;
      if (t2 >= 0 && t2 < FTR * 4 && (!PART || (c0 >> 5) + (t2 & 3) < ((g.L + 31) >> 5))) {
        const int row = (t2 >> 2) + 2, bw = (t2 & 3) + 4;
        const uint32_t *bp = st_S + row * (FSROWB / 4) + bw;
        const uint32_t c = bp[0], u = bp[-(FSROWB / 4)], d = bp[FSROWB / 4];
        const uint32_t l = (c << 1) | (bp[-1] >> 31), r = (c >> 1) | (bp[1] << 31);
        const uint32_t s1 = c ^ u ^ d, c1 = (c & u) | (d & (c | u));
        const uint32_t b0 = s1 ^ l ^ r, c2 = (s1 & l) | (r & (s1 | l));
        const uint32_t b1 = c1 ^ c2, b2 = c1 & c2;
        grp[0] += __popc(~b0 & ~b1 & ~b2); grp[1] += __popc(b0 & ~b1 & ~b2);
        grp[2] += __popc(~b0 & b1 & ~b2);  grp[3] += __popc(b0 & b1 & ~b2);
        grp[4] += __popc(~b0 & ~b1 & b2);  grp[5] += __popc(b0 & ~b1 & b2);
      }
    }
    __syncthreads();
    // ---- main phase: warp = one 128-site row segment, lane = 4 consecutive sites, so every
    // byte plane is read one 32-bit word and every reward row one float4 per lane
    const uint8_t *bCode = reinterpret_cast<const uint8_t *>(st_code);
    // fetch this warp's rows of the CTA's next tile into the other buffer (its previous content,
    // the rows of the previous tile, left by a tile store issued a whole tile ago)
    const int qb = stage;
    __syncwarp();
    if (lane == 0) {
      if (upd) tma_store_wait_read_n<0>();
      if (has_next) q_issue((ntx * TC) >> 3, nty * FTR + warp * SM::kRowsPerWarp, qb ^ 1);
    }
    mbar_wait(&qbar[qb], (uint32_t)(tiles_done >> 1) & 1u);
#pragma unroll
    for (int r2 = 0; r2 < SM::kRowsPerWarp; ++r2) {
      const int rr = warp * SM::kRowsPerWarp + r2;
      uint32_t w4[4] = {0, 0, 0, 0};
      if (sel) {
        // counter = (column / 4, global row, iteration, 0); one call -> this lane's 4 sites
        philox4x32_10_keys((uint32_t)((c0 >> 2) + lane), (uint32_t)(g.row0 + r0 + rr),
                           (uint32_t)(a.j + 1), 0u, s_rc.pkeys, w4);
      }
      const int wo = rr * FROWW + (CPAD / 4) + lane;      // word of (rr, 4*lane) in a tile-row-indexed plane
      const uint32_t RW = st_R[wo + M * FROWW];
      const uint32_t CW = wC[wo + 2 * FROWW];
      // post-action state of the 4 sites (= pre-action state of the next iteration, spgg.py:409/423)
      uint32_t StW;
      if constexpr (ACTION) {
        StW = CW;                                          // own previous action (spgg.py:291)
      } else {
        // reputation state (spgg.py:292-307): v = R + 16 in each byte (R in [-16, 15] units: spgg_set_state sends a wider R to k_step's
        // select, which clips it into [R_min, R_max], or rejects it on a strip); sum of n values v > 16 n  <=>  sum of R > 0
        const uint32_t *rp = st_R + wo + M * FROWW;
        auto bias = [](uint32_t x) { return (x ^ 0x10101010u) & 0x1F1F1F1Fu; };
        const uint32_t c = bias(RW), l = bias(rp[-1]), r = bias(rp[1]);
        const uint32_t u1 = bias(rp[-FROWW]), d1 = bias(rp[FROWW]);
        uint32_t sumA = c + u1 + d1 + sh_l1(l, c) + sh_r1(c, r);
        if constexpr (M == 1) {
          // 5 values in [1,31]: sum <= 155; sum > 80 <=> bit 7 of (sum + 47)
          StW = ((sumA + 0x2F2F2F2Fu) >> 7) & 0x01010101u;
        } else {
          const uint32_t ul = bias(rp[-FROWW - 1]), ur = bias(rp[-FROWW + 1]);
          const uint32_t dl = bias(rp[FROWW - 1]), dr = bias(rp[FROWW + 1]);
          const uint32_t sumB = bias(rp[-2 * FROWW]) + bias(rp[2 * FROWW]) + sh_2(l, c) + sh_2(c, r) +
                                sh_l1(ul, u1) + sh_r1(u1, ur) + sh_l1(dl, d1);
          sumA += sh_r1(d1, dr);  // 6 values <= 186; sumB: 7 values <= 217
          // 16-bit lanes: total > 16*13 = 208
          const uint32_t lo = (sumA & 0x00FF00FFu) + (sumB & 0x00FF00FFu);
          const uint32_t hi = ((sumA >> 8) & 0x00FF00FFu) + ((sumB >> 8) & 0x00FF00FFu);
          const uint32_t flo = ((lo + (0x8000u - 209u) * 0x00010001u) >> 15) & 0x00010001u;
          const uint32_t fhi = ((hi + (0x8000u - 209u) * 0x00010001u) >> 15) & 0x00010001u;
          StW = flo | (fhi << 8);
        }
      }
      sum_r = __dp4a((int)RW, (int)vm, sum_r);              // spgg.py:394
      uint32_t codeW = 0;
      float vc[4], vu[4], vd[4], vl[2], vr[2], vu2[4], vd2[4], vul = 0.f, vur = 0.f, vdl = 0.f, vdr = 0.f;
      const int vb = (rr + M) * FROWB + CPAD + 4 * lane;  // float / byte index of (rr, 4*lane) in the staged planes
      if (upd) {
        codeW = st_code[wo + M * FROWW];
        {  // integer statistics of iteration j: class = C_old*2 + coop (spgg.py:383,419-420), 4 sites per dp4a
          const uint32_t Cb = (codeW >> 2) & 0x01010101u, Ab = (codeW >> 1) & 0x01010101u;
          const uint32_t m3 = Cb & Ab & vm, m2 = (Cb & vm) ^ m3, m1 = (Ab & vm) ^ m3, m0 = vm & ~(Cb | Ab);
          const uint32_t sn = (codeW >> 3) & 0x1F1F1F1Fu;
          cls_n[0] = __dp4a(m0, 0x01010101u, cls_n[0]); cls_sn[0] = __dp4a(sn, m0, cls_sn[0]);
          cls_n[1] = __dp4a(m1, 0x01010101u, cls_n[1]); cls_sn[1] = __dp4a(sn, m1, cls_sn[1]);
          cls_n[2] = __dp4a(m2, 0x01010101u, cls_n[2]); cls_sn[2] = __dp4a(sn, m2, cls_sn[2]);
          cls_n[3] = __dp4a(m3, 0x01010101u, cls_n[3]); cls_sn[3] = __dp4a(sn, m3, cls_sn[3]);
        }
        const float4 c4 = *reinterpret_cast<const float4 *>(sm_val + vb);
        const float4 u4 = *reinterpret_cast<const float4 *>(sm_val + vb - FROWB);
        const float4 d4 = *reinterpret_cast<const float4 *>(sm_val + vb + FROWB);
        vc[0] = c4.x; vc[1] = c4.y; vc[2] = c4.z; vc[3] = c4.w;
        vu[0] = u4.x; vu[1] = u4.y; vu[2] = u4.z; vu[3] = u4.w;
        vd[0] = d4.x; vd[1] = d4.y; vd[2] = d4.z; vd[3] = d4.w;
        if constexpr (M == 2) {
          const float2 l2 = *reinterpret_cast<const float2 *>(sm_val + vb - 2);
          const float2 r2 = *reinterpret_cast<const float2 *>(sm_val + vb + 4);
          vl[0] = l2.x; vl[1] = l2.y; vr[0] = r2.x; vr[1] = r2.y;
          const float4 uu = *reinterpret_cast<const float4 *>(sm_val + vb - 2 * FROWB);
          const float4 dd = *reinterpret_cast<const float4 *>(sm_val + vb + 2 * FROWB);
          vu2[0] = uu.x; vu2[1] = uu.y; vu2[2] = uu.z; vu2[3] = uu.w;
          vd2[0] = dd.x; vd2[1] = dd.y; vd2[2] = dd.z; vd2[3] = dd.w;
          vul = sm_val[vb - FROWB - 1]; vur = sm_val[vb - FROWB + 4];
          vdl = sm_val[vb + FROWB - 1]; vdr = sm_val[vb + FROWB + 4];
        } else {
          vl[0] = 0.f; vl[1] = sm_val[vb - 1]; vr[0] = sm_val[vb + 4]; vr[1] = 0.f;
        }
      }
      unsigned char *qbuf = sQ + qb * SM::kQBufBytes + r2 * (TC * 16);
      // The four Q entries of a site stay in the landed segment: the entry being updated and
      // the row of the next state are addressed there (load/store pipe) instead of being
      // selected in registers - the integer/select pipe is the busy one in this loop.
      // Stages (all loads of a stage before the stores of the next, for all four sites):
      //   1 gather   2 arithmetic   3 write Q[s][a]   4 re-read the updated entries: statistics, greedy action
      uint32_t coopW = 0, rnewW = 0;
      float qfin[4];
      int eidx[4];
      const uint32_t rowoffW = StW << 3;  // byte offset of row s' inside a site's 16 bytes, 4 sites
      // per byte: the TD write lands in the row of s' (s' == s) and it is the C / the D entry
      const uint32_t coopCW = (codeW >> 1) & 0x01010101u;
      const uint32_t hitW = ~(StW ^ codeW) & 0x01010101u;
      const uint32_t hitCW = hitW & coopCW, hitDW = hitW ^ hitCW;
      if (upd) {
        float qe[4], na[4], nb_[4];
        // byte offset of Q[s][a] (a = !coop) inside a site's 16 bytes: 4 * (2 s + a), 4 sites at once
        const uint32_t eoffW = ((codeW & 0x01010101u) << 3) | ((((codeW >> 1) & 0x01010101u) ^ 0x01010101u) << 2);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const unsigned char *qs = qbuf + qoff[k];
          eidx[k] = (int)__byte_perm(eoffW, 0, 0x4440 + k);
          qe[k] = *reinterpret_cast<const float *>(qs + eidx[k]);
          const float2 nrow = *reinterpret_cast<const float2 *>(qs + __byte_perm(rowoffW, 0, 0x4440 + k));  // pre-update row of s'
          na[k] = nrow.x; nb_[k] = nrow.y;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint32_t code = (codeW >> (8 * k)) & 0xFFu;
          const float vx = vc[k];
          // neighbour-aware term inputs: spgg.py:486-494, offsets in the order of spgg.py:479-485
          // ((dx,dy) names the site (i-dx, j-dy)); the first arg-max wins
          float nv[NK];
          int no[NK];  // byte offset of the neighbour's code relative to this site's
          nv[0] = vu[k]; no[0] = -FROWB;                                // (1,0)
          nv[1] = vd[k]; no[1] = FROWB;                                 // (-1,0)
          nv[2] = (k == 0) ? vl[1] : vc[(k + 3) & 3]; no[2] = -1;       // (0,1)
          nv[3] = (k == 3) ? vr[0] : vc[(k + 1) & 3]; no[3] = 1;        // (0,-1)
          if constexpr (M == 2) {
            nv[4] = vu2[k]; no[4] = -2 * FROWB;                         // (2,0)
            nv[5] = vd2[k]; no[5] = 2 * FROWB;                          // (-2,0)
            nv[6] = (k == 0) ? vl[0] : (k == 1) ? vl[1] : vc[(k + 2) & 3]; no[6] = -2;   // (0,2)
            nv[7] = (k == 2) ? vr[0] : (k == 3) ? vr[1] : vc[(k + 2) & 3]; no[7] = 2;    // (0,-2)
            nv[8] = (k == 0) ? vul : vu[(k + 3) & 3]; no[8] = -FROWB - 1;                // (1,1)
            nv[9] = (k == 3) ? vur : vu[(k + 1) & 3]; no[9] = -FROWB + 1;                // (1,-1)
            nv[10] = (k == 0) ? vdl : vd[(k + 3) & 3]; no[10] = FROWB - 1;               // (-1,1)
            nv[11] = (k == 3) ? vdr : vd[(k + 1) & 3]; no[11] = FROWB + 1;               // (-1,-1)
          }
          float best = __fsub_rn(nv[0], vx);
          int boff = no[0];
          bool second = false;
#pragma unroll
          for (int q = 1; q < NK; ++q) {
            const float d = __fsub_rn(nv[q], vx);
            if (d > best) { best = d; boff = no[q]; if constexpr (M == 2) second = (q >= 4); }
          }
          if (lv) gbest = fmaxf(gbest, best);
          const bool same = ((((uint32_t)bCode[vb + k + boff] ^ code) >> 1) & 1u) == 0u;   // a* == a
          const float td = __fsub_rn(__fmaf_rn(gamma, fmaxf(na[k], nb_[k]), vx), qe[k]);  // algorithms.py:128
          const float qtd = __fmaf_rn(alpha, td, qe[k]);                                   // algorithms.py:131
          const float lam = __fmul_rn(__fmul_rn(kappa, fmaxf(0.0f, best)), inv_den);       // spgg.py:489
          const float nu = same ? lam : -lam;                                              // spgg.py:494-495
          // TD error on the table after the TD write (spgg.py:446-473), for the NI statistic
          const float na2 = ((hitCW >> (8 * k)) & 1u) ? qtd : na[k];
          const float nb2 = ((hitDW >> (8 * k)) & 1u) ? qtd : nb_[k];
          const float td2 = __fsub_rn(__fmaf_rn(gamma, fmaxf(na2, nb2), vx), qtd);
          qfin[k] = __fadd_rn(qtd, nu);                                                    // spgg.py:509
          const float an = fabsf(nu);
          if (lv) {
            s_ni += __fdividef(an, fabsf(alpha * td2) + an + 1e-8f);             // x100 at the fold; spgg.py:512
            if (has_ratio) s_ratio += sm_ratio[code >> 1];  // zero for defecting codes
            if (best > 0.f) pk_best += second ? 0x10001u : 1u;
          }
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) *reinterpret_cast<float *>(qbuf + qoff[k] + eidx[k]) = qfin[k];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float4 qn = *reinterpret_cast<const float4 *>(qbuf + qoff[k]);   // after both updates
          const float m = ((codeW >> (8 * k + 2)) & 1u) ? 1.0f : 0.0f;           // was a cooperator
          if (lv) {
            sq0 += qn.x; sq1 += qn.y; sq2 += qn.z; sq3 += qn.w;                  // spgg.py:562-583
            sc0 = fmaf(m, qn.x, sc0); sc1 = fmaf(m, qn.y, sc1); sc2 = fmaf(m, qn.z, sc2); sc3 = fmaf(m, qn.w, sc3);
          }
        }
      }
      if (sel) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float2 grow = *reinterpret_cast<const float2 *>(
              qbuf + qoff[k] + __byte_perm(rowoffW, 0, 0x4440 + k));             // Q[s'] after the update
          const bool explore = (w4[k] >> 8) < thr;
          const int rnd = (int)(w4[k] & 1u);
          const int greedy = (grow.y > grow.x) ? 1 : 0;  // np.argmax, tie -> 0   algorithms.py:107
          const int a_new = explore ? rnd : greedy;      // algorithms.py:109
          coopW |= (uint32_t)(a_new ^ 1) << (8 * k);
        }
        // reputation update (spgg.py:321-323) for the 4 sites at once, bytes biased so that no
        // carry crosses a byte: x = R + 48 = (R + 16) + 32 + (coop ? gain : -loss), clamped
        uint32_t x = ((RW ^ 0x10101010u) & 0x1F1F1F1Fu) + coopW * r_dsum + r_k;   // in [2, 94]
        uint32_t m = ((((x | 0x80808080u) - r_lo) >> 7) & 0x01010101u) * 0xFFu;  // x >= lo
        x = (x & m) | (r_lo & ~m);
        m = ((((r_hi | 0x80808080u) - x) >> 7) & 0x01010101u) * 0xFFu;           // hi >= x
        x = (x & m) | (r_hi & ~m);
        rnewW = (x + 0x50505050u) ^ 0x80808080u;                                 // back to int8 bytes: x - 48
      }
      if (sel) {
        // reward code of iteration j+1: SigmaN<<3 | C_j<<2 | coop<<1 | state, 4 sites per word
        // SigmaN = cooperators summed over the 5 groups the site belongs to (spgg.py:23-36,
        // 373-377) = 5 C(x) + 2 (4 nearest + 4 diagonal) + (4 straight second neighbours), bytewise
        const uint32_t *cp = wC + wo + 2 * FROWW;
        const uint32_t cl = cp[-1], cr = cp[1];
        const uint32_t u1 = cp[-FROWW], ul = cp[-FROWW - 1], ur = cp[-FROWW + 1];
        const uint32_t d1 = cp[FROWW], dl = cp[FROWW - 1], dr = cp[FROWW + 1];
        const uint32_t ring = u1 + d1 + sh_l1(cl, CW) + sh_r1(CW, cr) + sh_l1(ul, u1) + sh_r1(u1, ur) +
                              sh_l1(dl, d1) + sh_r1(d1, dr);
        const uint32_t far4 = cp[-2 * FROWW] + cp[2 * FROWW] + sh_2(cl, CW) + sh_2(CW, cr);
        const uint32_t SNW = 5u * CW + 2u * ring + far4;
        const int oo = rr * (TC / 4) + lane;
        reinterpret_cast<uint32_t *>(out_code)[oo] = (SNW << 3) | (CW << 2) | (coopW << 1) | StW;
        reinterpret_cast<uint32_t *>(out_R)[oo] = rnewW;
        // strategy bits: this lane's 4 coop flags -> nibble; 8 lanes -> one 32-site word (bit = 1: defect)
        const uint32_t nib = lv ? (((coopW * 0x01020408u) >> 24) & 0xFu) : 0u;   // phantom lanes count as defecting bits nobody stores
        uint32_t coopbits = nib << ((lane & 7) * 4);
        coopbits |= __shfl_xor_sync(0xffffffffu, coopbits, 1);
        coopbits |= __shfl_xor_sync(0xffffffffu, coopbits, 2);
        coopbits |= __shfl_xor_sync(0xffffffffu, coopbits, 4);
        if ((lane & 7) == 0) {
          out_S[rr * 4 + (lane >> 3)] = ~coopbits;
          n_sel += __popc(coopbits);  // cooperating actions just chosen
        }
      }
    }
    if (upd) {
      fence_proxy_async();  // the updated rows become visible to the TMA engine
      __syncwarp();
      if (lane == 0) {
        tma_store_4d_hint(&tm.q_st, sQ + qb * SM::kQBufBytes, 0, c0 >> 3, r0 + warp * SM::kRowsPerWarp, rep, pol);
        tma_store_commit();
      }
    }
    if (sel) fence_proxy_async();  // make out_* visible to the TMA engine
    __syncthreads();               // everyone is done with this stage, the work planes and out_*
    if (sel) {
      if (tid == 0) {
        tma_store_3d(&tm.st_code, out_code, CPAD + c0, r0 + GH, rep);
        tma_store_3d(&tm.st_R, out_R, CPAD + c0, r0 + GH, rep);
        // a partial last tile stores its strategy words with the edge path below (it is an edge tile anyway):
        // the 16-byte box would have to be cut inside a 16-byte unit, which is not something to ask of TMA
        if (!PART || c0 + TC <= g.L) tma_store_3d(&tm.st_S, out_S, (WPAD * 4) + (c0 >> 3), r0 + GH, rep);
        tma_store_commit();
      }
      // periodic copies other tiles read: ghost columns / ghost rows, edge tiles only; just the
      // cells that have copies are visited (store_cell writes the cell and all its copies)
      const bool ecol0 = tx == 0, ecol1 = tx == g.n_tx - 1;
      const bool erow0 = g.wrap_rows && ty == 0, erow1 = g.wrap_rows && ty == g.n_ty - 1;
      // strips: the rows a neighbour GPU needs go straight into its ghost rows (peer-mapped planes)
      const bool prow0 = a.peer_code[0] != nullptr && ty == 0, prow1 = a.peer_code[1] != nullptr && ty == g.n_ty - 1;
      const bool edge = ecol0 || ecol1 || erow0 || erow1 || prow0 || prow1;
      if (edge) {
        uint8_t *code_out = reinterpret_cast<uint8_t *>(a.code_out) + (long long)rep * g.plane_stride;
        int8_t *R_out = reinterpret_cast<int8_t *>(a.R_out) + (long long)rep * g.plane_stride;
        uint32_t *S_out = a.S_out + (long long)rep * g.bits_stride;
        // items 0..2*FTR*GC-1: the GC first / last columns; then 2*GH*TC: the GH first / last rows
        for (int e = tid; e < 2 * FTR * GC + 2 * GH * TC; e += FTHREADS) {
          int rr, cc;
          bool on, peer = false;
          int side = 0;
          if (e < 2 * FTR * GC) {
            side = e >= FTR * GC;
            const int q = side ? e - FTR * GC : e;
            rr = q / GC;
            const int wl = PART ? min(TC, g.L - c0) : TC;        // columns of this tile that exist
            cc = side ? wl - GC + (q % GC) : q % GC;
            on = side ? ecol1 : ecol0;
          } else {
            const int q0 = e - 2 * FTR * GC;
            side = q0 >= GH * TC;
            const int q = side ? q0 - GH * TC : q0;
            rr = side ? FTR - GH + q / TC : q / TC;
            cc = q % TC;
            const bool exists = !PART || c0 + cc < g.L;          // partial last tile column: columns beyond the lattice
            on = exists && (side ? erow1 : erow0);
            peer = exists && (side ? prow1 : prow0);
          }
          const int o = rr * TC + cc;
          if (on) {
            store_cell<uint8_t>(code_out, g, r0 + rr, c0 + cc, out_code[o]);
            store_cell<int8_t>(R_out, g, r0 + rr, c0 + cc, out_R[o]);
          }
          if (peer) {
            // row index in the neighbour's frame: my first rows are its rows peer_rows .. peer_rows+GH-1
            // (bottom ghosts), my last GH rows its rows -GH .. -1 (top ghosts); store_cell adds the column images
            const int pi = side ? (rr - FTR) : (a.peer_rows[0] + rr);
            store_cell<uint8_t>(reinterpret_cast<uint8_t *>(a.peer_code[side]), g, pi, c0 + cc, out_code[o]);
            store_cell<int8_t>(reinterpret_cast<int8_t *>(a.peer_R[side]), g, pi, c0 + cc, out_R[o]);
          }
        }
        for (int e = tid; e < FTR * 4; e += FTHREADS) {
          const int rr = e >> 2, wi = (c0 >> 5) + (e & 3);
          if (PART && wi >= ((g.L + 31) >> 5)) continue;       // words beyond the lattice
          if (ecol0 || ecol1 || erow0 || erow1) store_bits_word(S_out, g, r0 + rr, wi, out_S[e]);
          if (prow0 && rr < GH) store_bits_word(a.peer_S[0], g, a.peer_rows[0] + rr, wi, out_S[e]);
          if (prow1 && rr >= FTR - GH) store_bits_word(a.peer_S[1], g, rr - FTR, wi, out_S[e]);
        }
        __syncthreads();  // out_* is read above; the next tile overwrites it
      }
    }
    ty = nty; txs = ntxs; tx = ntx;
  }

#ifdef SPGG_TRACE
  if (tid == 0 && a.trace) {
    unsigned long long t_end; unsigned smid;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_end));
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    unsigned long long *tr = a.trace + (size_t)blockIdx.x * 4;
    tr[0] = t_start; tr[1] = t_end; tr[2] = smid; tr[3] = (unsigned long long)tiles_done;
  }
#endif
  // ---- per-CTA partial row, then the last CTA of the replica folds them in a fixed order
  double v[NSTAT];
#pragma unroll
  for (int z = 0; z < NSTAT; ++z) v[z] = 0.0;
  const double n0 = (double)cls_n[0], n1 = (double)cls_n[1], n2 = (double)cls_n[2], n3 = (double)cls_n[3];
  v[ST_NC_OLD] = n2 + n3; v[ST_N_CD] = n2; v[ST_N_DC] = n1; v[ST_NC_NEW] = n1 + n3;
  v[ST_SUM_P] = n0; v[ST_SUM_P_C] = n1; v[ST_SUM_P_D] = n2; v[ST_SUM_WP_P] = n3;  // raw class counts until the fold
#pragma unroll
  for (int z = 0; z < 4; ++z) v[ST_X_SN0 + z] = (double)cls_sn[z];
  v[ST_SUM_RATIO] = (double)s_ratio;
#pragma unroll
  for (int z = 0; z < 6; ++z) v[ST_GROUP0 + z] = (double)grp[z];
  v[ST_SUM_R] = (double)sum_r;
  v[ST_SUM_Q + 0] = (double)sq0; v[ST_SUM_Q + 1] = (double)sq1; v[ST_SUM_Q + 2] = (double)sq2; v[ST_SUM_Q + 3] = (double)sq3;
  v[ST_SUM_Q_C + 0] = (double)sc0; v[ST_SUM_Q_C + 1] = (double)sc1; v[ST_SUM_Q_C + 2] = (double)sc2; v[ST_SUM_Q_C + 3] = (double)sc3;
  v[ST_SUM_NI] = (double)s_ni * 100.0;
  v[ST_N_BEST_POS] = (double)(pk_best & 0xffffu);
  v[ST_N_BEST_2ND] = (double)(pk_best >> 16);
  v[ST_X_NSEL] = (double)n_sel;
  __syncthreads();
  block_reduce_bfly<NSTAT>(v, sm_red);
  double *part = a.partials + ((long long)rep * g.ctas_per_rep + cta) * NSTAT;
  if (tid < NSTAT) part[tid] = sm_red[tid];
  if (a.peer_code[0] != nullptr || a.peer_code[1] != nullptr) __threadfence_system();  // rows stored into a neighbour's planes
  if (upd) {
    // this launch's own global maximum: every unordered neighbour pair is seen from both ends and
    // fsub_rn(x, y) == -fsub_rn(y, x), so max over sites of the best signed difference == max |difference|
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) gbest = fmaxf(gbest, __shfl_down_sync(0xffffffffu, gbest, o));
    // non-negative IEEE floats order like unsigned integers
    if (lane == 0) atomicMax(reinterpret_cast<unsigned int *>(const_cast<void *>(a.gmax)) + (long long)rep * a.cap + a.rel,
                             __float_as_uint(gbest));
  }
  __threadfence();
  // the last tile's Q segments / tile planes were left in flight while the statistics were reduced
  if (lane == 0 && (upd || (tid == 0 && sel))) tma_store_wait_all();
  __syncthreads();
  if (tid == 0) {
    const unsigned t = atomicInc(a.tickets + rep, (unsigned)g.ctas_per_rep - 1u);
    s_is_last = (t == (unsigned)g.ctas_per_rep - 1u);
  }
  __syncthreads();
  if (!s_is_last) return;
  __threadfence();
  fold_partials(a.partials + (long long)rep * g.ctas_per_rep * NSTAT, g.ctas_per_rep, sm_red);
  if (tid == 0) {
    double *row = a.stats + ((long long)rep * a.cap + a.rel) * NSTAT;
    double *s = sm_red;
    s[ST_SUM_R] *= rc.rq;
    if (upd) {
      // exact-count payoff sums per class: P = ((rc*SN/5 - 5*cost*C) - lo)/span
      double Pc[4];
      const double nc[4] = {s[ST_SUM_P], s[ST_SUM_P_C], s[ST_SUM_P_D], s[ST_SUM_WP_P]};
      for (int z = 0; z < 4; ++z) {
        const double C = (z >> 1) ? 1.0 : 0.0;
        Pc[z] = ((rc.rc * s[ST_X_SN0 + z] / 5.0 - 5.0 * rc.cost * C * nc[z]) - rc.lo * nc[z]) / rc.span;
      }
      s[ST_SUM_P] = Pc[0] + Pc[1] + Pc[2] + Pc[3];
      s[ST_SUM_P_C] = Pc[2] + Pc[3];
      s[ST_SUM_P_D] = Pc[0] + Pc[1];
      s[ST_SUM_WP_P] = rc.wP * s[ST_SUM_P];
      s[ST_SUM_REW_C] = rc.wP * (Pc[1] + Pc[3]) + rc.wR * 0.5 * (nc[1] + nc[3]);
      s[ST_SUM_REW_D] = rc.wP * (Pc[0] + Pc[2]);
      for (int z = 0; z < 4; ++z) s[ST_SUM_Q_D + z] = s[ST_SUM_Q + z] - s[ST_SUM_Q_C + z];
      // every CTA's atomicMax is ordered before its ticket: the table entry is final here
      const float g_exact = __ldcg(reinterpret_cast<const float *>(a.gmax) + (long long)rep * a.cap + a.rel);
      s[ST_GMAX] = (double)g_exact;
      if (a.gvec) {
        a.gvec[4 * a.rel + 0] = g_exact;            // strip: report, k_strip_verify decides (spgg_kernels.cuh)
      } else {
        if (a.gcarry) a.gcarry[rep] = g_exact;
        if (a.spec && g_exact != gm_used) atomicMin(a.bad_at, a.rel);   // the host re-runs from this launch
      }
      for (int z = 0; z < ST_X_SN0; ++z) row[z] = s[z];
    } else {
      row[ST_SUM_R] = s[ST_SUM_R];
    }
    if (sel && g.wrap_rows) {  // uniform lattice after this action -> next iteration breaks (spgg.py:405)
      const double nsel = s[ST_X_NSEL];
      if (nsel == 0.0 || nsel == (double)g.site_stride) a.stop_at[rep] = a.j + 1;
    }
    if (a.gvec) {              // strip: does it hold a defecting / a cooperating action?
      const double nsel = s[ST_X_NSEL];
      const float anyD = (sel && nsel == (double)g.site_stride) ? 0.0f : 1.0f;
      const float anyC = (sel && nsel == 0.0) ? 0.0f : 1.0f;
      a.gvec[4 * a.rel + 1] = anyD;
      a.gvec[4 * a.rel + 2] = anyC;
      if (a.ring_world > 0) {
        // ring mode: combine the report into slot (gen & 3) of every rank, then count this rank in.  The
        // halo rows this launch stored into the neighbours' planes were fenced by their CTAs before they
        // took their tickets, and this thread saw every ticket: arrival implies the rows are there.
        const unsigned mbits = upd ? __float_as_uint(a.gvec[4 * a.rel + 0]) : 0u;
        const int so = (a.gen & (RING_SLOTS - 1)) * RING_WORDS;
        __threadfence_system();
        for (int p = 0; p < a.ring_world; ++p) {
          unsigned *slot = a.ring_peer[p] + so;
          atomicMax_system(slot + 0, mbits);
          if (anyD != 0.0f) atomicMax_system(slot + 1, 1u);
          if (anyC != 0.0f) atomicMax_system(slot + 2, 1u);
        }
        __threadfence_system();
        for (int p = 0; p < a.ring_world; ++p) atomicAdd_system(a.ring_peer[p] + so + 3, 1u);
      }
    }
  }
}

template <int M, bool ACTION, bool UPD, bool SEL, bool PART = false>
__global__ void __launch_bounds__(FTHREADS, 2)
k_step_fast(const __grid_constant__ FastMaps tm, KArgs a) {
  pdl_launch_dependents();
  pdl_wait();  // the planes, the stop flags and gmax come from the kernels before this one
  const int rep = blockIdx.x / a.g.ctas_per_rep;
  // a speculation of an EARLIER launch of this chunk failed: nothing after it may run (a failure another
  // replica records during this very launch has the value a.rel and does not stop its siblings half way)
  if (a.bad_at && *a.bad_at < a.rel) return;
  const int stop = a.stop_at[rep];
  if (stop >= 0 && a.j > stop) return;
  if (SEL && stop >= 0 && a.j == stop) {  // uniform lattice: finish iteration j, choose nothing (spgg.py:405)
    if constexpr (UPD) step_fast_body<M, ACTION, true, false, PART>(tm, a);
    return;
  }
  step_fast_body<M, ACTION, UPD, SEL, PART>(tm, a);
}

// lattice-global max |reward difference| of iteration j (spgg.py:486-488), fast path.
// Warp-autonomous: every warp walks its own 16x128-site tiles (TMA-staged code tile + halo,
// double-buffered per warp), top row to bottom row, a lane holding the rewards of 4 consecutive
// sites of the current and the previous row(s) in registers; rewards come from a reward table
// replicated 32 times (entry c of lane l at [c*32 + l]: conflict-free).  Every unordered
// neighbour pair is visited once (the offset set is symmetric, |d| too):
//   M=1: (1,0) (0,1)        M=2: + (2,0) (0,2) (1,1) (1,-1)
// No block-wide barrier after the prologue.
constexpr int GWARPS = 8;  // warps per CTA of k_gmax_fast
template <int M>
struct GmaxSmem {
  static constexpr int kRowsCR = FTR + 2 * M;
  static constexpr int kStageBytes = (kRowsCR * FROWB + 127) / 128 * 128;
  static constexpr int kOffTab = GWARPS * 2 * kStageBytes;       // 128 x 32 floats
  static constexpr int kOffBar = kOffTab + 128 * 32 * 4;         // 2 barriers per warp
  static constexpr int kTotal = kOffBar + GWARPS * 2 * 8 + 128;  // + base alignment slack
};

template <int M>
__global__ void __launch_bounds__(GWARPS * 32, 3)
k_gmax_fast(const __grid_constant__ CUtensorMap ld_code, GArgs a) {
  typedef GmaxSmem<M> SM;
  const Geom &g = a.g;
  const int ctas = gridDim.x / g.n_rep;
  const int rep = blockIdx.x / ctas, cta = blockIdx.x - rep * ctas;
  pdl_launch_dependents();
  extern __shared__ __align__(128) unsigned char smem_gfast[];
  unsigned char *smem = smem_gfast + ((128u - (smem_u32(smem_gfast) & 127u)) & 127u);
  float *tab32 = reinterpret_cast<float *>(smem + SM::kOffTab);
  __shared__ float s_wmax[GWARPS];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + SM::kOffBar) + warp * 2;
  unsigned char *stg = smem + warp * (2 * SM::kStageBytes);
  __shared__ float s_tab[128];
  if (tid < 128) s_tab[tid] = a.rc[rep].rewtab[tid];  // one global load per thread, then replicate on chip
  if (lane == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  pdl_wait();  // the code plane and the stop flags come from the k_step before this kernel
  const int stop = a.stop_at[rep];
  if (stop >= 0 && a.j > stop) return;
  if (lane == 0 && cta * GWARPS + warp < g.n_tx * g.n_ty) {  // first tile on its way while the table is built
    const int t0 = cta * GWARPS + warp;
    mbar_expect_tx(&bars[0], SM::kRowsCR * FROWB);
    tma_load_3d(stg, &ld_code, &bars[0], (t0 % g.n_tx) * TC, (t0 / g.n_tx) * FTR + GH - M, rep);
  }
#pragma unroll 4
  for (int i = tid; i < 128 * 32; i += GWARPS * 32) tab32[i] = s_tab[i >> 5];
  __syncthreads();
  const float *tl = tab32 + lane;
  const int n_tiles = g.n_tx * g.n_ty;
  const int gw = cta * GWARPS + warp, n_gw = ctas * GWARPS;
  auto issue = [&](int tile, int st) {
    const int r0 = (tile / g.n_tx) * FTR, c0 = (tile % g.n_tx) * TC;
    mbar_expect_tx(&bars[st], SM::kRowsCR * FROWB);
    tma_load_3d(stg + st * SM::kStageBytes, &ld_code, &bars[st], c0, r0 + GH - M, rep);
  };
  float lmax4[4] = {0.f, 0.f, 0.f, 0.f};  // one running maximum per site of the lane: short dependency chains
  auto upd = [&](int k, float x, float y) { lmax4[k] = fmaxf(lmax4[k], fabsf(__fsub_rn(x, y))); };
  int done = 0, stage = 0;
  for (int tile = gw; tile < n_tiles; tile += n_gw, ++done, stage ^= 1) {
    __syncwarp();  // every lane has left the stage about to be refilled
    if (lane == 0 && tile + n_gw < n_tiles) issue(tile + n_gw, stage ^ 1);
    mbar_wait(&bars[stage], (uint32_t)(done >> 1) & 1u);
    const uint32_t *cw = reinterpret_cast<const uint32_t *>(stg + stage * SM::kStageBytes) + (CPAD / 4);
    const bool lv = (tile % g.n_tx) * TC + 4 * lane < g.L;   // partial last tile column: lanes beyond the lattice
    float u1[4] = {0.f, 0.f, 0.f, 0.f}, u2[4] = {0.f, 0.f, 0.f, 0.f};  // rewards one / two rows up
    float u1l = 0.f, u1r = 0.f;                                        // ... and their row-neighbours
#pragma unroll 3
    for (int s = 0; s < FTR + M; ++s) {  // staged row s = tile row s - M
      const uint32_t w = cw[s * FROWW + lane];
      const uint32_t wl = cw[s * FROWW - 1];         // columns -4..-1 (same word for every lane)
      float c[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) c[k] = tl[((w >> (8 * k + 1)) & 0x7Fu) << 5];
      float l1 = __shfl_up_sync(0xffffffffu, c[3], 1);
      const float hl1 = tl[((wl >> 25) & 0x7Fu) << 5];
      if (lane == 0) l1 = hl1;
      float l2 = 0.f, r1 = 0.f;
      if constexpr (M == 2) {
        l2 = __shfl_up_sync(0xffffffffu, c[2], 1);
        const float hl2 = tl[((wl >> 17) & 0x7Fu) << 5];
        if (lane == 0) l2 = hl2;
        const uint32_t wr = cw[s * FROWW + 32];      // columns 128..131
        r1 = __shfl_down_sync(0xffffffffu, c[0], 1);
        const float hr1 = tl[((wr >> 1) & 0x7Fu) << 5];
        if (lane == 31) r1 = hr1;
      }
      if (s >= M && lv) {  // a row of the tile: pairs with the rows above and to the left
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          upd(k, u1[k], c[k]);                                   // (1,0)
          upd(k, k == 0 ? l1 : c[(k + 3) & 3], c[k]);            // (0,1)
          if constexpr (M == 2) {
            upd(k, u2[k], c[k]);                                 // (2,0)
            upd(k, k == 0 ? l2 : (k == 1 ? l1 : c[(k + 2) & 3]), c[k]);   // (0,2)
            upd(k, k == 0 ? u1l : u1[(k + 3) & 3], c[k]);        // (1,1)
            upd(k, k == 3 ? u1r : u1[(k + 1) & 3], c[k]);        // (1,-1)
          }
        }
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) { u2[k] = u1[k]; u1[k] = c[k]; }
      u1l = l1; u1r = r1;
    }
  }
  float lmax = fmaxf(fmaxf(lmax4[0], lmax4[1]), fmaxf(lmax4[2], lmax4[3]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) lmax = fmaxf(lmax, __shfl_down_sync(0xffffffffu, lmax, o));
  if (lane == 0) s_wmax[warp] = lmax;
  __syncthreads();
  if (tid == 0) {
    float m = s_wmax[0];
    for (int w = 1; w < GWARPS; ++w) m = fmaxf(m, s_wmax[w]);
    // non-negative IEEE floats order like unsigned integers
    atomicMax(reinterpret_cast<unsigned int *>(a.gmax) + (long long)rep * a.cap + a.rel, __float_as_uint(m));
  }
}

}  // namespace spgg
