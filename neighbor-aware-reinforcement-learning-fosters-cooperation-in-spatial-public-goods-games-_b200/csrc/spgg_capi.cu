// C ABI of libspgg_b200 (include/spgg.h): handle, device memory, launch sequencing.
// The arithmetic lives in spgg_kernels.cuh.  No CPU fallback: every entry point that
// computes needs a CUDA device and fails with SPGG_E_CUDA otherwise.
#include "../../include/spgg.h"
#include "spgg_kernels.cuh"
#include "spgg_dispatch.h"
#include "spgg_fast.cuh"
#include "spgg_resident.cuh"

#include <cudaTypedefs.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

using namespace spgg;

static thread_local std::string g_err;

static int fail(int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CUDA_TRY(expr)                                                                  \
  do {                                                                                  \
    cudaError_t e_ = (expr);                                                            \
    if (e_ != cudaSuccess)                                                              \
      return fail(SPGG_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_),  \
                  __FILE__, __LINE__);                                                  \
  } while (0)


struct spgg_handle {
  int device = 0;
  int n_rep = 1;
  int mode = MODE_F32_I8;
  int M = 1;
  int action = 0;
  std::vector<spgg_params_t> params;
  std::vector<RepConst> rc_host;
  Geom g{};
  int threads = 256;
  int gmax_ctas = 1;  // CTAs per replica of k_gmax_fast
  size_t smem_step = 0, smem_gmax = 0;
  // device memory
  RepConst *d_rc = nullptr;
  double *d_valtab = nullptr;  // fp64 mode: {reward, ratio} per reward code and replica (k_build_valtab)
  bool lean = false;           // Q-learning on the general path: update launches run k_step_lean
  int gmax_ctas_gen = 1;       // CTAs per replica of the general path's k_gmax_lean launch
  void *d_Qb[2] = {nullptr, nullptr};  // [1] only with spec: Q is then read from [qcur] and written to [qcur^1]
  int qcur = 0;
  void *Qcur() const { return d_Qb[qcur]; }
  // speculative global maximum (KArgs::spec): fast path only; SPGG_NO_SPEC=1 keeps the exact two-launch iteration
  bool spec = false;
  bool carry_valid = false;   // gcarry holds the maximum of the iteration before the next update launch
  float *d_gcarry = nullptr;
  int *d_bad = nullptr;
  CUtensorMap qmaps[2];
  bool spec_on = true;            // switched off for good when the maximum changes too often to be worth guessing
  long long spec_launches = 0, spec_failures = 0;
  long long spec_iterations = 0;  // iterations finished by launches that guessed (re-runs not counted twice)
  bool in_rerun = false;
  float *d_gvec = nullptr;        // strips: [cap][4] per-iteration report {max, any D, any C, -} (KArgs::gvec)
  // strips: planes of the strip above ([0]) / below ([1]) mapped into this process (cudaIpc), per plane parity
  void *peer_code[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
  void *peer_R[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
  uint32_t *peer_S[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
  int peer_rows[2] = {0, 0};
  bool peer_on = false;
  std::vector<void *> ipc_opened;
  // ring of report slots (KArgs::ring_peer): this strip's own, and every rank's mapped here
  unsigned *d_ring = nullptr;
  unsigned *ring_peer[SPGG_MAX_RING] = {nullptr};
  int ring_world = 0;
  int gen = 0;            // launches that pushed into the ring since the last reset (the same on every rank)
  int last_gen = -1;
  int last_rel = -1, last_upd = 0, last_spec = 0, last_sel = 0;  // the launch spgg_strip_verify refers to
  int pend_qcur0 = 0;
  std::vector<char> pend_cur_after, pend_q_after;  // plane / Q parity after the launch with relative index rel
  void *d_R[2] = {nullptr, nullptr};
  void *d_code[2] = {nullptr, nullptr};
  uint32_t *d_S[2] = {nullptr, nullptr};
  int cur = 0;  // planes holding the state of iteration `iter`
  void *d_gmax = nullptr;
  double *d_stats = nullptr;
  double *d_partials = nullptr;
  unsigned *d_tickets = nullptr;
  int *d_stop = nullptr;
  double *d_eps = nullptr;
  uint32_t *d_thr = nullptr;
  int cap = 0;  // rows per replica of stats/gmax/eps tables
  double *d_u = nullptr;
  uint8_t *d_b = nullptr;
  // staging scratch for set/get_state
  uint8_t *d_sc_S = nullptr;
  double *d_sc_R = nullptr, *d_sc_Q = nullptr;
  unsigned long long *d_sc_info = nullptr;
  // fast path (spgg_fast.cuh): TMA descriptors of the two plane sets
  bool fast = false;
  // an uploaded R lies outside [-16, 15] int8 units, which k_step_fast's biased bytes cannot hold: the
  // next select runs on k_step, whose reputation update clips every R into [R_min, R_max] ⊆ [-15, 15]
  bool r_wide = false;
  FastMaps fmaps[2];  // [cur]: loads from plane set cur, stores into cur^1
  // lattice-resident path (spgg_resident.cuh): one cluster per replica, whole chunks per launch
  bool resident = false;
  ResGeom rgeo{};
  size_t smem_res = 0;
  bool pend_resident = false;
  bool res_grid = false;            // grid mode: one lattice over a cooperative grid (spgg_resident.cuh, GRID)
  unsigned char *d_gimg = nullptr;
  double *d_gpart = nullptr;
  unsigned *d_gnsel = nullptr;
  int gnsel_cap = 0;
  std::vector<double> eps_host;
  std::vector<uint32_t> thr_host;
  int replay_pairs = 1;
  long long replay_first = 0, replay_n = 0;  // draws cover iterations replay_first+1 .. replay_first+replay_n
  // host bookkeeping
  long long iter = 0;
  std::vector<double> eps_cur;     // eps used at iteration iter+1
  std::vector<long long> stop_at;  // -1 or the t with uniform S_t
  std::vector<char> stale;         // replica still holds the state of the previous run (include/spgg.h)
  long long launches = 0;
  // pending asynchronous chunk
  bool pending = false;
  long long pend_t0 = 0;
  int pend_n = 0, pend_cur0 = 0, pend_rel = 0;
  cudaStream_t pend_stream = nullptr;
  // spgg_clusters: device scratch (spgg_clusters.cuh) and whether it holds the result of the current state
  CclScratch ccl;
  bool ccl_valid = false;
  int64_t ccl_n = 0;
  // spgg_strip_clusters: record / resolution scratch, and the strip-local pass awaiting its resolution
  CclStripScratch ccl_strip;
  bool ccl_local = false;
  int ccl_which = 0, ccl_flags = 0;
  int64_t ccl_local_n = 0;
  // spgg_pair_counts / spgg_strip_pair_counts (spgg_pairs.cuh): the device counts and a strip's tail rows
  unsigned long long *d_pair_cnt = nullptr;
  uint32_t *d_pair_tail = nullptr;
  size_t pair_cnt_n = 0, pair_tail_n = 0;
  // spgg_block_fields (spgg_blocks.cuh): counts, sums and pieces of the largest call so far
  void *d_blk = nullptr;
  size_t blk_bytes = 0;
  // spgg_value_ranges / spgg_histograms (spgg_hist.cuh): counts, extremes, edges of the largest call so far
  void *d_hist = nullptr;
  size_t hist_bytes = 0;
  // spgg_snapshot: copies of replica states in the handle's plane layout (snap_layout), kept until freed
  struct Snapshot {
    void *mem = nullptr;
    size_t bytes = 0;
    bool full = false;
    long long iter = 0;
    int rep0 = 0, n_rep = 0, flags = 0;
    std::vector<double> rq;   // int8 quantum of each replica at snapshot time
  };
  Snapshot snaps[SPGG_MAX_SNAPSHOTS];
  // spgg_overlap (spgg_overlap.cuh): counts, maxima, sums and tile partials of the largest call so far
  void *d_ov = nullptr;
  size_t ov_bytes = 0;
  size_t elem_code() const { return mode == MODE_F64 ? 4 : 1; }
  size_t elem_R() const { return mode == MODE_F64 ? 8 : (mode == MODE_F32_F ? 4 : 1); }
  size_t elem_Q() const { return mode == MODE_F64 ? 8 : 4; }
  size_t elem_val() const { return mode == MODE_F64 ? 8 : 4; }
  int nq() const { return params[0].algorithm == SPGG_ALGO_DOUBLE_QLEARNING ? 8 : 4; }  // Q values per site
  ~spgg_handle();  // frees whatever device memory and peer mappings the handle holds
};

// ---------------------------------------------------------------- constants
static bool int8_quantum(const spgg_params_t &p, double *rq, int *gi, int *li, int *mn, int *mx) {
  for (int k = 0; k <= 4; ++k) {
    const double s = (double)(1 << k);
    const double a = p.rep_gain_C * s, b = p.delta_R_D * s, c = p.R_min * s, d = p.R_max * s;
    if (a == std::floor(a) && b == std::floor(b) && c == std::floor(c) && d == std::floor(d) &&
        std::fabs(c) <= 127 && std::fabs(d) <= 127 && std::fabs(a) <= 127 && std::fabs(b) <= 127 &&
        c - b >= -128 && d + a <= 127) {
      *rq = 1.0 / s; *gi = (int)a; *li = (int)b; *mn = (int)c; *mx = (int)d;
      return true;
    }
  }
  return false;
}

static void build_repconst(const spgg_params_t &p, RepConst *rc) {
  memset(rc, 0, sizeof(*rc));
  rc->rc = p.r * p.c;
  for (int n = 0; n < 6; ++n) rc->g[n] = rc->rc * (double)n / 5.0;  // spgg.py:256
  rc->cost = p.cost;
  rc->lo = p.r - 5.0;                // spgg.py:149
  rc->span = 4.0 * p.r - rc->lo;     // spgg.py:148,377
  rc->wP = p.wP;
  rc->wR = 1.0 - p.wP;               // spgg.py:108
  rc->alpha = p.alpha; rc->gamma = p.gamma; rc->kappa = p.kappa; rc->leps = p.lambda_eps;
  rc->gainC = p.rep_gain_C; rc->lossD = p.delta_R_D; rc->rmin = p.R_min; rc->rmax = p.R_max;
  rc->alpha_f = (float)p.alpha; rc->gamma_f = (float)p.gamma; rc->kappa_f = (float)p.kappa;
  rc->leps_f = (float)p.lambda_eps;
  rc->gainC_f = (float)p.rep_gain_C; rc->lossD_f = (float)p.delta_R_D;
  rc->rmin_f = (float)p.R_min; rc->rmax_f = (float)p.R_max;
  rc->rq = 1.0;
  int8_quantum(p, &rc->rq, &rc->gain_i, &rc->loss_i, &rc->rmin_i, &rc->rmax_i);
  rc->seed_lo = (uint32_t)p.seed;
  rc->seed_hi = (uint32_t)(p.seed >> 32);
  for (uint32_t r = 0; r < 10; ++r) {
    rc->pkeys[2 * r] = rc->seed_lo + r * 0x9E3779B9u;
    rc->pkeys[2 * r + 1] = rc->seed_hi + r * 0xBB67AE85u;
  }
  rc->has_ratio = (rc->wR != 0.0);
  for (int code = 0; code < 128; ++code) {
    const int sn = code >> 2, C = (code >> 1) & 1, coop = code & 1;
    const double tot = rc->rc * (double)sn / 5.0 - (C ? 5.0 * p.cost : 0.0);
    const double P = (tot - rc->lo) / rc->span;
    const double rew = rc->wP * P + rc->wR * (coop ? 0.5 : 0.0);
    rc->rewtab[code] = (float)rew;
    rc->ratiotab[code] =
        coop ? (float)(std::fabs(rc->wR * 0.5) / (std::fabs(rew) + 1e-9) * 100.0) : 0.0f;
  }
}

// ---------------------------------------------------------------- dispatch
// f(ModeF32I8{}), f(ModeF32F{}) or f(ModeF64{}): the host side of a kernel templated on the arithmetic mode.
// The general and the lean kernels are instantiated in their own translation units (spgg_dispatch.h)
template <class F>
static auto with_mode(int mode, F &&f) {
  switch (mode) {
    case MODE_F32_I8: return f(ModeF32I8{});
    case MODE_F32_F: return f(ModeF32F{});
    default: return f(ModeF64{});
  }
}

static size_t step_smem(int mode, int TR) {
  return with_mode(mode, [&](auto md) { return SmemLayout<decltype(md)>(TR).total; });
}

// launch with programmatic stream serialization (the fast kernels call griddepcontrol.wait
// before touching anything an earlier kernel wrote)
template <class... KArgsT, class... Args>
static cudaError_t launch_pdl(void (*kern)(KArgsT...), int grid, int block, size_t smem, cudaStream_t st,
                              Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, args...);
}

// ---------------------------------------------------------------- fast path plumbing
typedef void (*fast_fn_t)(const FastMaps, KArgs);
template <int M, bool ACTION, bool PART>
static fast_fn_t pick_fast3(int upd, int sel) {
  if (upd) return sel ? k_step_fast<M, ACTION, true, true, PART> : k_step_fast<M, ACTION, true, false, PART>;
  return k_step_fast<M, ACTION, false, true, PART>;
}
template <int M, bool ACTION>
static fast_fn_t pick_fast2(int upd, int sel, bool part) {
  return part ? pick_fast3<M, ACTION, true>(upd, sel) : pick_fast3<M, ACTION, false>(upd, sel);
}
// part: the lattice side is a multiple of 32 but not of 128 (partial last tile column)
static fast_fn_t pick_fast(int M, int action, int upd, int sel, bool part) {
  if (M == 2) return action ? pick_fast2<2, true>(upd, sel, part) : pick_fast2<2, false>(upd, sel, part);
  return action ? pick_fast2<1, true>(upd, sel, part) : pick_fast2<1, false>(upd, sel, part);
}
static size_t fast_smem(int M) { return M == 2 ? FastSmem<2>::kTotal : FastSmem<1>::kTotal; }
typedef void (*gfast_fn_t)(const CUtensorMap, GArgs);
static gfast_fn_t pick_gfast(int M) { return M == 2 ? k_gmax_fast<2> : k_gmax_fast<1>; }
static size_t gfast_smem(int M) { return M == 2 ? GmaxSmem<2>::kTotal : GmaxSmem<1>::kTotal; }

// ---------------------------------------------------------------- resident path plumbing
typedef void (*res_fn_t)(RArgs);
template <bool FULL>
static res_fn_t pick_res2(int M, int action) {
  if (M == 2) return action ? k_resident<2, true, FULL> : k_resident<2, false, FULL>;
  return action ? k_resident<1, true, FULL> : k_resident<1, false, FULL>;
}
static res_fn_t pick_res(int M, int action, int L) {
  return (L % 4 == 0) ? pick_res2<true>(M, action) : pick_res2<false>(M, action);
}
template <bool FULL>
static res_fn_t pick_resg2(int M, int action) {
  if (M == 2) return action ? k_resident<2, true, FULL, true> : k_resident<2, false, FULL, true>;
  return action ? k_resident<1, true, FULL, true> : k_resident<1, false, FULL, true>;
}
static res_fn_t pick_res_grid(int M, int action, int L) {
  return (L % 4 == 0) ? pick_resg2<true>(M, action) : pick_resg2<false>(M, action);
}
// geometry of the decomposition into `cs` row blocks, or CS = 0 when a block does not fit on chip
static ResGeom resident_geom(int L, int cs, size_t smem_limit, int grid = 0) {
  ResGeom rg{};
  rg.grid = grid;
  if (L < 2 * cs) cs = 1;  // a block needs two rows: its ghost rows come from the adjacent blocks only
  rg.rows_max = (L + cs - 1) / cs;
  rg.prow = rg.rows_max + 4;
  rg.QR = (L + 3) / 4;
  rg.pitch = (RG + rg.QR * 4 + RG + 15) / 16 * 16;
  const int quads = rg.rows_max * rg.QR;
  rg.threads = std::max(64, std::min(RES_THREADS, (quads + 31) / 32 * 32));
  rg.CS = (ResSmem(rg).total <= smem_limit) ? cs : 0;
  return rg;
}

// the driver's cuTensorMapEncodeTiled, or 0 with the error set
static PFN_cuTensorMapEncodeTiled_v12000 tensor_map_encoder() {
  static PFN_cuTensorMapEncodeTiled_v12000 encode = nullptr;
  if (!encode) {
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    const cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
    if (e != cudaSuccess || !fn || q != cudaDriverEntryPointSuccess) {
      fail(SPGG_E_CUDA, "cuTensorMapEncodeTiled not available (%s)", cudaGetErrorString(e));
      return nullptr;
    }
    encode = (PFN_cuTensorMapEncodeTiled_v12000)fn;
  }
  return encode;
}

static int make_map(CUtensorMap *map, void *base, uint64_t row_bytes, uint64_t n_rows, uint64_t n_rep,
                    uint64_t rep_stride_bytes, uint32_t box_bytes, uint32_t box_rows, uint64_t visible_bytes = 0) {
  const PFN_cuTensorMapEncodeTiled_v12000 encode = tensor_map_encoder();
  if (!encode) return SPGG_E_CUDA;
  // visible_bytes < row_bytes: the tensor ends before the pitch (loads beyond it give zeros, stores are dropped)
  const cuuint64_t dims[3] = {visible_bytes ? visible_bytes : row_bytes, n_rows, n_rep};
  const cuuint64_t strides[2] = {row_bytes, rep_stride_bytes};
  const cuuint32_t box[3] = {box_bytes, box_rows, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, base, dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(SPGG_E_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return SPGG_OK;
}

// Q table of the fast path: bytes (128 = 8 sites, L/8 chunks, rows, replicas), boxes of one
// 128-site row segment, 128-byte swizzle so that a lane's four consecutive float4 are
// conflict-free in shared memory
static int make_map_q(CUtensorMap *map, void *base, uint64_t L, uint64_t n_rows, uint64_t n_rep) {
  const PFN_cuTensorMapEncodeTiled_v12000 encode = tensor_map_encoder();
  if (!encode) return SPGG_E_CUDA;
  const cuuint64_t dims[4] = {128, L / 8, n_rows, n_rep};
  const cuuint64_t strides[3] = {128, L * 16, n_rows * L * 16};
  const cuuint32_t box[4] = {128, TC / 8, (cuuint32_t)FastSmem<1>::kRowsPerWarp, 1};  // a warp's rows of a tile
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, base, dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(SPGG_E_CUDA, "cuTensorMapEncodeTiled (Q) failed (%d)", (int)r);
  return SPGG_OK;
}

// ---------------------------------------------------------------- lifetime
extern "C" int spgg_abi_version(void) { return SPGG_ABI_VERSION; }
extern "C" const char *spgg_last_error(void) { return g_err.c_str(); }

spgg_handle::~spgg_handle() {
  for (void *p : ipc_opened) cudaIpcCloseMemHandle(p);
  cudaFree(d_rc); cudaFree(d_valtab); cudaFree(d_Qb[0]); cudaFree(d_Qb[1]); cudaFree(d_gcarry); cudaFree(d_bad); cudaFree(d_gvec); cudaFree(d_ring);
  for (int i = 0; i < 2; ++i) { cudaFree(d_R[i]); cudaFree(d_code[i]); cudaFree(d_S[i]); }
  cudaFree(d_gmax); cudaFree(d_stats); cudaFree(d_partials); cudaFree(d_tickets);
  cudaFree(d_stop); cudaFree(d_eps); cudaFree(d_thr); cudaFree(d_u); cudaFree(d_b);
  cudaFree(d_sc_S); cudaFree(d_sc_R); cudaFree(d_sc_Q); cudaFree(d_sc_info);
  cudaFree(d_gimg); cudaFree(d_gpart); cudaFree(d_gnsel);
  ccl_free(&ccl);
  ccl_strip_free(&ccl_strip);
  cudaFree(d_pair_cnt); cudaFree(d_pair_tail);
  cudaFree(d_blk);
  cudaFree(d_hist);
  for (Snapshot &sn : snaps) cudaFree(sn.mem);
  cudaFree(d_ov);
}

extern "C" void spgg_destroy(spgg_t *h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  delete h;
}

extern "C" int spgg_create(const spgg_params_t *params, int n_replicas, int device, spgg_t **out) {
  if (!params || !out || n_replicas < 1) return fail(SPGG_E_INVALID, "spgg_create: null argument or n_replicas < 1");
  const spgg_params_t &p0 = params[0];
  if (p0.L < 4) return fail(SPGG_E_INVALID, "L must be >= 4 (got %d)", p0.L);
  if (p0.rows < 2 * GH || p0.rows > p0.L)
    return fail(SPGG_E_INVALID, "rows must be in [%d, L] (got %d)", 2 * GH, p0.rows);
  if (p0.M != 1 && p0.M != 2) return fail(SPGG_E_INVALID, "M must be 1 or 2 (got %d)", p0.M);
  if (p0.state_mode != SPGG_STATE_REPUTATION && p0.state_mode != SPGG_STATE_ACTION)
    return fail(SPGG_E_INVALID, "Unknown state_representation code %d", p0.state_mode);
  if (p0.precision != SPGG_PREC_FP32 && p0.precision != SPGG_PREC_FP64)
    return fail(SPGG_E_INVALID, "unknown precision %d", p0.precision);
  if (p0.algorithm != SPGG_ALGO_QLEARNING && p0.algorithm != SPGG_ALGO_SARSA &&
      p0.algorithm != SPGG_ALGO_EXPECTED_SARSA && p0.algorithm != SPGG_ALGO_DOUBLE_QLEARNING)
    return fail(SPGG_E_UNSUPPORTED, "algorithm code %d is not built into the fused kernel", p0.algorithm);
  if (p0.row0 < 0 || p0.row0 + p0.rows > p0.L) return fail(SPGG_E_INVALID, "row0/rows outside the lattice");
  for (int r = 1; r < n_replicas; ++r) {
    const spgg_params_t &p = params[r];
    if (p.L != p0.L || p.rows != p0.rows || p.row0 != p0.row0 || p.M != p0.M ||
        p.state_mode != p0.state_mode || p.precision != p0.precision ||
        p.algorithm != p0.algorithm || p.r_storage != p0.r_storage)
      return fail(SPGG_E_INVALID, "replica %d differs in a batch-invariant field (L, rows, M, state, precision)", r);
  }
  int ndev = 0;
  CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(SPGG_E_CUDA, "device %d not available (%d devices)", device, ndev);
  CUDA_TRY(cudaSetDevice(device));

  // owned until it is complete: every error return below frees what was built so far
  std::unique_ptr<spgg_handle> hp(new spgg_handle());
  spgg_handle *h = hp.get();
  h->device = device;
  h->n_rep = n_replicas;
  h->params.assign(params, params + n_replicas);
  h->M = p0.M;
  h->action = p0.state_mode == SPGG_STATE_ACTION;
  h->rc_host.resize(n_replicas);
  bool all_i8 = true;
  for (int r = 0; r < n_replicas; ++r) {
    build_repconst(params[r], &h->rc_host[r]);
    double rq; int a, b, c, d;
    all_i8 = all_i8 && int8_quantum(params[r], &rq, &a, &b, &c, &d);
  }
  if (p0.precision == SPGG_PREC_FP64) h->mode = MODE_F64;
  else if (p0.r_storage == SPGG_RSTORE_FP32) h->mode = MODE_F32_F;
  else if (p0.r_storage == SPGG_RSTORE_INT8) {
    if (!all_i8) return fail(SPGG_E_INVALID, "reputation parameters are not representable in int8 units");
    h->mode = MODE_F32_I8;
  } else h->mode = all_i8 ? MODE_F32_I8 : MODE_F32_F;

  Geom &g = h->g;
  g.L = p0.L; g.rows = p0.rows; g.row0 = p0.row0; g.wrap_rows = (p0.rows == p0.L);
  g.pitchB = CPAD + (p0.L + 15) / 16 * 16 + CPAD;
  g.pitchW = WPAD + ((p0.L + 31) / 32 + 3) / 4 * 4 + WPAD;
  // fast path (spgg_fast.cuh): int8 throughput mode on 128-aligned lattices, |R| <= 15 units
  {
    bool ok = (h->mode == MODE_F32_I8) && (g.L % 32 == 0) && (g.L >= TC) && (g.rows % FTR == 0) &&
              p0.algorithm == SPGG_ALGO_QLEARNING && getenv("SPGG_NO_FAST") == nullptr;
    for (int r = 0; r < n_replicas && ok; ++r)
      ok = h->rc_host[r].rmin_i >= -15 && h->rc_host[r].rmax_i <= 15 && h->rc_host[r].gain_i >= 0 &&
           h->rc_host[r].loss_i >= 0;
    h->fast = ok;
  }
  // resident path (spgg_resident.cuh): whole lattice, int8 throughput mode, Q-learning, on-chip fit
  {
    cudaDeviceProp prop0;
    CUDA_TRY(cudaGetDeviceProperties(&prop0, device));
    res_fn_t rf = pick_res(h->M, h->action, h->g.L);
    cudaFuncAttributes fa;
    CUDA_TRY(cudaFuncGetAttributes(&fa, rf));
    const size_t lim = prop0.sharedMemPerBlockOptin - fa.sharedSizeBytes - 1024;
    const bool eligible = (h->mode == MODE_F32_I8) && g.wrap_rows && p0.row0 == 0 &&
                          p0.algorithm == SPGG_ALGO_QLEARNING && getenv("SPGG_NO_RESIDENT") == nullptr;
    // clusters of 8 CTAs (15 co-resident on a B200) serve batches best; a lattice that is alone (or
    // nearly) on the GPU, or too large for 8 blocks, is spread over a non-portable cluster of 16
    ResGeom rg = resident_geom(g.L, 8, lim);
    if (eligible && g.L >= 32 && (rg.CS == 0 || n_replicas <= 4) && getenv("SPGG_RES_CS8") == nullptr) {
      const ResGeom rg16 = resident_geom(g.L, 16, lim);
      if (rg16.CS == 16 &&
          cudaFuncSetAttribute(rf, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess &&
          cudaFuncSetAttribute(rf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lim) == cudaSuccess) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(16u * (unsigned)n_replicas);
        cfg.blockDim = dim3((unsigned)rg16.threads);
        cfg.dynamicSmemBytes = ResSmem(rg16).total;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 16; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        int n_clusters = 0;
        if (cudaOccupancyMaxActiveClusters(&n_clusters, rf, &cfg) == cudaSuccess && n_clusters >= 1) rg = rg16;
      }
      (void)cudaGetLastError();  // a refused opt-in leaves the portable geometry in place
    }
    h->resident = eligible && rg.CS > 0;
    if (h->resident) {
      h->rgeo = rg;
      h->smem_res = ResSmem(rg).total;
      // the opt-in is per function, not per handle: always the largest size any geometry may ask for
      CUDA_TRY(cudaFuncSetAttribute(rf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lim));
    } else if (eligible && n_replicas == 1 && getenv("SPGG_NO_RESIDENT_GRID") == nullptr) {
      // grid mode: a lone lattice too large for one cluster is spread over every SM (cooperative
      // launch, one CTA per SM) as long as a row block still fits in shared memory
      res_fn_t gf = pick_res_grid(h->M, h->action, h->g.L);
      cudaFuncAttributes gfa;
      CUDA_TRY(cudaFuncGetAttributes(&gfa, gf));
      const size_t glim = prop0.sharedMemPerBlockOptin - gfa.sharedSizeBytes - 1024;
      int coop = 0;
      CUDA_TRY(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device));
      const int nb_ctas = std::min(prop0.multiProcessorCount, g.L / 2);
      ResGeom gg = resident_geom(g.L, nb_ctas, glim, 1);
      if (coop && nb_ctas >= RES_RING && gg.CS == nb_ctas &&
          cudaFuncSetAttribute(gf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)glim) == cudaSuccess) {
        int occ_g = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_g, gf, gg.threads, ResSmem(gg).total) == cudaSuccess &&
            (long long)occ_g * prop0.multiProcessorCount >= nb_ctas) {
          h->resident = true;
          h->res_grid = true;
          h->rgeo = gg;
          h->smem_res = ResSmem(gg).total;
        }
      }
      (void)cudaGetLastError();
    }
  }
  g.TR = h->fast ? FTR : (g.rows >= 512 ? 16 : (g.rows >= 64 ? 8 : 4));
  h->threads = h->fast ? FTHREADS : 32 * std::min(8, g.TR);
  g.n_tx = (g.L + TC - 1) / TC;
  g.n_ty = (g.rows + g.TR - 1) / g.TR;
  g.n_rep = n_replicas;
  g.plane_stride = (long long)(g.rows + 2 * GH) * g.pitchB;
  g.bits_stride = (long long)(g.rows + 2 * GH) * g.pitchW;
  g.site_stride = (long long)g.rows * g.L;
  h->smem_step = step_smem(h->mode, g.TR);
  h->smem_gmax = (h->elem_val() * (size_t)(g.TR + 2 * HR) * SMW + 15) / 16 * 16 + 512;

  // opt in to the shared memory each instantiation needs and size the persistent grid
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  int occ = 1;
  h->lean = !h->fast && p0.algorithm == 0 && getenv("SPGG_NO_LEAN") == nullptr;
  if (h->lean) h->smem_step = step_smem(h->mode, LEAN_TR_MAX);   // k_step_lean addresses the 16-row layout
  for (int replay = 0; replay < 2; ++replay) {
    step_fn_t f = pick_step(h->mode, h->M, h->action, replay);
    CUDA_TRY(cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_step));
    if (!replay)
      CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, f, h->threads, h->smem_step));
    if (h->lean) {
      // the persistent grid is sized for the kernel that runs every iteration
      step_fn_t fl = pick_lean(h->mode, h->M, h->action, replay);
      CUDA_TRY(cudaFuncSetAttribute(fl, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_step));
      if (!replay)
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fl, h->threads, h->smem_step));
    }
  }
  if (h->fast) {
    for (int v = 0; v < 3; ++v) {
      fast_fn_t fv = pick_fast(h->M, h->action, v != 2, v != 1, g.L % TC != 0);
      CUDA_TRY(cudaFuncSetAttribute(fv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fast_smem(h->M)));
    }
    fast_fn_t ff = pick_fast(h->M, h->action, 1, 1, g.L % TC != 0);
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ff, FTHREADS, fast_smem(h->M)));
    CUDA_TRY(cudaFuncSetAttribute(pick_gfast(h->M), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gfast_smem(h->M)));
    int gocc = 1;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&gocc, pick_gfast(h->M), GWARPS * 32, gfast_smem(h->M)));
    const long long n_tiles_g = (long long)((p0.L + TC - 1) / TC) * (p0.rows / FTR);
    h->gmax_ctas = (int)std::max<long long>(1, std::min<long long>((n_tiles_g + GWARPS - 1) / GWARPS,
                       ((long long)prop.multiProcessorCount * std::max(1, gocc)) / n_replicas));
  }
  CUDA_TRY(cudaFuncSetAttribute(pick_gmax_lean(h->mode, h->M), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)h->smem_gmax));
  if (occ < 1) return fail(SPGG_E_CUDA, "kernel does not fit on an SM (smem %zu)", h->smem_step);
  const long long n_tiles = (long long)g.n_tx * g.n_ty;
  long long per_rep = std::max<long long>(1, ((long long)prop.multiProcessorCount * occ) / n_replicas);
  g.ctas_per_rep = (int)std::min<long long>(n_tiles, per_rep);
  {
    int gocc = 1;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&gocc, pick_gmax_lean(h->mode, h->M), h->threads, h->smem_gmax));
    h->gmax_ctas_gen = (int)std::min<long long>(n_tiles, std::max<long long>(1, ((long long)prop.multiProcessorCount * std::max(1, gocc)) / n_replicas));
  }
  // the fast kernel's packed 16-bit counters bound the sites one thread may visit per launch
  if (h->fast && (g.site_stride / ((long long)g.ctas_per_rep * FTHREADS)) > 60000) h->fast = false;
  h->spec = h->fast && getenv("SPGG_NO_SPEC") == nullptr;

  const size_t nQ = (size_t)n_replicas * g.site_stride * h->nq() * h->elem_Q();
  const size_t nR = (size_t)n_replicas * g.plane_stride * h->elem_R();
  const size_t nC = (size_t)n_replicas * g.plane_stride * h->elem_code();
  const size_t nS = (size_t)n_replicas * g.bits_stride * 4;
#define ALLOC(ptr, bytes)                                                                   \
  do {                                                                                      \
    cudaError_t e_ = cudaMalloc((void **)&(ptr), (bytes));                                  \
    if (e_ != cudaSuccess)                                                                  \
      return fail(SPGG_E_CUDA, "cudaMalloc(%zu bytes) failed: %s", (size_t)(bytes), cudaGetErrorString(e_)); \
    cudaMemset((ptr), 0, (bytes));                                                          \
  } while (0)
  ALLOC(h->d_rc, sizeof(RepConst) * n_replicas);
  ALLOC(h->d_Qb[0], nQ);
  if (h->spec) { ALLOC(h->d_Qb[1], nQ); ALLOC(h->d_gcarry, sizeof(float) * n_replicas); ALLOC(h->d_bad, sizeof(int)); }
  for (int i = 0; i < 2; ++i) { ALLOC(h->d_R[i], nR); ALLOC(h->d_code[i], nC); ALLOC(h->d_S[i], nS); }
  ALLOC(h->d_partials, sizeof(double) * (size_t)n_replicas * g.ctas_per_rep * NSTAT);
  ALLOC(h->d_tickets, sizeof(unsigned) * n_replicas);
  ALLOC(h->d_stop, sizeof(int) * n_replicas);
  if (h->res_grid) {
    ALLOC(h->d_gimg, (size_t)h->rgeo.CS * 6 * h->rgeo.prow * h->rgeo.pitch);
    ALLOC(h->d_gpart, sizeof(double) * (size_t)RES_RING * h->rgeo.CS * RES_NRED);
  }
#undef ALLOC
  if (h->fast) {
    const int rowsCR = FTR + 2 * h->M, rowsS = FTR + 4;
    const uint64_t nrows = (uint64_t)(g.rows + 2 * GH);
    for (int i = 0; i < 2; ++i) {
      FastMaps &fm = h->fmaps[i];
      int e = make_map(&fm.ld_code, h->d_code[i], (uint64_t)g.pitchB, nrows, n_replicas, (uint64_t)g.plane_stride, FROWB, rowsCR);
      if (!e) e = make_map(&fm.ld_R, h->d_R[i], (uint64_t)g.pitchB, nrows, n_replicas, (uint64_t)g.plane_stride, FROWB, rowsCR);
      if (!e) e = make_map(&fm.ld_S, h->d_S[i], (uint64_t)g.pitchW * 4, nrows, n_replicas, (uint64_t)g.bits_stride * 4, FSROWB, rowsS);
      // the store maps end at the last column of the lattice: a partial last tile writes nothing beyond it
      // (ghost columns and padding are the edge path's business)
      if (!e) e = make_map(&fm.st_code, h->d_code[i ^ 1], (uint64_t)g.pitchB, nrows, n_replicas, (uint64_t)g.plane_stride, TC, FTR, (uint64_t)(CPAD + g.L));
      if (!e) e = make_map(&fm.st_R, h->d_R[i ^ 1], (uint64_t)g.pitchB, nrows, n_replicas, (uint64_t)g.plane_stride, TC, FTR, (uint64_t)(CPAD + g.L));
      if (!e) e = make_map(&fm.st_S, h->d_S[i ^ 1], (uint64_t)g.pitchW * 4, nrows, n_replicas, (uint64_t)g.bits_stride * 4, TC / 8, FTR);
      if (!e) e = make_map_q(&h->qmaps[i], h->d_Qb[(i == 1 && h->spec) ? 1 : 0], (uint64_t)g.L, (uint64_t)g.rows, (uint64_t)n_replicas);
      if (e) return e;
    }
  }
  CUDA_TRY(cudaMemcpy(h->d_rc, h->rc_host.data(), sizeof(RepConst) * n_replicas, cudaMemcpyHostToDevice));
  if (h->mode == MODE_F64) {
    const size_t vb = sizeof(double) * 2 * ((size_t)n_replicas << VALTAB_BITS);
    if (cudaMalloc((void **)&h->d_valtab, vb) != cudaSuccess)
      return fail(SPGG_E_CUDA, "cudaMalloc(%zu bytes) failed (reward table)", vb);
    CUDA_TRY(launch_build_valtab(h->d_rc, h->d_valtab, n_replicas));
  }
  std::vector<int> neg(n_replicas, -1);
  CUDA_TRY(cudaMemcpy(h->d_stop, neg.data(), sizeof(int) * n_replicas, cudaMemcpyHostToDevice));
  if (h->spec) {
    const int none = 0x7fffffff;
    CUDA_TRY(cudaMemcpy(h->d_bad, &none, sizeof(int), cudaMemcpyHostToDevice));
  }
  h->eps_cur.resize(n_replicas);
  for (int r = 0; r < n_replicas; ++r) h->eps_cur[r] = params[r].epsilon;
  h->stop_at.assign(n_replicas, -1);
  h->stale.assign(n_replicas, 0);
  *out = hp.release();
  return SPGG_OK;
}

// ---------------------------------------------------------------- pending chunk
static int launch_step(spgg_handle *h, int do_update, int do_select, cudaStream_t st, bool allow_spec);

// A speculative update launch found that the global maximum it assumed was not the one it computed
// (KArgs::spec): every later launch of the chunk returned without touching anything, so the inputs of
// the failed launch are intact (planes and Q are ping-pong pairs).  Re-run from there; the failed
// launch left the exact maximum in gcarry, so the re-run's guess is right.
// put the handle back where it was just before launch `bad` of the pending chunk (its inputs are intact)
static int rewind_to_failed_launch(spgg_handle *h, int bad) {
  h->spec_failures += 1;
  // small lattices change their maximum every few iterations: not worth guessing there
  if (h->spec_failures > 8 && h->spec_failures * 16 > h->spec_iterations) h->spec_on = false;
  const int none = 0x7fffffff;
  CUDA_TRY(cudaMemcpy(h->d_bad, &none, sizeof(int), cudaMemcpyHostToDevice));
  // a uniform-lattice flag raised by the failed launch itself is not to be trusted
  std::vector<int> stop(h->n_rep);
  CUDA_TRY(cudaMemcpy(stop.data(), h->d_stop, sizeof(int) * h->n_rep, cudaMemcpyDeviceToHost));
  for (int r = 0; r < h->n_rep; ++r)
    if (stop[r] == (int)(h->pend_t0 + bad) + 1) stop[r] = -1;
  CUDA_TRY(cudaMemcpy(h->d_stop, stop.data(), sizeof(int) * h->n_rep, cudaMemcpyHostToDevice));
  // parities as launch bad-1 left them
  h->cur = h->pend_cur_after[bad - 1];
  h->qcur = h->pend_q_after[bad - 1];
  h->carry_valid = true;
  h->pend_rel = bad - 1;
  return SPGG_OK;
}

static int rerun_failed_speculation(spgg_handle *h) {
  for (;;) {
    int bad = 0x7fffffff;
    CUDA_TRY(cudaMemcpy(&bad, h->d_bad, sizeof(int), cudaMemcpyDeviceToHost));
    if (bad == 0x7fffffff) return SPGG_OK;
    if (bad < 1 || bad > h->pend_n) return fail(SPGG_E_STATE, "speculation bookkeeping out of range (%d of %d)", bad, h->pend_n);
    int rcode0 = rewind_to_failed_launch(h, bad);
    if (rcode0) return rcode0;
    h->in_rerun = true;
    const int n = h->pend_n;
    for (int s = bad; s <= n; ++s) {
      h->pend_rel += 1;
      int rcode = launch_step(h, 1, s < n ? 1 : 0, h->pend_stream, true);
      if (rcode) return rcode;
      if (!h->spec_on && s < n) {  // speculation was just switched off: the rest of the chunk runs exactly
        for (++s; s <= n; ++s) {
          rcode = spgg_phase_gmax(h, h->pend_stream);
          if (!rcode) rcode = launch_step(h, 1, s < n ? 1 : 0, h->pend_stream, false);
          if (rcode) return rcode;
        }
      }
    }
    h->in_rerun = false;
    CUDA_TRY(cudaStreamSynchronize(h->pend_stream));
    CUDA_TRY(cudaGetLastError());
  }
}

static int finish_pending(spgg_handle *h) {
  if (!h->pending) return SPGG_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaStreamSynchronize(h->pend_stream));
  CUDA_TRY(cudaGetLastError());
  if (h->spec && h->g.wrap_rows && h->pend_rel == h->pend_n && !h->pend_resident) {  // strips: spgg_strip_failed
    int rcode = rerun_failed_speculation(h);
    if (rcode) return rcode;
  }
  std::vector<int> stop(h->n_rep);
  CUDA_TRY(cudaMemcpy(stop.data(), h->d_stop, sizeof(int) * h->n_rep, cudaMemcpyDeviceToHost));
  // Replicas stop independently; plane parity is shared, so a stopped replica's planes are
  // copied forward to the parity the running replicas ended on (single-replica: adjust cur).
  const long long t_end = h->pend_t0 + h->pend_rel;
  for (int r = 0; r < h->n_rep; ++r) {
    h->stop_at[r] = stop[r];
    const long long done = (stop[r] >= 0 && stop[r] < t_end) ? (long long)stop[r] : t_end;
    double e = h->eps_cur[r];
    for (long long t = h->pend_t0; t < done; ++t)
      e = std::max(e * h->params[r].epsilon_decay, h->params[r].epsilon_min);  // algorithms.py:42
    h->eps_cur[r] = e;
  }
  if (h->pend_resident) {
    // the resident kernel wrote every replica's final state into plane set `cur`
    h->iter = (h->n_rep == 1 && stop[0] >= 0 && stop[0] < t_end) ? (long long)stop[0] : t_end;
    h->pend_resident = false;
  } else if (h->n_rep == 1 && stop[0] >= 0 && stop[0] < t_end) {
    h->cur = h->pend_cur0 ^ (int)((stop[0] - h->pend_t0) & 1);
    h->qcur = h->pend_q_after[(size_t)(stop[0] - h->pend_t0)];  // the launch that finished iteration stop[0] wrote Q last
    h->iter = stop[0];
  } else {
    if (h->n_rep > 1) {
      for (int r = 0; r < h->n_rep; ++r) {
        if (stop[r] >= 0 && stop[r] < t_end) {
          // k < 0: the replica stopped in an earlier chunk and no launch of this one touched it
          const long long k = (long long)stop[r] - h->pend_t0;
          const int src = k >= 0 ? (h->pend_cur0 ^ (int)(k & 1)) : h->pend_cur0;
          if (src != h->cur) {
            const Geom &g = h->g;
            CUDA_TRY(cudaMemcpy((char *)h->d_R[h->cur] + (size_t)r * g.plane_stride * h->elem_R(),
                                (char *)h->d_R[src] + (size_t)r * g.plane_stride * h->elem_R(),
                                (size_t)g.plane_stride * h->elem_R(), cudaMemcpyDeviceToDevice));
            CUDA_TRY(cudaMemcpy(h->d_S[h->cur] + (size_t)r * g.bits_stride,
                                h->d_S[src] + (size_t)r * g.bits_stride,
                                (size_t)g.bits_stride * 4, cudaMemcpyDeviceToDevice));
          }
          const int qsrc = k >= 0 ? h->pend_q_after[(size_t)k] : h->pend_qcur0;
          if (qsrc != h->qcur) {   // ping-pong Q: the stopped replica's table stayed in the other buffer
            const size_t qb = (size_t)h->g.site_stride * h->nq() * h->elem_Q();
            CUDA_TRY(cudaMemcpy((char *)h->d_Qb[h->qcur] + (size_t)r * qb, (char *)h->d_Qb[qsrc] + (size_t)r * qb, qb,
                                cudaMemcpyDeviceToDevice));
          }
        }
      }
    }
    h->iter = t_end;
  }
  h->pending = false;
  return SPGG_OK;
}

extern "C" int spgg_sync(spgg_t *h) {
  if (!h) return fail(SPGG_E_INVALID, "null handle");
  return finish_pending(h);
}

// ---------------------------------------------------------------- state I/O
// Host arrays are staged through device scratch in row chunks and packed/unpacked by
// kernels (k_import_rows / k_export_rows), so host<->device copies are plain memcpys of the
// reference's own array layouts.
static int stage_rows(const spgg_handle *h) {
  const long long budget = 32ll << 20;  // sites per chunk
  return (int)std::max<long long>(1, std::min<long long>(h->g.rows, budget / h->g.L));
}

static int ensure_scratch(spgg_handle *h, bool want_q) {
  const size_t n = (size_t)stage_rows(h) * h->g.L;
  if (!h->d_sc_S) {
    CUDA_TRY(cudaMalloc((void **)&h->d_sc_S, n));
    CUDA_TRY(cudaMalloc((void **)&h->d_sc_R, n * sizeof(double)));
    CUDA_TRY(cudaMalloc((void **)&h->d_sc_info, 3 * sizeof(unsigned long long)));
  }
  if (want_q && !h->d_sc_Q) CUDA_TRY(cudaMalloc((void **)&h->d_sc_Q, n * h->nq() * sizeof(double)));
  return SPGG_OK;
}

// a state upload after iterations have run starts a new run (include/spgg.h): the handle-wide
// iteration counter rewinds and the other replicas must be given a state before stepping
static void begin_new_run(spgg_handle *h, int rep) {
  if (h->iter != 0) {
    h->iter = 0;
    std::fill(h->stale.begin(), h->stale.end(), 1);
  }
  h->stale[rep] = 0;
  h->carry_valid = false;  // the global maximum of the run before says nothing about this one
  if (h->d_ring) {         // ring mode: a new run starts with empty slots (the caller synchronises the ranks)
    cudaMemset(h->d_ring, 0, sizeof(unsigned) * RING_SLOTS * RING_WORDS);
    h->gen = 0;
    h->last_gen = -1;
  }
}

extern "C" int spgg_set_state(spgg_t *h, int rep, const uint8_t *S, const double *R, const double *Q) {
  if (!h || !S || !R || !Q) return fail(SPGG_E_INVALID, "spgg_set_state: null argument");
  if (rep < 0 || rep >= h->n_rep) return fail(SPGG_E_INVALID, "replica %d out of range", rep);
  int rcode = finish_pending(h);
  if (rcode) return rcode;
  h->ccl_valid = h->ccl_local = false;
  CUDA_TRY(cudaSetDevice(h->device));
  rcode = ensure_scratch(h, true);
  if (rcode) return rcode;
  const Geom &g = h->g;
  const RepConst &rc = h->rc_host[rep];
  CUDA_TRY(cudaMemset(h->d_sc_info, 0, 3 * sizeof(unsigned long long)));
  const int chunk = stage_rows(h);
  for (int i0 = 0; i0 < g.rows; i0 += chunk) {
    const int nr = std::min(chunk, g.rows - i0);
    const size_t n = (size_t)nr * g.L, off = (size_t)i0 * g.L;
    CUDA_TRY(cudaMemcpyAsync(h->d_sc_S, S + off, n, cudaMemcpyHostToDevice, 0));
    CUDA_TRY(cudaMemcpyAsync(h->d_sc_R, R + off, n * sizeof(double), cudaMemcpyHostToDevice, 0));
    CUDA_TRY(cudaMemcpyAsync(h->d_sc_Q, Q + off * h->nq(), n * h->nq() * sizeof(double), cudaMemcpyHostToDevice, 0));
    const int grid = (int)std::min<long long>(148 * 16, ((long long)nr * ((g.L + 31) / 32) * 32 + 255) / 256);
    with_mode(h->mode, [&](auto md) {
      k_import_rows<decltype(md)><<<std::max(1, grid), 256>>>(g, rep, i0, nr, h->d_sc_S, h->d_sc_R, h->d_sc_Q,
          h->Qcur(), h->d_R[h->cur], h->d_S[h->cur], rc.rq, h->d_sc_info, h->nq());
    });
    CUDA_TRY(cudaGetLastError());
    h->launches += 1;
  }
  unsigned long long info[3];
  CUDA_TRY(cudaMemcpy(info, h->d_sc_info, sizeof(info), cudaMemcpyDeviceToHost));
  if (info[0] == 1) return fail(SPGG_E_INVALID, "strategy array holds values other than 0/1");
  if (info[0] == 2)
    return fail(SPGG_E_INVALID, "R is not representable in int8 units of %g; use r_storage=FP32", rc.rq);
  if (info[2] && h->fast) {
    // a strip's boundary rows reach its neighbours from k_step_fast itself (peer-mapped stores, the
    // report ring), so a strip cannot take the k_step detour of the whole lattice
    if (!g.wrap_rows)
      return fail(SPGG_E_INVALID, "R outside [%g, %g] (int8 units -16..15 of %g): a strip on the fast path "
                  "cannot hold it", -16.0 * rc.rq, 15.0 * rc.rq, rc.rq);
    h->r_wide = true;
  }
  begin_new_run(h, rep);
  h->eps_cur[rep] = h->params[rep].epsilon;
  int stop = -1;
  if (g.wrap_rows && (info[1] == 0 || info[1] == (unsigned long long)g.site_stride))
    stop = (int)h->iter;  // uniform start: iteration iter+1 breaks (spgg.py:405)
  h->stop_at[rep] = stop;
  CUDA_TRY(cudaMemcpy(h->d_stop + rep, &stop, sizeof(int), cudaMemcpyHostToDevice));
  return SPGG_OK;
}

extern "C" int spgg_get_state(spgg_t *h, int rep, uint8_t *S, double *R, double *Q) {
  if (!h) return fail(SPGG_E_INVALID, "null handle");
  if (rep < 0 || rep >= h->n_rep) return fail(SPGG_E_INVALID, "replica %d out of range", rep);
  int rcode = finish_pending(h);
  if (rcode) return rcode;
  CUDA_TRY(cudaSetDevice(h->device));
  rcode = ensure_scratch(h, Q != nullptr);
  if (rcode) return rcode;
  const Geom &g = h->g;
  const RepConst &rc = h->rc_host[rep];
  const int chunk = stage_rows(h);
  for (int i0 = 0; i0 < g.rows; i0 += chunk) {
    const int nr = std::min(chunk, g.rows - i0);
    const size_t n = (size_t)nr * g.L, off = (size_t)i0 * g.L;
    const int grid = (int)std::min<long long>(148 * 16, ((long long)n + 255) / 256);
    with_mode(h->mode, [&](auto md) {
      k_export_rows<decltype(md)><<<std::max(1, grid), 256>>>(g, rep, i0, nr, S ? h->d_sc_S : nullptr,
          R ? h->d_sc_R : nullptr, Q ? h->d_sc_Q : nullptr, h->Qcur(), h->d_R[h->cur], h->d_S[h->cur], rc.rq, h->nq());
    });
    CUDA_TRY(cudaGetLastError());
    h->launches += 1;
    if (S) CUDA_TRY(cudaMemcpyAsync(S + off, h->d_sc_S, n, cudaMemcpyDeviceToHost, 0));
    if (R) CUDA_TRY(cudaMemcpyAsync(R + off, h->d_sc_R, n * sizeof(double), cudaMemcpyDeviceToHost, 0));
    if (Q) CUDA_TRY(cudaMemcpyAsync(Q + off * h->nq(), h->d_sc_Q, n * h->nq() * sizeof(double), cudaMemcpyDeviceToHost, 0));
    CUDA_TRY(cudaStreamSynchronize(0));
  }
  return SPGG_OK;
}

extern "C" int spgg_set_replay(spgg_t *h, int n_steps, const double *u, const uint8_t *b) {
  return spgg_set_replay_pairs(h, n_steps, 1, u, b);
}

extern "C" int spgg_set_replay_pairs(spgg_t *h, int n_steps, int n_pairs, const double *u, const uint8_t *b) {
  if (!h) return fail(SPGG_E_INVALID, "null handle");
  const int want_pairs = h->params[0].algorithm == SPGG_ALGO_SARSA ? 3
                         : (h->params[0].algorithm == SPGG_ALGO_DOUBLE_QLEARNING ? 2 : 1);
  if (n_steps > 0 && n_pairs != want_pairs)
    return fail(SPGG_E_INVALID, "this TD rule consumes %d draw pair(s) per iteration, got %d", want_pairs, n_pairs);
  if (h->n_rep != 1) return fail(SPGG_E_UNSUPPORTED, "replay draws are supported for a single replica");
  int rcode = finish_pending(h);
  if (rcode) return rcode;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaFree(h->d_u); cudaFree(h->d_b);
  h->d_u = nullptr; h->d_b = nullptr; h->replay_n = 0;
  if (n_steps <= 0) return SPGG_OK;
  if (!u || !b) return fail(SPGG_E_INVALID, "spgg_set_replay: null draw arrays");
  const size_t n = (size_t)n_steps * n_pairs * h->g.site_stride;
  h->replay_pairs = n_pairs;
  CUDA_TRY(cudaMalloc((void **)&h->d_u, n * sizeof(double)));
  CUDA_TRY(cudaMalloc((void **)&h->d_b, n));
  CUDA_TRY(cudaMemcpy(h->d_u, u, n * sizeof(double), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(h->d_b, b, n, cudaMemcpyHostToDevice));
  h->replay_first = h->iter;
  h->replay_n = n_steps;
  return SPGG_OK;
}

// ---------------------------------------------------------------- stepping
static int ensure_tables(spgg_handle *h, int n_steps) {
  const int need = n_steps + 1;
  if (need <= h->cap) return SPGG_OK;
  cudaFree(h->d_gmax); cudaFree(h->d_stats); cudaFree(h->d_eps); cudaFree(h->d_thr); cudaFree(h->d_gvec);
  h->d_gmax = nullptr; h->d_stats = nullptr; h->d_eps = nullptr; h->d_thr = nullptr; h->d_gvec = nullptr;
  h->cap = 0;
  CUDA_TRY(cudaMalloc(&h->d_gmax, h->elem_val() * (size_t)h->n_rep * need));
  CUDA_TRY(cudaMalloc((void **)&h->d_stats, sizeof(double) * (size_t)h->n_rep * need * NSTAT));
  CUDA_TRY(cudaMalloc((void **)&h->d_eps, sizeof(double) * (size_t)h->n_rep * (need + 1)));
  CUDA_TRY(cudaMalloc((void **)&h->d_thr, sizeof(uint32_t) * (size_t)h->n_rep * (need + 1)));
  if (h->spec && !h->g.wrap_rows) CUDA_TRY(cudaMalloc((void **)&h->d_gvec, sizeof(float) * 4 * (size_t)need));
  h->cap = need;
  return SPGG_OK;
}

static uint32_t thr24(double eps) {
  double t = std::ceil(eps * 16777216.0);
  if (t < 0) t = 0;
  if (t > 16777216.0) t = 16777216.0;
  return (uint32_t)t;
}

extern "C" int spgg_begin_steps(spgg_t *h, int n_steps, void *stream_) {
  if (!h) return fail(SPGG_E_INVALID, "null handle");
  if (n_steps < 1) return fail(SPGG_E_INVALID, "n_steps must be >= 1");
  int rcode = finish_pending(h);
  if (rcode) return rcode;
  h->ccl_valid = h->ccl_local = false;
  for (int r = 0; r < h->n_rep; ++r)
    if (h->stale[r])
      return fail(SPGG_E_STATE, "replica %d still holds the state of the previous run: give every replica of a "
                                "batch a state (spgg_set_state / spgg_init_random) before stepping", r);
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream_;
  rcode = ensure_tables(h, n_steps);
  if (rcode) return rcode;
  // eps used at iteration iter+idx, idx = 1..n_steps (+1 spare entry); algorithms.py:40-42
  std::vector<double> &eps = h->eps_host;   // kept alive by the handle: the copies are async
  std::vector<uint32_t> &thr = h->thr_host;
  eps.assign((size_t)(h->cap + 1) * h->n_rep, 0.0);
  thr.assign(eps.size(), 0u);
  for (int r = 0; r < h->n_rep; ++r) {
    double e = h->eps_cur[r];
    for (int idx = 1; idx <= n_steps + 1 && idx <= h->cap; ++idx) {
      eps[(size_t)idx * h->n_rep + r] = e;
      thr[(size_t)idx * h->n_rep + r] = thr24(e);
      e = std::max(e * h->params[r].epsilon_decay, h->params[r].epsilon_min);
    }
  }
  CUDA_TRY(cudaMemcpyAsync(h->d_eps, eps.data(), eps.size() * sizeof(double), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(h->d_thr, thr.data(), thr.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemsetAsync(h->d_gmax, 0, h->elem_val() * (size_t)h->n_rep * h->cap, st));
  CUDA_TRY(cudaMemsetAsync(h->d_stats, 0, sizeof(double) * (size_t)h->n_rep * h->cap * NSTAT, st));
  if (h->d_gvec) CUDA_TRY(cudaMemsetAsync(h->d_gvec, 0, sizeof(float) * 4 * (size_t)h->cap, st));
  h->pending = true;
  h->pend_t0 = h->iter;
  h->pend_n = n_steps;
  h->pend_cur0 = h->cur;
  h->pend_qcur0 = h->qcur;
  h->in_rerun = false;
  h->pend_cur_after.assign((size_t)n_steps + 1, (char)h->cur);
  h->pend_q_after.assign((size_t)n_steps + 1, (char)h->qcur);
  h->pend_rel = 0;
  h->pend_stream = st;
  return SPGG_OK;
}

// does the launch that follows iteration index j (choosing the action of j+1) read replayed draws?
static bool launch_replays(const spgg_handle *h, long long j, int do_select) {
  const long long draw = j - h->replay_first;  // draws of iteration j+1 are entry `draw`
  return do_select && h->d_u && draw >= 0 && draw < h->replay_n;
}
// may the update launch that finishes iteration pend_rel+1 guess the global maximum (KArgs::spec)?
static bool can_speculate(const spgg_handle *h, int do_select) {
  return h->fast && h->spec && h->spec_on && h->carry_valid &&
         !launch_replays(h, h->pend_t0 + h->pend_rel + 1, do_select);
}

// one k_step launch at relative index pend_rel (finishing iteration pend_t0+pend_rel)
static int launch_step(spgg_handle *h, int do_update, int do_select, cudaStream_t st, bool allow_spec) {
  const long long j = h->pend_t0 + h->pend_rel;
  const long long draw = j - h->replay_first;  // draws of iteration j+1 are entry `draw`
  const bool replay = launch_replays(h, j, do_select);
  KArgs a;
  a.g = h->g;
  a.rc = h->d_rc;
  a.Q = h->Qcur();
  a.R_in = h->d_R[h->cur]; a.R_out = h->d_R[h->cur ^ 1];
  a.code_in = h->d_code[h->cur]; a.code_out = h->d_code[h->cur ^ 1];
  a.S_in = h->d_S[h->cur]; a.S_out = h->d_S[h->cur ^ 1];
  a.gmax = h->d_gmax; a.stats = h->d_stats; a.partials = h->d_partials;
  a.valtab = h->d_valtab;
  a.tickets = h->d_tickets; a.stop_at = h->d_stop;
  a.eps_tab = h->d_eps; a.thr_tab = h->d_thr;
  const size_t np_ = (size_t)h->replay_pairs, ss = (size_t)h->g.site_stride;
  a.u = replay ? h->d_u + (size_t)draw * np_ * ss : nullptr;
  a.b = replay ? h->d_b + (size_t)draw * np_ * ss : nullptr;
  a.algo = h->params[0].algorithm;
  // SARSA: pairs 1 and 2 of iteration j (entry j-1-replay_first) feed the update launched now
  const long long ue = j - 1 - h->replay_first;
  const bool upd_replay = do_update && np_ >= 2 && h->d_u && ue >= 0 && ue < h->replay_n;
  a.u2 = upd_replay ? h->d_u + ((size_t)ue * np_ + 1) * ss : nullptr;   // SARSA next action / Double-Q table choice
  a.b2 = upd_replay ? h->d_b + ((size_t)ue * np_ + 1) * ss : nullptr;
  a.u3 = (upd_replay && np_ == 3) ? h->d_u + ((size_t)ue * 3 + 2) * ss : nullptr;
  a.b3 = (upd_replay && np_ == 3) ? h->d_b + ((size_t)ue * 3 + 2) * ss : nullptr;
  a.j = (int)j; a.rel = h->pend_rel; a.cap = h->cap;
  a.do_update = do_update; a.do_select = do_select;
  const bool use_fast = h->fast && !replay && !(do_select && h->r_wide);
  a.spec = 0; a.gcarry = nullptr; a.bad_at = nullptr; a.gvec = nullptr;
  for (int d = 0; d < 2; ++d) {   // ghost rows of the neighbours' OUTPUT planes (parity cur^1), fast path only
    const bool on = h->peer_on && use_fast && do_select;
    a.peer_code[d] = on ? h->peer_code[d][h->cur ^ 1] : nullptr;
    a.peer_R[d] = on ? h->peer_R[d][h->cur ^ 1] : nullptr;
    a.peer_S[d] = on ? h->peer_S[d][h->cur ^ 1] : nullptr;
    a.peer_rows[d] = h->peer_rows[d];
  }
  a.ring_world = 0; a.gen = 0;
  for (int p = 0; p < SPGG_MAX_RING; ++p) a.ring_peer[p] = nullptr;
  if (h->ring_world > 0 && use_fast && h->d_gvec && (do_update || do_select)) {
    a.ring_world = h->ring_world;
    a.gen = h->gen;
    for (int p = 0; p < h->ring_world; ++p) a.ring_peer[p] = h->ring_peer[p];
  }
  if (use_fast && h->spec && !h->g.wrap_rows && h->n_rep == 1) a.gvec = h->d_gvec;
  if (use_fast && h->spec) {
    a.gcarry = h->d_gcarry;
    a.bad_at = h->d_bad;
    a.spec = (allow_spec && do_update && h->spec_on && h->carry_valid) ? 1 : 0;
  }
#ifdef SPGG_TRACE
  {  // debug builds only: dump the per-CTA timeline of the previous fused launch
    static unsigned long long *d_trace = nullptr;
    static int n_dump = 0;
    const int n_cta = h->g.ctas_per_rep * h->n_rep;
    if (!d_trace) { cudaMalloc(&d_trace, sizeof(unsigned long long) * 4 * 65536); cudaMemset(d_trace, 0, sizeof(unsigned long long) * 4 * 65536); }
    else if (getenv("SPGG_TRACE_FILE") && n_dump < 3 && do_update && do_select) {
      std::vector<unsigned long long> t(4 * (size_t)n_cta);
      cudaDeviceSynchronize();
      cudaMemcpy(t.data(), d_trace, t.size() * 8, cudaMemcpyDeviceToHost);
      char name[256]; snprintf(name, sizeof(name), "%s.%d", getenv("SPGG_TRACE_FILE"), n_dump++);
      FILE *f = fopen(name, "wb"); if (f) { fwrite(t.data(), 8, t.size(), f); fclose(f); }
    }
    a.trace = d_trace;
  }
#endif
  if (use_fast) {
    if (!do_update && !do_select) return SPGG_OK;
    fast_fn_t ff = pick_fast(h->M, h->action, do_update, do_select, h->g.L % TC != 0);
    FastMaps fm = h->fmaps[h->cur];
    const int q_out = (do_update && h->spec) ? (h->qcur ^ 1) : h->qcur;   // ping-pong only where a re-run must be possible
    fm.q_ld = h->qmaps[h->qcur];
    fm.q_st = h->qmaps[q_out];
    if (a.spec) {
      // test hook (tests/test_gpu_speculation.py): SPGG_SPEC_TEST_POISON=n makes every n-th speculative
      // launch guess a value that cannot be right (spec = 2), so the re-run path is exercised on demand
      static const int poison = getenv("SPGG_SPEC_TEST_POISON") ? atoi(getenv("SPGG_SPEC_TEST_POISON")) : 0;
      if (poison > 0 && !h->in_rerun && h->spec_launches % poison == poison - 1) a.spec = 2;
    }
    CUDA_TRY(launch_pdl(ff, h->g.ctas_per_rep * h->n_rep, FTHREADS, fast_smem(h->M), st, fm, a));
    h->qcur = q_out;
    if (do_update) {
      h->carry_valid = h->spec;   // every fast update launch leaves its own exact maximum in gcarry
      if (a.spec) {
        h->spec_launches += 1;
        if (!h->in_rerun) h->spec_iterations += 1;
      }
    }
  } else {
    if (do_update) h->carry_valid = false;
    step_fn_t f = (h->lean && do_update) ? pick_lean(h->mode, h->M, h->action, replay ? 1 : 0)
                                          : pick_step(h->mode, h->M, h->action, replay ? 1 : 0);
    // programmatic dependent launch pays only when a launch is short (at most one tile per SM;
    // measured: 25.0 -> 23.4 us per iteration at L=100, but 366 -> 428 us for 60 batched L=200 replicas)
    const int grid = h->g.ctas_per_rep * h->n_rep;
    if ((long long)h->g.n_tx * h->g.n_ty * h->n_rep <= 160) CUDA_TRY(launch_pdl(f, grid, h->threads, h->smem_step, st, a));
    else f<<<grid, h->threads, h->smem_step, st>>>(a);
  }
  CUDA_TRY(cudaGetLastError());
  h->launches += 1;
  h->last_rel = h->pend_rel; h->last_upd = do_update; h->last_spec = a.spec; h->last_sel = do_select;
  h->last_gen = a.ring_world > 0 ? h->gen++ : -1;
  if (do_select) {
    h->cur ^= 1;
    h->r_wide = false;   // every R was just clipped into [R_min, R_max]
  }
  if (h->pend_rel >= 0 && h->pend_rel < (int)h->pend_cur_after.size()) {
    h->pend_cur_after[h->pend_rel] = (char)h->cur;
    h->pend_q_after[h->pend_rel] = (char)h->qcur;
  }
  return SPGG_OK;
}

extern "C" int spgg_phase_kernel(spgg_t *h, int do_update, int do_select, void *stream_) {
  if (!h || !h->pending) return fail(SPGG_E_STATE, "spgg_phase_kernel outside begin/end");
  return launch_step(h, do_update, do_select, (cudaStream_t)stream_, false);  // the caller supplies the exact maximum
}

// finish the next iteration (and choose the action of the one after it when do_select): one speculative
// launch when the handle can guess the global maximum, else the exact pair (maximum kernel, then update kernel)
extern "C" int spgg_phase_iteration(spgg_t *h, int do_select, void *stream_) {
  if (!h || !h->pending) return fail(SPGG_E_STATE, "spgg_phase_iteration outside begin/end");
  if (h->pend_rel >= h->pend_n) return fail(SPGG_E_STATE, "the chunk announced to spgg_begin_steps is complete");
  int rcode = SPGG_OK;
  if (can_speculate(h, do_select)) h->pend_rel += 1;
  else rcode = spgg_phase_gmax(h, stream_);
  if (!rcode) rcode = launch_step(h, 1, do_select, (cudaStream_t)stream_, true);
  return rcode;
}

// gmax of the iteration about to be finished (pend_rel+1); advances pend_rel
extern "C" int spgg_phase_gmax(spgg_t *h, void *stream_) {
  if (!h || !h->pending) return fail(SPGG_E_STATE, "spgg_phase_gmax outside begin/end");
  cudaStream_t st = (cudaStream_t)stream_;
  h->pend_rel += 1;
  GArgs a;
  a.g = h->g;
  a.rc = h->d_rc;
  a.code_in = h->d_code[h->cur];
  a.gmax = h->d_gmax;
  a.valtab = h->d_valtab;
  a.stop_at = h->d_stop;
  a.j = (int)(h->pend_t0 + h->pend_rel); a.rel = h->pend_rel; a.cap = h->cap;
  if (h->fast) {
    CUDA_TRY(launch_pdl(pick_gfast(h->M), h->gmax_ctas * h->n_rep, GWARPS * 32, gfast_smem(h->M), st,
                        h->fmaps[h->cur].ld_code, a));
  } else {
    gmax_fn_t f = pick_gmax_lean(h->mode, h->M);
    a.g.ctas_per_rep = h->gmax_ctas_gen;   // a light kernel: its own persistent grid (more CTAs per SM than k_step)
    const int grid = h->gmax_ctas_gen * h->n_rep;
    if ((long long)h->g.n_tx * h->g.n_ty * h->n_rep <= 160) CUDA_TRY(launch_pdl(f, grid, h->threads, h->smem_gmax, st, a));
    else f<<<grid, h->threads, h->smem_gmax, st>>>(a);
  }
  CUDA_TRY(cudaGetLastError());
  h->launches += 1;
  return SPGG_OK;
}

extern "C" void *spgg_gmax_device_ptr(spgg_t *h) {
  if (!h || !h->pending) return nullptr;
  return (char *)h->d_gmax + h->elem_val() * (size_t)h->pend_rel;  // replica 0
}

extern "C" int spgg_end_steps(spgg_t *h, void *stream_) {
  (void)stream_;
  if (!h || !h->pending) return fail(SPGG_E_STATE, "spgg_end_steps without spgg_begin_steps");
  return SPGG_OK;  // bookkeeping is finished lazily by the next synchronising call
}

// the whole chunk in one launch: one cluster per replica keeps its lattice in shared memory
static int resident_chunk(spgg_handle *h, int n_steps, cudaStream_t st) {
  RArgs a;
  a.g = h->g;
  a.rg = h->rgeo;
  a.rc = h->d_rc;
  a.Q = h->Qcur();
  a.R = h->d_R[h->cur];
  a.S = h->d_S[h->cur];
  a.stats = h->d_stats;
  a.stop_at = h->d_stop;
  a.thr_tab = h->d_thr;
  a.t0 = (int)h->pend_t0;
  a.n_steps = n_steps;
  a.cap = h->cap;
#ifdef SPGG_RES_TRACE
  {  // debug builds only: print the per-phase cycle sums of the previous resident launch
    static long long *d_tr = nullptr;
    const int n_cta = h->rgeo.CS * h->n_rep;
    if (!d_tr) { cudaMalloc(&d_tr, sizeof(long long) * 8 * 4096); cudaMemset(d_tr, 0, sizeof(long long) * 8 * 4096); }
    else if (getenv("SPGG_RES_TRACE_PRINT")) {
      std::vector<long long> t(8 * (size_t)n_cta);
      cudaDeviceSynchronize();
      cudaMemcpy(t.data(), d_tr, t.size() * 8, cudaMemcpyDeviceToHost);
      for (int c = 0; c < std::min(n_cta, 16); ++c) {
        fprintf(stderr, "res_trace cta %2d:", c);
        for (int z = 0; z < 7; ++z) fprintf(stderr, " %10lld", t[(size_t)c * 8 + z]);
        fprintf(stderr, "\n");
      }
    }
    a.trace = d_tr;
  }
#endif
  a.gimg = h->d_gimg;
  a.gpart = h->d_gpart;
  a.gnsel = nullptr;
  a.gmaxtab = reinterpret_cast<float *>(h->d_gmax);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(h->rgeo.CS * h->n_rep));
  cfg.blockDim = dim3((unsigned)h->rgeo.threads);
  cfg.dynamicSmemBytes = h->smem_res;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (h->res_grid) {
    if (h->gnsel_cap < h->cap) {
      cudaFree(h->d_gnsel);
      h->d_gnsel = nullptr; h->gnsel_cap = 0;
      CUDA_TRY(cudaMalloc((void **)&h->d_gnsel, sizeof(unsigned) * (size_t)h->cap));
      h->gnsel_cap = h->cap;
    }
    CUDA_TRY(cudaMemsetAsync(h->d_gnsel, 0, sizeof(unsigned) * (size_t)h->cap, st));
    a.gnsel = h->d_gnsel;
    attr[0].id = cudaLaunchAttributeCooperative;   // every block resident at once: grid-wide barriers
    attr[0].val.cooperative = 1;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, pick_res_grid(h->M, h->action, h->g.L), a));
  } else {
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)h->rgeo.CS;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, pick_res(h->M, h->action, h->g.L), a));
  }
  {  // raw statistics rows -> public layout
    const int n_rows = n_steps + 1, total = n_rows * h->n_rep;
    k_resident_rows<<<(total + 127) / 128, 128, 0, st>>>(h->d_rc, h->d_stats, h->n_rep, h->cap, n_rows);
    CUDA_TRY(cudaGetLastError());
  }
  h->launches += 2;
  h->pend_rel = n_steps;
  h->pend_resident = true;
  return SPGG_OK;
}

extern "C" int spgg_step(spgg_t *h, int n_steps, void *stream_) {
  int rcode = spgg_begin_steps(h, n_steps, stream_);
  if (rcode) return rcode;
  if (h->resident && !h->d_u) {  // replayed draws go through the general kernel
    rcode = resident_chunk(h, n_steps, (cudaStream_t)stream_);
    if (rcode) return rcode;
    return spgg_end_steps(h, stream_);
  }
  rcode = spgg_phase_kernel(h, 0, 1, stream_);  // choose the action of iteration iter+1
  for (int s = 1; s <= n_steps && !rcode; ++s) rcode = spgg_phase_iteration(h, s < n_steps ? 1 : 0, stream_);
  if (rcode) return rcode;
  return spgg_end_steps(h, stream_);
}

extern "C" int spgg_get_stats(spgg_t *h, int rep, int first, int n, double *rows_out) {
  if (!h || !rows_out) return fail(SPGG_E_INVALID, "spgg_get_stats: null argument");
  if (rep < 0 || rep >= h->n_rep) return fail(SPGG_E_INVALID, "replica %d out of range", rep);
  int rcode = finish_pending(h);
  if (rcode) return rcode;
  if (first < 0 || n < 0 || first + n > h->cap) return fail(SPGG_E_INVALID, "rows [%d,%d) outside the last chunk (%d rows)", first, first + n, h->cap);
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaMemcpy(rows_out, h->d_stats + ((size_t)rep * h->cap + first) * NSTAT,
                      sizeof(double) * (size_t)n * NSTAT, cudaMemcpyDeviceToHost));
  return SPGG_OK;
}

extern "C" int spgg_query(spgg_t *h, int rep, spgg_status_t *out) {
  if (!h || !out) return fail(SPGG_E_INVALID, "spgg_query: null argument");
  if (rep < 0 || rep >= h->n_rep) return fail(SPGG_E_INVALID, "replica %d out of range", rep);
  int rcode = finish_pending(h);
  if (rcode) return rcode;
  out->iteration = (h->stop_at[rep] >= 0 && h->stop_at[rep] < h->iter) ? h->stop_at[rep] : h->iter;
  out->stopped_at = h->stop_at[rep];
  out->epsilon = h->eps_cur[rep];
  out->n_replicas = h->n_rep;
  out->r_is_int8 = h->mode == MODE_F32_I8;
  out->kernel_launches = h->launches;
  out->speculative_launches = h->spec_launches;
  out->speculation_failures = h->spec_failures;
  return SPGG_OK;
}

extern "C" int spgg_describe(spgg_t *h, char *buf, int n) {
  if (!h) return fail(SPGG_E_INVALID, "null handle");
  char tmp[256];
  const char *arith = h->mode == MODE_F64 ? "fp64 Q and R" : (h->mode == MODE_F32_F ? "fp32 Q, fp32 R" : "fp32 Q, int8 R");
  int len;
  if (h->resident && h->res_grid)
    len = snprintf(tmp, sizeof(tmp), "resident: cooperative grid of %d CTAs x %d threads, %zu KB shared memory per CTA, "
                   "ghost rows through L2 (%s)", h->rgeo.CS, h->rgeo.threads, h->smem_res >> 10, arith);
  else if (h->resident)
    len = snprintf(tmp, sizeof(tmp), "resident: cluster of %d CTAs x %d threads per replica, %zu KB shared memory per CTA, "
                   "ghost rows through DSMEM (%s)", h->rgeo.CS, h->rgeo.threads, h->smem_res >> 10, arith);
  else if (h->fast)
    len = snprintf(tmp, sizeof(tmp), "fast: TMA-staged %dx%d tiles, %d persistent CTAs per replica, %s (%s)",
                   FTR, TC, h->g.ctas_per_rep,
                   (h->spec && h->spec_on) ? "one launch per iteration (speculative global maximum, verified)"
                                           : "two launches per iteration (k_gmax_fast + k_step_fast)", arith);
  else
    len = snprintf(tmp, sizeof(tmp), "general: %dx%d tiles, %d CTAs per replica, two launches per iteration (k_gmax_lean + %s) (%s)", h->g.TR, TC,
                   h->g.ctas_per_rep, h->lean ? "k_step_lean" : "k_step", arith);
  if (buf && n > 0) {
    strncpy(buf, tmp, (size_t)n - 1);
    buf[n - 1] = 0;
  }
  return len + 1;
}

// device-side random initial state (distributions of spgg.py:121,129,162)
extern "C" int spgg_init_random(spgg_t *h, int rep, uint64_t seed) {
  if (!h) return fail(SPGG_E_INVALID, "null handle");
  if (rep < 0 || rep >= h->n_rep) return fail(SPGG_E_INVALID, "replica %d out of range", rep);
  int rcode = finish_pending(h);
  if (rcode) return rcode;
  h->ccl_valid = h->ccl_local = false;
  CUDA_TRY(cudaSetDevice(h->device));
  const uint32_t lo = (uint32_t)seed, hi = (uint32_t)(seed >> 32);
  const int grid = 148 * 8;
  with_mode(h->mode, [&](auto md) {
    k_init_random<decltype(md)><<<grid, 256>>>(h->g, rep, h->Qcur(), h->d_R[h->cur], h->d_S[h->cur], lo, hi, h->nq());
  });
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaDeviceSynchronize());
  h->launches += 1;
  begin_new_run(h, rep);
  h->eps_cur[rep] = h->params[rep].epsilon;
  int stop = -1;
  h->stop_at[rep] = -1;
  CUDA_TRY(cudaMemcpy(h->d_stop + rep, &stop, sizeof(int), cudaMemcpyHostToDevice));
  return SPGG_OK;
}

// ---------------------------------------------------------------- checkpoint / digests
extern "C" int spgg_set_progress(spgg_t *h, int64_t iteration, const double *epsilon) {
  if (!h || !epsilon) return fail(SPGG_E_INVALID, "spgg_set_progress: null argument");
  if (iteration < 0 || iteration > 0x7fffffff - (1 << 20))
    return fail(SPGG_E_INVALID, "iteration %lld outside the 31-bit Philox counter word", (long long)iteration);
  int rcode = finish_pending(h);
  if (rcode) return rcode;
  for (int r = 0; r < h->n_rep; ++r) {
    if (h->stale[r]) return fail(SPGG_E_STATE, "replica %d has no state of the run being resumed", r);
    if (!(epsilon[r] >= 0.0 && epsilon[r] <= 1.0)) return fail(SPGG_E_INVALID, "epsilon[%d] = %g outside [0, 1]", r, epsilon[r]);
  }
  if (h->iter != 0) return fail(SPGG_E_STATE, "spgg_set_progress follows the state uploads of a resumed run");
  h->ccl_valid = h->ccl_local = false;
  CUDA_TRY(cudaSetDevice(h->device));
  h->iter = (long long)iteration;
  h->replay_first = h->iter;
  for (int r = 0; r < h->n_rep; ++r) {
    h->eps_cur[r] = epsilon[r];
    if (h->stop_at[r] >= 0) h->stop_at[r] = h->iter;  // uniform lattice uploaded: iteration iter+1 breaks
  }
  std::vector<int> stop(h->stop_at.begin(), h->stop_at.end());
  CUDA_TRY(cudaMemcpy(h->d_stop, stop.data(), sizeof(int) * h->n_rep, cudaMemcpyHostToDevice));
  return SPGG_OK;
}

extern "C" int spgg_state_digest(spgg_t *h, int rep, uint64_t out[3]) {
  if (!h || !out) return fail(SPGG_E_INVALID, "spgg_state_digest: null argument");
  if (rep < 0 || rep >= h->n_rep) return fail(SPGG_E_INVALID, "replica %d out of range", rep);
  int rcode = finish_pending(h);
  if (rcode) return rcode;
  CUDA_TRY(cudaSetDevice(h->device));
  unsigned long long *d_out = nullptr;
  CUDA_TRY(cudaMalloc((void **)&d_out, 3 * sizeof(unsigned long long)));
  CUDA_TRY(cudaMemset(d_out, 0, 3 * sizeof(unsigned long long)));
  const int grid = 148 * 8;
  const double rq = h->rc_host[rep].rq;
  with_mode(h->mode, [&](auto md) {
    k_state_digest<decltype(md)><<<grid, 256>>>(h->g, rep, h->Qcur(), h->d_R[h->cur], h->d_S[h->cur], h->nq(), rq, d_out);
  });
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpy(out, d_out, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
  cudaFree(d_out);
  if (e != cudaSuccess) return fail(SPGG_E_CUDA, "spgg_state_digest: %s", cudaGetErrorString(e));
  h->launches += 1;
  return SPGG_OK;
}

extern "C" int spgg_r_histogram(spgg_t *h, int rep, int n_bins, const double *edges, int64_t *counts) {
  if (!h || !edges || !counts) return fail(SPGG_E_INVALID, "spgg_r_histogram: null argument");
  if (rep < 0 || rep >= h->n_rep) return fail(SPGG_E_INVALID, "replica %d out of range", rep);
  if (n_bins < 1 || n_bins > 64) return fail(SPGG_E_INVALID, "n_bins must be in [1, 64] (got %d)", n_bins);
  int rcode = finish_pending(h);
  if (rcode) return rcode;
  CUDA_TRY(cudaSetDevice(h->device));
  double *d_edges = nullptr;
  unsigned long long *d_cnt = nullptr;
  CUDA_TRY(cudaMalloc((void **)&d_edges, sizeof(double) * 65));
  if (cudaMalloc((void **)&d_cnt, sizeof(unsigned long long) * 64) != cudaSuccess) { cudaFree(d_edges); return fail(SPGG_E_CUDA, "cudaMalloc failed"); }
  cudaMemcpy(d_edges, edges, sizeof(double) * (n_bins + 1), cudaMemcpyHostToDevice);
  cudaMemset(d_cnt, 0, sizeof(unsigned long long) * 64);
  const double rq = h->rc_host[rep].rq;
  const int grid = 148 * 8;
  with_mode(h->mode, [&](auto md) {
    k_r_histogram<decltype(md)><<<grid, 256>>>(h->g, rep, h->d_R[h->cur], rq, n_bins, d_edges, d_cnt);
  });
  unsigned long long host_cnt[64];
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpy(host_cnt, d_cnt, sizeof(unsigned long long) * 64, cudaMemcpyDeviceToHost);
  cudaFree(d_edges); cudaFree(d_cnt);
  if (e != cudaSuccess) return fail(SPGG_E_CUDA, "spgg_r_histogram: %s", cudaGetErrorString(e));
  for (int i = 0; i < n_bins; ++i) counts[i] = (int64_t)host_cnt[i];
  h->launches += 1;
  return SPGG_OK;
}

// ---------------------------------------------------------------- clusters
// scipy.ndimage.label of one replica's strategies (include/spgg.h); the kernels live in spgg_clusters.cu
extern "C" int spgg_clusters(spgg_t *h, int rep, int which, int flags, int64_t *n_clusters) {
  if (!h || !n_clusters) return fail(SPGG_E_INVALID, "spgg_clusters: null argument");
  if (rep < 0 || rep >= h->n_rep) return fail(SPGG_E_INVALID, "replica %d out of range", rep);
  if (which != 0 && which != 1) return fail(SPGG_E_INVALID, "which must be 0 (cooperators) or 1 (defectors), got %d", which);
  if (flags & ~SPGG_CLUSTER_PERIODIC) return fail(SPGG_E_INVALID, "unknown cluster flags 0x%x", flags);
  if (!h->g.wrap_rows) return fail(SPGG_E_UNSUPPORTED, "cluster labelling needs the whole lattice (rows == L), not a strip");
  if ((long long)h->g.rows * h->g.L >= (1ll << 31)) return fail(SPGG_E_UNSUPPORTED, "cluster labelling needs rows*L < 2^31");
  int rcode = finish_pending(h);
  if (rcode) return rcode;
  h->ccl_valid = h->ccl_local = false;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaError_t e = ccl_alloc(&h->ccl, h->g.rows, h->g.L);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    return fail(SPGG_E_CUDA, "spgg_clusters: scratch for L=%d: %s", h->g.L, cudaGetErrorString(e));
  }
  const Geom &g = h->g;
  const uint32_t *S = h->d_S[h->cur] + (size_t)rep * g.bits_stride + (size_t)GH * g.pitchW + WPAD;
  int64_t n = 0;
  e = launch_clusters(h->ccl, S, g.pitchW, which, flags & SPGG_CLUSTER_PERIODIC, &n);
  if (e != cudaSuccess) return fail(SPGG_E_CUDA, "spgg_clusters: %s", cudaGetErrorString(e));
  h->launches += 5;
  h->ccl.base = 0;
  h->ccl_n = n;
  h->ccl_valid = true;
  *n_clusters = n;
  return SPGG_OK;
}

extern "C" int spgg_cluster_sizes(spgg_t *h, int64_t *sizes, int64_t n) {
  if (!h || !sizes) return fail(SPGG_E_INVALID, "spgg_cluster_sizes: null argument");
  if (!h->ccl_valid) return fail(SPGG_E_STATE, "spgg_cluster_sizes: no spgg_clusters result for the current state");
  if (n != h->ccl_n) return fail(SPGG_E_INVALID, "spgg_cluster_sizes: n = %lld, the labelling found %lld clusters", (long long)n, (long long)h->ccl_n);
  CUDA_TRY(cudaSetDevice(h->device));
  if (n > 0) CUDA_TRY(cudaMemcpy(sizes, h->ccl.sizes, sizeof(int64_t) * (size_t)n, cudaMemcpyDeviceToHost));
  return SPGG_OK;
}

extern "C" int spgg_cluster_labels(spgg_t *h, int32_t *labels) {
  if (!h || !labels) return fail(SPGG_E_INVALID, "spgg_cluster_labels: null argument");
  if (!h->ccl_valid) return fail(SPGG_E_STATE, "spgg_cluster_labels: no spgg_clusters result for the current state");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaError_t e = launch_cluster_labels(h->ccl);
  if (e == cudaSuccess)
    e = cudaMemcpy(labels, h->ccl.total, sizeof(int32_t) * (size_t)h->g.rows * h->g.L, cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) return fail(SPGG_E_CUDA, "spgg_cluster_labels: %s", cudaGetErrorString(e));
  h->launches += 1;
  return SPGG_OK;
}

// Row strips (include/spgg.h): the strip-local labelling writes a boundary record; the records of all
// ranks, gathered by the caller, are resolved into this strip's part of the whole lattice's labelling
static int strip_clusters_supported(spgg_t *h, const char *fn) {
  if (h->n_rep != 1) return fail(SPGG_E_UNSUPPORTED, "%s: strip labelling serves single-replica handles", fn);
  if ((long long)h->g.L * h->g.L >= (1ll << 31))
    return fail(SPGG_E_UNSUPPORTED, "%s: global site indices need L*L < 2^31 (L=%d)", fn, h->g.L);
  return SPGG_OK;
}

extern "C" int64_t spgg_strip_cluster_record_bytes(spgg_t *h) {
  if (!h) return fail(SPGG_E_INVALID, "null handle");
  int rcode = strip_clusters_supported(h, "spgg_strip_cluster_record_bytes");
  return rcode ? rcode : ccl_record_bytes(h->g.L);
}

extern "C" int spgg_strip_clusters(spgg_t *h, int which, int flags, void *dev_record) {
  if (!h || !dev_record) return fail(SPGG_E_INVALID, "spgg_strip_clusters: null argument");
  if (which != 0 && which != 1) return fail(SPGG_E_INVALID, "which must be 0 (cooperators) or 1 (defectors), got %d", which);
  if (flags & ~SPGG_CLUSTER_PERIODIC) return fail(SPGG_E_INVALID, "unknown cluster flags 0x%x", flags);
  int rcode = strip_clusters_supported(h, "spgg_strip_clusters");
  if (rcode) return rcode;
  rcode = finish_pending(h);
  if (rcode) return rcode;
  h->ccl_valid = h->ccl_local = false;
  CUDA_TRY(cudaSetDevice(h->device));
  const Geom &g = h->g;
  cudaError_t e = ccl_alloc(&h->ccl, g.rows, g.L);
  if (e == cudaSuccess) e = ccl_strip_alloc(&h->ccl_strip, g.L, 0);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    return fail(SPGG_E_CUDA, "spgg_strip_clusters: scratch for %d x %d sites: %s", g.rows, g.L, cudaGetErrorString(e));
  }
  const uint32_t *S = h->d_S[h->cur] + (size_t)GH * g.pitchW + WPAD;
  e = launch_strip_clusters(h->ccl, h->ccl_strip, S, g.pitchW, g.row0, which, flags & SPGG_CLUSTER_PERIODIC, dev_record,
                            &h->ccl_local_n);
  if (e != cudaSuccess) return fail(SPGG_E_CUDA, "spgg_strip_clusters: %s", cudaGetErrorString(e));
  h->launches += 9;   // seven kernels of ours, CUB's sort and unique counted as one each
  h->ccl_local = true;
  h->ccl_which = which;
  h->ccl_flags = flags;
  return SPGG_OK;
}

extern "C" int spgg_strip_clusters_resolve(spgg_t *h, int world, int rank, const void *dev_records, int64_t *n_owned,
                                           int64_t *first_label, int64_t *n_total) {
  if (!h || !dev_records || !n_owned || !first_label || !n_total)
    return fail(SPGG_E_INVALID, "spgg_strip_clusters_resolve: null argument");
  if (world < 1 || rank < 0 || rank >= world) return fail(SPGG_E_INVALID, "rank %d outside a world of %d", rank, world);
  if (!h->ccl_local) return fail(SPGG_E_STATE, "spgg_strip_clusters_resolve: no spgg_strip_clusters pass of the current state");
  const Geom &g = h->g;
  const long long rb = ccl_record_bytes(g.L);
  std::vector<int> hd((size_t)world * CCL_REC_HDR);
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaMemcpy2D(hd.data(), CCL_REC_HDR * sizeof(int), dev_records, (size_t)rb, CCL_REC_HDR * sizeof(int), world,
                        cudaMemcpyDeviceToHost));
  int next = 0;
  for (int k = 0; k < world; ++k) {
    const int *r = hd.data() + (size_t)k * CCL_REC_HDR;
    if (r[CCL_H_MAGIC] != CCL_REC_MAGIC) return fail(SPGG_E_INVALID, "record %d is not a strip cluster record", k);
    if (r[CCL_H_L] != g.L) return fail(SPGG_E_INVALID, "record %d: L = %d, this handle's L = %d", k, r[CCL_H_L], g.L);
    if (r[CCL_H_WHICH] != h->ccl_which || r[CCL_H_FLAGS] != h->ccl_flags)
      return fail(SPGG_E_INVALID, "record %d: which %d / flags 0x%x, this strip labelled which %d / flags 0x%x", k,
                  r[CCL_H_WHICH], r[CCL_H_FLAGS], h->ccl_which, h->ccl_flags);
    if (r[CCL_H_ROW0] != next || r[CCL_H_ROWS] < 1 || r[CCL_H_ROWS] > g.L - next)
      return fail(SPGG_E_INVALID, "record %d: rows [%d, %d) do not continue the strips above at row %d", k, r[CCL_H_ROW0],
                  r[CCL_H_ROW0] + r[CCL_H_ROWS], next);
    if (r[CCL_H_NPARTS] < 0 || r[CCL_H_NPARTS] > 2 * g.L || r[CCL_H_NLOCAL] < r[CCL_H_NPARTS])
      return fail(SPGG_E_INVALID, "record %d: %d boundary roots of %d roots", k, r[CCL_H_NPARTS], r[CCL_H_NLOCAL]);
    next += r[CCL_H_ROWS];
  }
  if (next != g.L) return fail(SPGG_E_INVALID, "the %d records cover rows [0, %d) of %d", world, next, g.L);
  const int *mine = hd.data() + (size_t)rank * CCL_REC_HDR;
  if (mine[CCL_H_ROW0] != g.row0 || mine[CCL_H_ROWS] != g.rows || mine[CCL_H_NLOCAL] != h->ccl_local_n)
    return fail(SPGG_E_INVALID, "record %d is not this strip's (rows [%d, %d))", rank, g.row0, g.row0 + g.rows);
  cudaError_t e = ccl_strip_alloc(&h->ccl_strip, g.L, world);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    return fail(SPGG_E_CUDA, "spgg_strip_clusters_resolve: scratch for %d records: %s", world, cudaGetErrorString(e));
  }
  h->ccl_local = false;   // the resolution rewrites the strip-local result
  e = launch_strip_resolve(h->ccl, h->ccl_strip, dev_records, world, rank, h->ccl_flags & SPGG_CLUSTER_PERIODIC, n_owned,
                           first_label, n_total);
  if (e != cudaSuccess) return fail(SPGG_E_CUDA, "spgg_strip_clusters_resolve: %s", cudaGetErrorString(e));
  h->launches += 10;
  h->ccl_n = *n_owned;
  h->ccl_valid = true;
  return SPGG_OK;
}

// ---------------------------------------------------------------- pair counts
// n_CC and n_diff of one replica's strategies at every offset 0..max_d along both axes (include/spgg.h); the
// kernels live in spgg_pairs.cu.  Nothing here touches the state or a cluster-labelling result.
static int pair_max_d(spgg_t *h, int max_d, const char *fn) {
  if (max_d < 1 || max_d > h->g.L / 2) return fail(SPGG_E_INVALID, "%s: max_d = %d outside [1, L/2 = %d]", fn, max_d, h->g.L / 2);
  return SPGG_OK;
}

// device counts for max_d, and room for tail_words words of tail rows
static int pair_scratch(spgg_handle *h, int max_d, size_t tail_words) {
  const size_t n = 4 * (size_t)(max_d + 1);
  if (h->pair_cnt_n < n) {
    cudaFree(h->d_pair_cnt);
    h->d_pair_cnt = nullptr;
    h->pair_cnt_n = 0;
    CUDA_TRY(cudaMalloc((void **)&h->d_pair_cnt, n * sizeof(unsigned long long)));
    h->pair_cnt_n = n;
  }
  if (h->pair_tail_n < tail_words) {
    cudaFree(h->d_pair_tail);
    h->d_pair_tail = nullptr;
    h->pair_tail_n = 0;
    CUDA_TRY(cudaMalloc((void **)&h->d_pair_tail, tail_words * sizeof(uint32_t)));
    h->pair_tail_n = tail_words;
  }
  return SPGG_OK;
}

static const uint32_t *pair_plane(const spgg_handle *h, int rep) {
  const Geom &g = h->g;
  return h->d_S[h->cur] + (size_t)rep * g.bits_stride + (size_t)GH * g.pitchW + WPAD;
}

extern "C" int spgg_pair_counts(spgg_t *h, int rep, int max_d, int64_t *out) {
  if (!h || !out) return fail(SPGG_E_INVALID, "spgg_pair_counts: null argument");
  if (rep < 0 || rep >= h->n_rep) return fail(SPGG_E_INVALID, "replica %d out of range", rep);
  if (!h->g.wrap_rows)
    return fail(SPGG_E_UNSUPPORTED, "spgg_pair_counts needs the whole lattice (rows == L), not a strip: see spgg_strip_pair_counts");
  int rcode = pair_max_d(h, max_d, "spgg_pair_counts");
  if (rcode) return rcode;
  rcode = finish_pending(h);
  if (rcode) return rcode;
  CUDA_TRY(cudaSetDevice(h->device));
  rcode = pair_scratch(h, max_d, 0);
  if (rcode) return rcode;
  const Geom &g = h->g;
  const uint32_t *S = pair_plane(h, rep);
  cudaError_t e = launch_pair_counts(S, g.pitchW, g.rows, g.L, S, g.pitchW, max_d, h->d_pair_cnt, out);
  if (e != cudaSuccess) return fail(SPGG_E_CUDA, "spgg_pair_counts: %s", cudaGetErrorString(e));
  h->launches += 2;
  return SPGG_OK;
}

// Row strips (include/spgg.h): a record of the strip's first min(max_d, rows) rows, padded to max_rows rows;
// from the records of all ranks each strip assembles the max_d rows below it and counts its own sites' pairs
static int strip_pairs_supported(spgg_t *h, int max_d, int max_rows, const char *fn) {
  if (h->n_rep != 1) return fail(SPGG_E_UNSUPPORTED, "%s: strip pair counts serve single-replica handles", fn);
  int rcode = pair_max_d(h, max_d, fn);
  if (rcode) return rcode;
  if (max_rows < std::min(max_d, h->g.rows) || max_rows > max_d)
    return fail(SPGG_E_INVALID, "%s: max_rows = %d outside [min(max_d, rows) = %d, max_d = %d]", fn, max_rows,
                std::min(max_d, h->g.rows), max_d);
  return SPGG_OK;
}

extern "C" int64_t spgg_strip_pair_record_bytes(spgg_t *h, int max_d, int max_rows) {
  if (!h) return fail(SPGG_E_INVALID, "null handle");
  int rcode = strip_pairs_supported(h, max_d, max_rows, "spgg_strip_pair_record_bytes");
  return rcode ? rcode : pair_record_bytes(h->g.L, max_rows);
}

extern "C" int spgg_strip_pair_record(spgg_t *h, int max_d, int max_rows, void *dev_record) {
  if (!h || !dev_record) return fail(SPGG_E_INVALID, "spgg_strip_pair_record: null argument");
  int rcode = strip_pairs_supported(h, max_d, max_rows, "spgg_strip_pair_record");
  if (rcode) return rcode;
  rcode = finish_pending(h);
  if (rcode) return rcode;
  CUDA_TRY(cudaSetDevice(h->device));
  const Geom &g = h->g;
  cudaError_t e = launch_pair_record(pair_plane(h, 0), g.pitchW, g.row0, g.rows, g.L, max_d, max_rows, dev_record);
  if (e == cudaSuccess) e = cudaStreamSynchronize(0);
  if (e != cudaSuccess) return fail(SPGG_E_CUDA, "spgg_strip_pair_record: %s", cudaGetErrorString(e));
  h->launches += 1;
  return SPGG_OK;
}

extern "C" int spgg_strip_pair_counts(spgg_t *h, int world, int rank, const void *dev_records, int max_d, int max_rows,
                                      int64_t *out) {
  if (!h || !dev_records || !out) return fail(SPGG_E_INVALID, "spgg_strip_pair_counts: null argument");
  if (world < 1 || rank < 0 || rank >= world) return fail(SPGG_E_INVALID, "rank %d outside a world of %d", rank, world);
  int rcode = strip_pairs_supported(h, max_d, max_rows, "spgg_strip_pair_counts");
  if (rcode) return rcode;
  const Geom &g = h->g;
  const long long rb = pair_record_bytes(g.L, max_rows);
  std::vector<int> hd((size_t)world * PAIR_REC_HDR);
  CUDA_TRY(cudaSetDevice(h->device));
  for (int k = 0; k < world; ++k)
    CUDA_TRY(cudaMemcpy(hd.data() + (size_t)k * PAIR_REC_HDR, (const char *)dev_records + k * rb, PAIR_REC_HDR * sizeof(int),
                        cudaMemcpyDeviceToHost));
  int next = 0;
  for (int k = 0; k < world; ++k) {
    const int *r = hd.data() + (size_t)k * PAIR_REC_HDR;
    if (r[PAIR_H_MAGIC] != PAIR_REC_MAGIC) return fail(SPGG_E_INVALID, "record %d is not a strip pair record", k);
    if (r[PAIR_H_L] != g.L) return fail(SPGG_E_INVALID, "record %d: L = %d, this handle's L = %d", k, r[PAIR_H_L], g.L);
    if (r[PAIR_H_MAXD] != max_d || r[PAIR_H_MAXROWS] != max_rows)
      return fail(SPGG_E_INVALID, "record %d: max_d %d / max_rows %d, this call's max_d %d / max_rows %d", k, r[PAIR_H_MAXD],
                  r[PAIR_H_MAXROWS], max_d, max_rows);
    if (r[PAIR_H_ROW0] != next || r[PAIR_H_ROWS] < 1 || r[PAIR_H_ROWS] > g.L - next)
      return fail(SPGG_E_INVALID, "record %d: rows [%d, %d) do not continue the strips above at row %d", k, r[PAIR_H_ROW0],
                  r[PAIR_H_ROW0] + r[PAIR_H_ROWS], next);
    if (r[PAIR_H_NROWS] != std::min(max_d, r[PAIR_H_ROWS]) || r[PAIR_H_NROWS] > max_rows)   // the tail copy reads NROWS rows
      return fail(SPGG_E_INVALID, "record %d holds %d rows, not min(max_d, rows) = %d within max_rows = %d", k,
                  r[PAIR_H_NROWS], std::min(max_d, r[PAIR_H_ROWS]), max_rows);
    next += r[PAIR_H_ROWS];
  }
  if (next != g.L) return fail(SPGG_E_INVALID, "the %d records cover rows [0, %d) of %d", world, next, g.L);
  const int *mine = hd.data() + (size_t)rank * PAIR_REC_HDR;
  if (mine[PAIR_H_ROW0] != g.row0 || mine[PAIR_H_ROWS] != g.rows)
    return fail(SPGG_E_INVALID, "record %d is not this strip's (rows [%d, %d))", rank, g.row0, g.row0 + g.rows);
  rcode = finish_pending(h);
  if (rcode) return rcode;
  const int nW = (g.L + 31) / 32;
  rcode = pair_scratch(h, max_d, (size_t)max_d * nW);
  if (rcode) return rcode;
  // the max_d rows below this strip: the first rows of the strips that follow it, in order, around the torus
  // (every record holds min(max_d, rows) rows, so the walk ends within one turn)
  for (int t = 0, k = (rank + 1) % world; t < max_d; k = (k + 1) % world) {
    const int n = std::min(hd[(size_t)k * PAIR_REC_HDR + PAIR_H_NROWS], max_d - t);
    CUDA_TRY(cudaMemcpy(h->d_pair_tail + (size_t)t * nW, (const char *)dev_records + k * rb + PAIR_REC_HDR * sizeof(int),
                        (size_t)n * nW * sizeof(uint32_t), cudaMemcpyDeviceToDevice));
    t += n;
  }
  cudaError_t e = launch_pair_counts(pair_plane(h, 0), g.pitchW, g.rows, g.L, h->d_pair_tail, nW, max_d, h->d_pair_cnt, out);
  if (e != cudaSuccess) return fail(SPGG_E_CUDA, "spgg_strip_pair_counts: %s", cudaGetErrorString(e));
  h->launches += 2;
  return SPGG_OK;
}

// ---------------------------------------------------------------- block fields
// Counts and fp64 sums of R and Q over b x b blocks of one replica (include/spgg.h); the kernels live in
// spgg_blocks.cu.  Reads the planes spgg_state_digest reads; touches neither the state nor any other result.
extern "C" int spgg_block_fields(spgg_t *h, int rep, int b, int flags, int64_t *counts, double *sums) {
  if (!h || !counts || (flags && !sums)) return fail(SPGG_E_INVALID, "spgg_block_fields: null argument");
  if (rep < 0 || rep >= h->n_rep) return fail(SPGG_E_INVALID, "replica %d out of range", rep);
  if (flags & ~(SPGG_BLOCK_R | SPGG_BLOCK_Q)) return fail(SPGG_E_INVALID, "spgg_block_fields: unknown flags 0x%x", flags);
  const Geom &g = h->g;
  if (b < 1 || b > g.L) return fail(SPGG_E_INVALID, "spgg_block_fields: b = %d outside [1, L = %d]", b, g.L);
  const long long B = (g.L + b - 1) / b;
  if (B * B > BLK_MAX_BLOCKS)
    return fail(SPGG_E_INVALID, "spgg_block_fields: %lld x %lld blocks exceed 2^24 (b = %d, L = %d)", B, B, b, g.L);
  int rcode = finish_pending(h);
  if (rcode) return rcode;
  CUDA_TRY(cudaSetDevice(h->device));
  const bool want_r = flags & SPGG_BLOCK_R, want_q = flags & SPGG_BLOCK_Q;
  const BlockGeom q = block_geom(g.L, g.row0, g.rows, b);
  const size_t need = block_scratch_bytes(q, (want_r ? 1 : 0) + (want_q ? h->nq() : 0));
  if (h->blk_bytes < need) {
    cudaFree(h->d_blk);
    h->d_blk = nullptr;
    h->blk_bytes = 0;
    CUDA_TRY(cudaMalloc(&h->d_blk, need));
    h->blk_bytes = need;
  }
  const uint32_t *S = h->d_S[h->cur] + (size_t)rep * g.bits_stride + (size_t)GH * g.pitchW + WPAD;
  const void *R = (const char *)h->d_R[h->cur] + ((size_t)rep * g.plane_stride + (size_t)GH * g.pitchB + CPAD) * h->elem_R();
  const void *Q = (const char *)h->Qcur() + (size_t)rep * g.site_stride * h->nq() * h->elem_Q();
  const double rq = h->rc_host[rep].rq;
  const cudaError_t e = with_mode(h->mode, [&](auto md) {
    return launch_block_fields<decltype(md)>(q, g.pitchW, g.pitchB, S, R, Q, rq, h->nq(), want_r, want_q, h->d_blk,
                                             counts, sums);
  });
  if (e != cudaSuccess) return fail(SPGG_E_CUDA, "spgg_block_fields: %s", cudaGetErrorString(e));
  h->launches += flags ? 2 + (q.nrc * q.ncs > 1) : 1;
  return SPGG_OK;
}

// ---------------------------------------------------------------- value distributions
// Extremes, np.histogram counts and greedy-policy counts of replicas rep0 .. rep0 + n_rep - 1 (include/spgg.h); the
// kernels live in spgg_hist.cu.  Reads the planes spgg_block_fields reads; touches neither the state nor any other
// result.
static int hist_args(spgg_t *h, const char *fn, int rep0, int n_rep, int flags) {
  if (rep0 < 0 || n_rep < 1 || rep0 > h->n_rep - n_rep)
    return fail(SPGG_E_INVALID, "%s: replicas [%d, %d + %d) outside [0, %d)", fn, rep0, rep0, n_rep, h->n_rep);
  if (flags & ~(SPGG_HIST_R | SPGG_HIST_Q)) return fail(SPGG_E_INVALID, "%s: unknown flags 0x%x", fn, flags);
  return SPGG_OK;
}

// the planes of replica rep0 and the int8 quanta of the replicas; grows the scratch to `need` bytes
static int hist_prepare(spgg_t *h, int rep0, int n_rep, size_t need, HistPlanes *p, std::vector<double> *rq) {
  int rcode = finish_pending(h);
  if (rcode) return rcode;
  CUDA_TRY(cudaSetDevice(h->device));
  if (h->hist_bytes < need) {
    cudaFree(h->d_hist);
    h->d_hist = nullptr;
    h->hist_bytes = 0;
    CUDA_TRY(cudaMalloc(&h->d_hist, need));
    h->hist_bytes = need;
  }
  const Geom &g = h->g;
  p->L = g.L; p->rows = g.rows; p->pitchW = g.pitchW; p->pitchB = g.pitchB; p->nq = h->nq(); p->n_rep = n_rep;
  p->S = h->d_S[h->cur] + (size_t)rep0 * g.bits_stride + (size_t)GH * g.pitchW + WPAD;
  p->R = (const char *)h->d_R[h->cur] + ((size_t)rep0 * g.plane_stride + (size_t)GH * g.pitchB + CPAD) * h->elem_R();
  p->Q = (const char *)h->Qcur() + (size_t)rep0 * g.site_stride * h->nq() * h->elem_Q();
  p->bits_stride = g.bits_stride; p->plane_stride = g.plane_stride; p->q_stride = g.site_stride * h->nq();
  rq->resize(n_rep);
  for (int r = 0; r < n_rep; ++r) (*rq)[r] = h->rc_host[rep0 + r].rq;
  return SPGG_OK;
}

extern "C" int spgg_value_ranges(spgg_t *h, int rep0, int n_rep, int flags, double *minmax) {
  if (!h || !minmax) return fail(SPGG_E_INVALID, "spgg_value_ranges: null argument");
  int rcode = hist_args(h, "spgg_value_ranges", rep0, n_rep, flags);
  if (rcode) return rcode;
  const bool want_r = flags & SPGG_HIST_R, want_q = flags & SPGG_HIST_Q;
  const int m = (want_r ? 1 : 0) + (want_q ? h->nq() : 0);
  HistPlanes p;
  std::vector<double> rq;
  rcode = hist_prepare(h, rep0, n_rep, hist_scratch_bytes(n_rep, m, 1), &p, &rq);
  if (rcode) return rcode;
  const cudaError_t e = with_mode(h->mode, [&](auto md) {
    return launch_value_ranges<decltype(md)>(p, want_r, want_q, rq.data(), h->d_hist, minmax);
  });
  if (e != cudaSuccess) return fail(SPGG_E_CUDA, "spgg_value_ranges: %s", cudaGetErrorString(e));
  h->launches += m > 0;
  return SPGG_OK;
}

extern "C" int spgg_histograms(spgg_t *h, int rep0, int n_rep, int flags, int n_bins, const double *edges,
                               int64_t *counts, int64_t *policy) {
  if (!h) return fail(SPGG_E_INVALID, "spgg_histograms: null argument");
  int rcode = hist_args(h, "spgg_histograms", rep0, n_rep, flags);
  if (rcode) return rcode;
  if (n_bins < 1 || n_bins > HIST_MAX_BINS)
    return fail(SPGG_E_INVALID, "spgg_histograms: n_bins = %d outside [1, %d]", n_bins, HIST_MAX_BINS);
  const bool want_r = flags & SPGG_HIST_R, want_q = flags & SPGG_HIST_Q;
  const int m = (want_r ? 1 : 0) + (want_q ? h->nq() : 0);
  if (m > 0 && (!edges || !counts)) return fail(SPGG_E_INVALID, "spgg_histograms: null argument");
  for (long long row = 0; row < (long long)n_rep * m; ++row) {
    const double *e = edges + row * (n_bins + 1);
    bool ok = std::isfinite(e[0]) && e[0] < e[n_bins];
    for (int i = 1; ok && i <= n_bins; ++i) ok = std::isfinite(e[i]) && e[i] >= e[i - 1];
    if (!ok)
      return fail(SPGG_E_INVALID, "spgg_histograms: edge row %lld is not finite and increasing from edges[0] to "
                  "edges[n_bins]", row);
  }
  HistPlanes p;
  std::vector<double> rq;
  rcode = hist_prepare(h, rep0, n_rep, hist_scratch_bytes(n_rep, m, n_bins), &p, &rq);
  if (rcode) return rcode;
  const cudaError_t e = with_mode(h->mode, [&](auto md) {
    return launch_histograms<decltype(md)>(p, want_r, want_q, n_bins, edges, rq.data(), h->d_hist, counts, policy);
  });
  if (e != cudaSuccess) return fail(SPGG_E_CUDA, "spgg_histograms: %s", cudaGetErrorString(e));
  h->launches += (m > 0 || policy) + (want_r && h->mode == MODE_F32_I8);
  return SPGG_OK;
}

// ---------------------------------------------------------------- state overlaps
// Snapshots of replica states kept on the handle, and what changed since (include/spgg.h); the kernels live in
// spgg_overlap.cu.  Reads the planes spgg_histograms reads; touches neither the state nor any other result.
static int snap_args(spgg_t *h, const char *fn, int slot, int rep0, int n_rep, int flags) {
  if (slot < 0 || slot >= SPGG_MAX_SNAPSHOTS)
    return fail(SPGG_E_INVALID, "%s: slot %d outside [0, %d)", fn, slot, SPGG_MAX_SNAPSHOTS);
  if (rep0 < 0 || n_rep < 1 || rep0 > h->n_rep - n_rep)
    return fail(SPGG_E_INVALID, "%s: replicas [%d, %d + %d) outside [0, %d)", fn, rep0, rep0, n_rep, h->n_rep);
  if (flags & ~(SPGG_SNAP_R | SPGG_SNAP_Q)) return fail(SPGG_E_INVALID, "%s: unknown flags 0x%x", fn, flags);
  return SPGG_OK;
}

// Byte offsets of a slot's planes for n_rep replicas: the bit plane at 0, R at off[1] (SPGG_SNAP_R), Q at off[2]
// (SPGG_SNAP_Q), each a whole replica range of the live buffer; returns the slot's size
static size_t snap_layout(const spgg_handle *h, int n_rep, int flags, size_t off[3]) {
  auto up = [](size_t x) { return (x + 255) / 256 * 256; };
  const Geom &g = h->g;
  off[0] = 0;
  off[1] = up((size_t)n_rep * g.bits_stride * 4);
  off[2] = off[1] + ((flags & SPGG_SNAP_R) ? up((size_t)n_rep * g.plane_stride * h->elem_R()) : 0);
  return off[2] + ((flags & SPGG_SNAP_Q) ? up((size_t)n_rep * g.site_stride * h->nq() * h->elem_Q()) : 0);
}

extern "C" int spgg_snapshot(spgg_t *h, int slot, int rep0, int n_rep, int flags) {
  if (!h) return fail(SPGG_E_INVALID, "spgg_snapshot: null argument");
  int rcode = snap_args(h, "spgg_snapshot", slot, rep0, n_rep, flags);
  if (rcode) return rcode;
  rcode = finish_pending(h);
  if (rcode) return rcode;
  CUDA_TRY(cudaSetDevice(h->device));
  spgg_handle::Snapshot &s = h->snaps[slot];
  size_t off[3];
  const size_t need = snap_layout(h, n_rep, flags, off);
  s.full = false;
  if (s.bytes != need) {
    cudaFree(s.mem);
    s.mem = nullptr;
    s.bytes = 0;
    const cudaError_t e = cudaMalloc(&s.mem, need);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      s.mem = nullptr;
      return fail(SPGG_E_CUDA, "spgg_snapshot: %zu bytes for slot %d: %s", need, slot, cudaGetErrorString(e));
    }
    s.bytes = need;
  }
  const Geom &g = h->g;
  char *mem = (char *)s.mem;
  CUDA_TRY(cudaMemcpyAsync(mem, h->d_S[h->cur] + (size_t)rep0 * g.bits_stride, (size_t)n_rep * g.bits_stride * 4,
                           cudaMemcpyDeviceToDevice, 0));
  if (flags & SPGG_SNAP_R) {
    const size_t pb = (size_t)g.plane_stride * h->elem_R();
    CUDA_TRY(cudaMemcpyAsync(mem + off[1], (const char *)h->d_R[h->cur] + (size_t)rep0 * pb, (size_t)n_rep * pb,
                             cudaMemcpyDeviceToDevice, 0));
  }
  if (flags & SPGG_SNAP_Q) {
    const size_t qb = (size_t)g.site_stride * h->nq() * h->elem_Q();
    CUDA_TRY(cudaMemcpyAsync(mem + off[2], (const char *)h->Qcur() + (size_t)rep0 * qb, (size_t)n_rep * qb,
                             cudaMemcpyDeviceToDevice, 0));
  }
  // a step on another (non-blocking) stream must not overwrite the planes while they are being copied
  CUDA_TRY(cudaStreamSynchronize(0));
  s.iter = h->iter;
  s.rep0 = rep0;
  s.n_rep = n_rep;
  s.flags = flags;
  s.rq.resize(n_rep);
  for (int r = 0; r < n_rep; ++r) s.rq[r] = h->rc_host[rep0 + r].rq;
  s.full = true;
  return SPGG_OK;
}

extern "C" int spgg_snapshot_info(spgg_t *h, int slot, int64_t *iteration, int *rep0, int *n_rep, int *flags) {
  if (!h) return fail(SPGG_E_INVALID, "spgg_snapshot_info: null argument");
  if (slot < 0 || slot >= SPGG_MAX_SNAPSHOTS)
    return fail(SPGG_E_INVALID, "spgg_snapshot_info: slot %d outside [0, %d)", slot, SPGG_MAX_SNAPSHOTS);
  const spgg_handle::Snapshot &s = h->snaps[slot];
  if (!s.full) return fail(SPGG_E_STATE, "spgg_snapshot_info: slot %d holds no snapshot", slot);
  if (iteration) *iteration = s.iter;
  if (rep0) *rep0 = s.rep0;
  if (n_rep) *n_rep = s.n_rep;
  if (flags) *flags = s.flags;
  return SPGG_OK;
}

extern "C" int spgg_snapshot_free(spgg_t *h, int slot) {
  if (!h) return fail(SPGG_E_INVALID, "spgg_snapshot_free: null argument");
  if (slot < 0 || slot >= SPGG_MAX_SNAPSHOTS)
    return fail(SPGG_E_INVALID, "spgg_snapshot_free: slot %d outside [0, %d)", slot, SPGG_MAX_SNAPSHOTS);
  spgg_handle::Snapshot &s = h->snaps[slot];
  if (!s.mem) return SPGG_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaFree(s.mem);
  s = spgg_handle::Snapshot();
  return SPGG_OK;
}

extern "C" int spgg_overlap(spgg_t *h, int slot, int rep0, int n_rep, int flags, int64_t *counts, int64_t *changed,
                            double *diffs) {
  if (!h || !counts) return fail(SPGG_E_INVALID, "spgg_overlap: null argument");
  int rcode = snap_args(h, "spgg_overlap", slot, rep0, n_rep, flags);
  if (rcode) return rcode;
  const bool want_r = flags & SPGG_SNAP_R, want_q = flags & SPGG_SNAP_Q;
  const int m = (want_r ? 1 : 0) + (want_q ? h->nq() : 0);
  if (m > 0 && (!changed || !diffs)) return fail(SPGG_E_INVALID, "spgg_overlap: null argument");
  const spgg_handle::Snapshot &s = h->snaps[slot];
  if (!s.full) return fail(SPGG_E_STATE, "spgg_overlap: slot %d holds no snapshot", slot);
  if (n_rep != s.n_rep)
    return fail(SPGG_E_INVALID, "spgg_overlap: n_rep = %d, slot %d holds %d replicas", n_rep, slot, s.n_rep);
  if (flags & ~s.flags)
    return fail(SPGG_E_INVALID, "spgg_overlap: flags 0x%x, slot %d holds 0x%x", flags, slot, s.flags);
  rcode = finish_pending(h);
  if (rcode) return rcode;
  CUDA_TRY(cudaSetDevice(h->device));
  const Geom &g = h->g;
  const size_t need = overlap_scratch_bytes(g.L, g.rows, n_rep, m);
  if (h->ov_bytes < need) {
    cudaFree(h->d_ov);
    h->d_ov = nullptr;
    h->ov_bytes = 0;
    CUDA_TRY(cudaMalloc(&h->d_ov, need));
    h->ov_bytes = need;
  }
  size_t off[3];
  snap_layout(h, n_rep, s.flags, off);
  const char *mem = (const char *)s.mem;
  const size_t r0 = ((size_t)GH * g.pitchB + CPAD) * h->elem_R();
  OvPlanes p;
  p.L = g.L; p.rows = g.rows; p.pitchW = g.pitchW; p.pitchB = g.pitchB; p.nq = h->nq(); p.n_rep = n_rep;
  p.S[0] = h->d_S[h->cur] + (size_t)rep0 * g.bits_stride + (size_t)GH * g.pitchW + WPAD;
  p.S[1] = (const uint32_t *)mem + (size_t)GH * g.pitchW + WPAD;
  p.R[0] = (const char *)h->d_R[h->cur] + (size_t)rep0 * g.plane_stride * h->elem_R() + r0;
  p.R[1] = mem + off[1] + r0;
  p.Q[0] = (const char *)h->Qcur() + (size_t)rep0 * g.site_stride * h->nq() * h->elem_Q();
  p.Q[1] = mem + off[2];
  p.bits_stride = g.bits_stride; p.plane_stride = g.plane_stride; p.q_stride = g.site_stride * h->nq();
  std::vector<double> rq(2 * (size_t)n_rep);
  for (int r = 0; r < n_rep; ++r) {
    rq[r] = h->rc_host[rep0 + r].rq;
    rq[n_rep + r] = s.rq[r];
  }
  const cudaError_t e = with_mode(h->mode, [&](auto md) {
    return launch_overlap<decltype(md)>(p, want_r, want_q, rq.data(), h->d_ov, counts, changed, diffs);
  });
  if (e != cudaSuccess) return fail(SPGG_E_CUDA, "spgg_overlap: %s", cudaGetErrorString(e));
  h->launches += 1 + (m > 0);
  return SPGG_OK;
}

// ---------------------------------------------------------------- strips
// Peer-mapped planes: each strip exports the IPC handles of its six planes (code, R, S x two parities);
// the neighbours open them and their boundary tiles store straight into this strip's ghost rows.
extern "C" int spgg_ipc_export(spgg_t *h, unsigned char *handles /* 6 x 64 bytes */) {
  if (!h || !handles) return fail(SPGG_E_INVALID, "spgg_ipc_export: null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  CUDA_TRY(cudaSetDevice(h->device));
  void *ptrs[6] = {h->d_code[0], h->d_code[1], h->d_R[0], h->d_R[1], h->d_S[0], h->d_S[1]};
  for (int i = 0; i < 6; ++i) {
    cudaIpcMemHandle_t hd;
    CUDA_TRY(cudaIpcGetMemHandle(&hd, ptrs[i]));
    memcpy(handles + 64 * i, &hd, 64);
  }
  return SPGG_OK;
}

// which: 0 = the strip above (row0 - 1), 1 = the strip below.  same_as_other != 0: that neighbour is the
// one already attached on the other side (two strips), reuse its mappings instead of opening them twice.
extern "C" int spgg_ipc_attach(spgg_t *h, int which, const unsigned char *handles, int peer_rows, int same_as_other) {
  if (!h || (which != 0 && which != 1)) return fail(SPGG_E_INVALID, "spgg_ipc_attach: bad argument");
  if (!h->fast || h->n_rep != 1 || h->g.wrap_rows) return fail(SPGG_E_UNSUPPORTED, "peer-mapped halos serve single-replica strips on the TMA fast path");
  int rcode = finish_pending(h);
  if (rcode) return rcode;
  CUDA_TRY(cudaSetDevice(h->device));
  void *ptrs[6];
  if (same_as_other) {
    const int o = which ^ 1;
    ptrs[0] = h->peer_code[o][0]; ptrs[1] = h->peer_code[o][1]; ptrs[2] = h->peer_R[o][0];
    ptrs[3] = h->peer_R[o][1]; ptrs[4] = h->peer_S[o][0]; ptrs[5] = h->peer_S[o][1];
    if (!ptrs[0]) return fail(SPGG_E_STATE, "the other neighbour is not attached yet");
  } else {
    if (!handles) return fail(SPGG_E_INVALID, "spgg_ipc_attach: null handles");
    for (int i = 0; i < 6; ++i) {
      cudaIpcMemHandle_t hd;
      memcpy(&hd, handles + 64 * i, 64);
      cudaError_t e = cudaIpcOpenMemHandle(&ptrs[i], hd, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return fail(SPGG_E_CUDA, "cudaIpcOpenMemHandle failed: %s", cudaGetErrorString(e));
      }
      h->ipc_opened.push_back(ptrs[i]);
    }
  }
  h->peer_code[which][0] = ptrs[0]; h->peer_code[which][1] = ptrs[1];
  h->peer_R[which][0] = ptrs[2]; h->peer_R[which][1] = ptrs[3];
  h->peer_S[which][0] = (uint32_t *)ptrs[4]; h->peer_S[which][1] = (uint32_t *)ptrs[5];
  h->peer_rows[which] = peer_rows;
  h->peer_on = h->peer_code[0][0] != nullptr && h->peer_code[1][0] != nullptr;
  return SPGG_OK;
}

// The ring of report slots: spgg_ring_export() gives the cudaIpc handle of this strip's ring (64 bytes);
// spgg_ring_attach() receives the handles of ALL ranks in rank order (its own entry is not opened).
extern "C" int spgg_ring_export(spgg_t *h, unsigned char *handle64) {
  if (!h || !handle64) return fail(SPGG_E_INVALID, "spgg_ring_export: null argument");
  CUDA_TRY(cudaSetDevice(h->device));
  if (!h->d_ring) {
    CUDA_TRY(cudaMalloc((void **)&h->d_ring, 2 << 20));   // its own allocation: IPC handles name whole allocations
    CUDA_TRY(cudaMemset(h->d_ring, 0, 2 << 20));
  }
  cudaIpcMemHandle_t hd;
  CUDA_TRY(cudaIpcGetMemHandle(&hd, h->d_ring));
  memcpy(handle64, &hd, 64);
  return SPGG_OK;
}

extern "C" int spgg_ring_attach(spgg_t *h, int world, int rank, const unsigned char *handles /* world x 64 */) {
  if (!h || !handles || world < 2 || world > SPGG_MAX_RING || rank < 0 || rank >= world)
    return fail(SPGG_E_INVALID, "spgg_ring_attach: bad argument (world %d, at most %d)", world, SPGG_MAX_RING);
  if (!h->d_ring || !h->peer_on) return fail(SPGG_E_STATE, "spgg_ring_attach follows spgg_ring_export and the neighbours' spgg_ipc_attach");
  CUDA_TRY(cudaSetDevice(h->device));
  for (int p = 0; p < world; ++p) {
    if (p == rank) { h->ring_peer[p] = h->d_ring; continue; }
    cudaIpcMemHandle_t hd;
    memcpy(&hd, handles + 64 * p, 64);
    void *ptr = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&ptr, hd, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      h->ring_world = 0;
      return fail(SPGG_E_CUDA, "cudaIpcOpenMemHandle (ring of rank %d) failed: %s", p, cudaGetErrorString(e));
    }
    h->ipc_opened.push_back(ptr);
    h->ring_peer[p] = (unsigned *)ptr;
  }
  h->ring_world = world;
  h->gen = 0;
  return SPGG_OK;
}

extern "C" int spgg_strip_can_speculate(spgg_t *h, int do_select) {
  return (h && h->pending && h->d_gvec && h->n_rep == 1 && can_speculate(h, do_select)) ? 1 : 0;
}

extern "C" int spgg_strip_iteration(spgg_t *h, int do_select, void *stream_) {
  if (!h || !h->pending) return fail(SPGG_E_STATE, "spgg_strip_iteration outside begin/end");
  if (!spgg_strip_can_speculate(h, do_select)) return fail(SPGG_E_STATE, "this strip cannot guess the maximum now: run the exact pair");
  h->pend_rel += 1;
  return launch_step(h, 1, do_select, (cudaStream_t)stream_, true);
}

extern "C" void *spgg_strip_report_ptr(spgg_t *h) {
  if (!h || !h->pending || !h->d_gvec || h->last_rel < 0) return nullptr;
  return h->d_gvec + 4 * (size_t)h->last_rel;
}

extern "C" int spgg_strip_verify(spgg_t *h, void *stream_) {
  if (!h || !h->pending || !h->d_gvec || h->last_rel < 0) return fail(SPGG_E_STATE, "spgg_strip_verify: no strip launch to verify");
  if (h->last_gen >= 0)   // ring mode: the ranks combined their reports themselves; wait for all of them, then the verdict
    k_ring_verify<<<1, 32, 0, (cudaStream_t)stream_>>>(h->d_ring, h->last_gen, h->ring_world, h->d_gvec, h->last_rel,
                                                      (int)(h->pend_t0 + h->last_rel), h->last_upd, h->last_spec, h->last_sel,
                                                      h->d_gcarry, reinterpret_cast<float *>(h->d_gmax), h->d_bad, h->d_stop);
  else
    k_strip_verify<<<1, 32, 0, (cudaStream_t)stream_>>>(h->d_gvec, h->last_rel, (int)(h->pend_t0 + h->last_rel), h->last_upd,
                                                         h->last_spec, h->last_sel, h->d_gcarry,
                                                         reinterpret_cast<float *>(h->d_gmax), h->d_bad, h->d_stop);
  CUDA_TRY(cudaGetLastError());
  h->launches += 1;
  if (h->last_upd) h->carry_valid = true;   // written by the kernel above, from the reduced report
  return SPGG_OK;
}

// after the streams of the chunk have been synchronised: 0, or the relative index (>= 1) of the launch
// whose guess was wrong - the same on every rank, since every rank saw the same reduced values
extern "C" int spgg_strip_failed(spgg_t *h) {
  if (!h || !h->d_bad) return 0;
  int bad = 0x7fffffff;
  if (cudaMemcpy(&bad, h->d_bad, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return fail(SPGG_E_CUDA, "spgg_strip_failed: copy failed");
  return bad == 0x7fffffff ? 0 : bad;
}

// back to just before that launch: the caller re-runs iterations bad .. n of the chunk
extern "C" int spgg_strip_rewind(spgg_t *h, int bad) {
  if (!h || !h->pending || !h->d_bad) return fail(SPGG_E_STATE, "spgg_strip_rewind outside a chunk");
  if (bad < 1 || bad > h->pend_n) return fail(SPGG_E_INVALID, "launch %d outside the chunk of %d", bad, h->pend_n);
  h->in_rerun = true;   // (the test hook does not spoil re-runs; cleared by the next spgg_begin_steps)
  h->ccl_valid = h->ccl_local = false;
  if (h->d_ring) {      // ring mode: every rank empties its own ring and starts counting launches again; the
    CUDA_TRY(cudaMemset(h->d_ring, 0, sizeof(unsigned) * RING_SLOTS * RING_WORDS));  // caller puts a barrier
    h->gen = 0;                                                                        // between this and the re-run
    h->last_gen = -1;
  }
  return rewind_to_failed_launch(h, bad);
}

extern "C" int64_t spgg_halo_bytes(spgg_t *h) {
  if (!h) return 0;
  const Geom &g = h->g;
  const int64_t per_rep = (int64_t)GH * g.pitchB * (int64_t)(h->elem_code() + h->elem_R()) + (int64_t)GH * g.pitchW * 4;
  return per_rep * h->n_rep;
}

extern "C" int spgg_halo_pack(spgg_t *h, void *to_up, void *to_down, void *stream_) {
  if (!h || !to_up || !to_down) return fail(SPGG_E_INVALID, "spgg_halo_pack: null argument");
  cudaStream_t st = (cudaStream_t)stream_;
  const long long rep_bytes = spgg_halo_bytes(h) / h->n_rep;
  const dim3 grid(std::max(1, std::min(64, (GH * h->g.pitchB + 255) / 256)), h->n_rep);
  with_mode(h->mode, [&](auto md) {
    k_halo_pack<decltype(md)><<<grid, 256, 0, st>>>(h->g, h->d_code[h->cur], h->d_R[h->cur], h->d_S[h->cur],
        (unsigned char *)to_up, (unsigned char *)to_down, rep_bytes);
  });
  CUDA_TRY(cudaGetLastError());
  h->launches += 1;
  return SPGG_OK;
}

extern "C" int spgg_halo_unpack(spgg_t *h, const void *from_up, const void *from_down, void *stream_) {
  if (!h || !from_up || !from_down) return fail(SPGG_E_INVALID, "spgg_halo_unpack: null argument");
  cudaStream_t st = (cudaStream_t)stream_;
  const long long rep_bytes = spgg_halo_bytes(h) / h->n_rep;
  const dim3 grid(std::max(1, std::min(64, (GH * h->g.pitchB + 255) / 256)), h->n_rep);
  with_mode(h->mode, [&](auto md) {
    k_halo_unpack<decltype(md)><<<grid, 256, 0, st>>>(h->g, h->d_code[h->cur], h->d_R[h->cur], h->d_S[h->cur],
        (const unsigned char *)from_up, (const unsigned char *)from_down, rep_bytes);
  });
  CUDA_TRY(cudaGetLastError());
  h->launches += 1;
  return SPGG_OK;
}
