// Kernel pickers shared by the translation units of libspgg_b200.  The library is compiled as three units in
// parallel (__graft_entry__.build): spgg_capi.cu (C ABI, host logic, fast / resident / helper kernels),
// spgg_inst_general.cu (every instantiation of k_step), spgg_inst_lean.cu (k_step_lean / k_gmax_lean /
// k_build_valtab), spgg_clusters.cu (cluster labelling, k_ccl_*), spgg_pairs.cu (pair counts, k_pair*) and spgg_blocks.cu
// (block fields, k_block_*).  A kernel is compiled in the unit that instantiates it; the others launch it through the
// function pointer or the launcher declared here.
#pragma once
#include "spgg_kernels.cuh"
#include "spgg_clusters.cuh"
#include "spgg_pairs.cuh"
#include "spgg_blocks.cuh"

namespace spgg {

enum { MODE_F32_I8 = 0, MODE_F32_F = 1, MODE_F64 = 2 };

typedef void (*step_fn_t)(KArgs);
typedef void (*gmax_fn_t)(GArgs);

// spgg_inst_general.cu
step_fn_t pick_step(int mode, int M, int action, int replay);
// spgg_inst_lean.cu
step_fn_t pick_lean(int mode, int M, int action, int replay);
gmax_fn_t pick_gmax_lean(int mode, int M);
cudaError_t launch_build_valtab(const RepConst *rc_all, double *tab, int n_rep);
constexpr int LEAN_TR_MAX = 16;   // k_step_lean addresses the shared-memory layout of 16-row tiles
// spgg_clusters.cu: ccl_alloc / ccl_free / launch_clusters / launch_cluster_labels (spgg_clusters.cuh)
// spgg_pairs.cu: launch_pair_counts / launch_pair_record (spgg_pairs.cuh)
// spgg_blocks.cu: block_scratch_bytes / launch_block_fields (spgg_blocks.cuh)

}  // namespace spgg
