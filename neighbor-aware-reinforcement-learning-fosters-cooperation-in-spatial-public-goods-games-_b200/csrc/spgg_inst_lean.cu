// Instantiations of the lean kernels (spgg_lean.cuh): one translation unit of libspgg_b200, see spgg_dispatch.h.
#include "spgg_dispatch.h"
#include "spgg_lean.cuh"

namespace spgg {

template <class Md, int M>
static step_fn_t pick_lean2(int action, int replay) {
  if (action) return replay ? k_step_lean<Md, M, true, true> : k_step_lean<Md, M, true, false>;
  return replay ? k_step_lean<Md, M, false, true> : k_step_lean<Md, M, false, false>;
}
template <class Md>
static step_fn_t pick_lean1(int M, int action, int replay) {
  return M == 2 ? pick_lean2<Md, 2>(action, replay) : pick_lean2<Md, 1>(action, replay);
}
// the lean Q-learning update of the general path
step_fn_t pick_lean(int mode, int M, int action, int replay) {
  switch (mode) {
    case MODE_F32_I8: return pick_lean1<ModeF32I8>(M, action, replay);
    case MODE_F32_F: return pick_lean1<ModeF32F>(M, action, replay);
    default: return pick_lean1<ModeF64>(M, action, replay);
  }
}
// the global maximum of the general path
gmax_fn_t pick_gmax_lean(int mode, int M) {
  switch (mode) {
    case MODE_F32_I8: return M == 2 ? k_gmax_lean<ModeF32I8, 2> : k_gmax_lean<ModeF32I8, 1>;
    case MODE_F32_F: return M == 2 ? k_gmax_lean<ModeF32F, 2> : k_gmax_lean<ModeF32F, 1>;
    default: return M == 2 ? k_gmax_lean<ModeF64, 2> : k_gmax_lean<ModeF64, 1>;
  }
}
cudaError_t launch_build_valtab(const RepConst *rc_all, double *tab, int n_rep) {
  k_build_valtab<<<dim3((1u << VALTAB_BITS) / 256, (unsigned)n_rep), 256>>>(rc_all, tab);
  return cudaGetLastError();
}

}  // namespace spgg
