// Instantiations of the general kernels (spgg_kernels.cuh): one translation unit of libspgg_b200, see spgg_dispatch.h.
#include "spgg_dispatch.h"

namespace spgg {

template <class Md, int M>
static step_fn_t pick_step2(int action, int replay) {
  if (action) return replay ? k_step<Md, M, true, true> : k_step<Md, M, true, false>;
  return replay ? k_step<Md, M, false, true> : k_step<Md, M, false, false>;
}
template <class Md>
static step_fn_t pick_step1(int M, int action, int replay) {
  return M == 2 ? pick_step2<Md, 2>(action, replay) : pick_step2<Md, 1>(action, replay);
}
step_fn_t pick_step(int mode, int M, int action, int replay) {
  switch (mode) {
    case MODE_F32_I8: return pick_step1<ModeF32I8>(M, action, replay);
    case MODE_F32_F: return pick_step1<ModeF32F>(M, action, replay);
    default: return pick_step1<ModeF64>(M, action, replay);
  }
}

}  // namespace spgg
