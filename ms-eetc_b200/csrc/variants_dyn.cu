// Translation unit of libmseetc_b200.so: interval kernels with the spline loss map of efficiency.py (see variants.h).
#include "variants.h"

namespace mseetc {
namespace {
// the row gradients of the loss rows come from the stage-QP record (see cell_step)
MS_CELL_KERNEL(k_cell_init_dyn, 2, cell_init<true>(c, k, s))
MS_CELL_KERNEL(k_cell_trial_eval_dyn, 2, (cell_eval<true, true>(c, k, s)))
MS_CELL_KERNEL(k_cell_eval_dyn, 2, (cell_eval<true, false>(c, k, s)))
MS_CELL_KERNEL(k_cell_step_dyn, CELL_STEP_MINB, cell_step<true>(c, k, s))
}  // namespace

void launch_variant_dyn(int which, unsigned grid, cudaStream_t st, const Ctx& c, const BatchIO& io) {
    switch (which) {
        case VK_INIT_DYN: k_cell_init_dyn<<<grid, 128, 0, st>>>(c, io); break;
        case VK_EVAL_DYN: k_cell_eval_dyn<<<grid, 128, 0, st>>>(c, io); break;
        case VK_TRIAL_DYN: k_cell_trial_eval_dyn<<<grid, 128, 0, st>>>(c, io); break;
        case VK_STEP_DYN: k_cell_step_dyn<<<grid, 128, 0, st>>>(c, io); break;
        default: break;
    }
}

}  // namespace mseetc
