// Kernels of the less common problem variants -- spline loss map, collocation integrator ('IRK' / 'CVODES'), integrated losses --
// compiled in their own translation units (variants_dyn.cu, variants_irk.cu, variants_intl.cu, variants_intl_irk.cu) so that all units build side by side
// (these kernels take most of the compile time); launched from mseetc_b200.cu through launch_variant.
#pragma once
#include <cuda_runtime.h>
#include "io.cuh"

namespace mseetc {

enum VariantKernel {
    VK_INIT_DYN, VK_EVAL_DYN, VK_TRIAL_DYN, VK_STEP_DYN,                // spline loss map (efficiency.py)
    VK_EVAL_IRK, VK_EVAL_DYN_IRK, VK_TRIAL_IRK, VK_TRIAL_DYN_IRK,      // cell_eval with collocation steps
    VK_INIT_INTL, VK_EVAL_INTL, VK_TRIAL_INTL, VK_STEP_INTL, VK_LAM_INTL,     // integrateLosses = True
    VK_INIT_INTL_IRK, VK_EVAL_INTL_IRK, VK_TRIAL_INTL_IRK, VK_LAM_INTL_IRK     // ... with collocation steps
};
// one launch of 128-thread blocks on `st` (same grid-stride cell loop as the kernels of mseetc_b200.cu)
void launch_variant_dyn(int which, unsigned grid, cudaStream_t st, const Ctx& c, const BatchIO& io);
void launch_variant_irk(int which, unsigned grid, cudaStream_t st, const Ctx& c, const BatchIO& io);
void launch_variant_intl(int which, unsigned grid, cudaStream_t st, const Ctx& c, const BatchIO& io);
void launch_variant_intl_irk(int which, unsigned grid, cudaStream_t st, const Ctx& c, const BatchIO& io);
inline void launch_variant(int which, unsigned grid, cudaStream_t st, const Ctx& c, const BatchIO& io) {
    if (which <= VK_STEP_DYN) launch_variant_dyn(which, grid, st, c, io);
    else if (which <= VK_TRIAL_DYN_IRK) launch_variant_irk(which, grid, st, c, io);
    else if (which <= VK_LAM_INTL) launch_variant_intl(which, grid, st, c, io);
    else launch_variant_intl_irk(which, grid, st, c, io);
}
// mseetc_eval_interval with collocation steps (`irk`: device pointer)
void launch_eval_interval_irk(int n, int numSteps, int numApprox, const double* in, double* out, const IrkTab* irk, cudaStream_t st);

// minimum resident blocks per SM of k_cell_step and k_cell_step_dyn (3 measured faster than 2 or 4)
enum { CELL_STEP_MINB = 3 };

#define MS_CELL_KERNEL(NAME, MINB, CALL)                                        \
    __global__ void __launch_bounds__(128, MINB) NAME(Ctx c, BatchIO io) {      \
        const size_t total = (size_t)c.cfg.NK * c.cfg.S;                        \
        const size_t stride = (size_t)gridDim.x * 128;                          \
        for (size_t idx = (size_t)blockIdx.x * 128 + threadIdx.x; idx < total; idx += stride) { \
            const int s = (int)(idx % c.cfg.S);                                 \
            const int k = (int)(idx / c.cfg.S);                                 \
            CALL;                                                               \
        }                                                                       \
    }

}  // namespace mseetc
