// Library-internal entry of the single-run gradient diagnostics (uml_linear_grad_diag, step.cu): the kernels live in
// sweep.cu next to the sweep's diagnostics, whose reduction and finish they share.  Hidden: not part of the C ABI.
#pragma once

#include "common.cuh"

namespace uml {

// Exact path: the step's fp32 G ([n0 + n1, ldg], image rows first) and its rows - run s dense from rows[s] (idx[s] NULL)
// or gathered by idx[s], ld[s] apart - through the sweep's tensor-core diagnostics pass as a one-head problem, then its
// fixed-order finish into out[4].  Two launches.
__attribute__((visibility("hidden"))) int grad_diag_f32_one(const float* const rows[2], const int64_t* const idx[2],
                                                            const int64_t ld[2], int64_t n0, int64_t n1, int32_t dim,
                                                            int32_t n_classes, const float* G, int64_t ldg, float alpha,
                                                            float* scratch, float* out, cudaStream_t st);

// bf16 path: the four sums from the split-K partials of A ([na][n], NULL when na == 0) and of B ([nb][n]) of n = C * D
// elements (n % 4 == 0), summed per element in split order, reduced into per-block slots (grad_diag_partial_slots() * 4
// floats) and finished in a fixed order into out[4], the text side divided by alpha / alpha^2 when n1 > 0.  Two launches.
__attribute__((visibility("hidden"))) int grad_diag_partials_one(const float* pa, int32_t na, const float* pb, int32_t nb,
                                                                 int64_t n, int64_t n1, float alpha, float* slots, float* out,
                                                                 cudaStream_t st);
__attribute__((visibility("hidden"))) int32_t grad_diag_partial_slots();

}  // namespace uml
