// One covariance entry from the scaled squared distance r2 = sum_d ((a_d - b_d) w_d)^2 (oracle/SPEC.md), shared by the
// covariance builder (cov.cu) and the slice-step kernel (slice_step.cu): one expression, so that both make the same
// operations (and the same contractions) of it.
#pragma once
#include "b7_internal.h"
#include "exp_neg.cuh"

namespace {

template <int KERNEL>
__device__ __forceinline__ double cov_value(double r2, double sf2, const double* __restrict__ tab) {
  if (KERNEL == B7_KERNEL_ARDSE) return sf2 * exp_neg(-0.5 * r2, tab);
  double rr = sqrt(r2), s5r = 2.23606797749978969641 * rr;
  return sf2 * ((1.0 + s5r + (5.0 / 3.0) * r2) * exp_neg(-s5r, tab));
}

}  // namespace
