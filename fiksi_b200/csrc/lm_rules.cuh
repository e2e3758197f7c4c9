// When the LM decisions of the global-memory paths (sparse_path.cu: host loop, sparse_batch.cu: one CTA per sketch) must be
// taken on the reference's sums.  The reference's norm_squared (fiksi/src/solve/lm.rs:195-197) is a sequential, non-fused
// sum; both paths sum squares with tree reductions, which round differently in the last bits.  A decision taken on a tree
// sum is trusted only when it is farther from its threshold than the two sums can differ; otherwise the caller redoes the
// sums left to right and decides on those.  One rule for both paths, so that they take the same decisions.
#pragma once
#include <cstdint>

namespace fk {

// Relative distance within which a tree sum and the sequential sum of `len` squares can differ.
__host__ __device__ inline double lm_sum_tolerance(uint32_t len) { return 8.0 * 1.1102230246251565e-16 * (double)len + 1e-13; }

// The first lm.rs:110 test (ssr < 1e-8 before the loop) on a tree sum over m residuals.
__host__ __device__ inline bool lm_initial_ssr_needs_exact(double ssr, uint32_t m) {
    return isfinite(ssr) && fabs(ssr - 1e-8) <= 1e-8 * lm_sum_tolerance(m);
}

// The decisions of lm.rs:139,151,164,110 after a damping iteration whose factorisation status is `fstat` (0: every pivot
// positive): step norm dn against 1e-12, trial ssr_s against ssr and 1e-8, and the relative decrease against 1e-6.
__host__ __device__ inline bool lm_step_needs_exact(int fstat, double dn, double ssr_s, double ssr, uint32_t n, uint32_t m) {
    const double tol = lm_sum_tolerance(n > m ? n : m);
    auto near = [&](double a, double b) { return fabs(a - b) <= tol * fmax(fabs(a), fabs(b)); };
    return fstat == 0 && isfinite(ssr_s) && isfinite(dn) &&
           (near(dn, 1e-12) || near(ssr_s, ssr) || near(ssr_s, 1e-8) || (ssr_s < ssr && fabs((ssr - ssr_s) / ssr - 1e-6) <= 4.0 * tol));
}

}  // namespace fk
