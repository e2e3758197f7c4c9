// assemble::solve's pre-processing arithmetic (fiksi/src/assemble/mod.rs:32-44,58-79,113-124), shared by every kernel that
// scales and perturbs on the device (fk_batch_prepare_kernel, fk_system_batch_prepare_kernel), so that all of them produce
// the bits of fk_system_solve's host loop.  The including translation units are built with -fmad=false: nothing here may be
// contracted into an FMA.
#pragma once
#include <cstdint>

#include "../../include/fiksi_b200.h"

namespace fk {

__device__ __forceinline__ bool prepare_is_distance(uint32_t kind) {
    return kind == FK_POINT_POINT_DISTANCE || kind == FK_POINT_LINE_DISTANCE;
}

// Raw parameter of expression e in variant v of a System batch: raw_param[v][c] where e holds constraint c's parameter
// (expr_constraint[e] = c, 0xFFFFFFFF for none; update_parameter writes it at the constraint's first expression, constraints/mod.rs:992-1046) and
// raw_param is given, tmpl_param[e] otherwise.
__device__ __forceinline__ double variant_param(const double* __restrict__ raw_param, uint32_t n_constraints,
                                                const uint32_t* __restrict__ expr_constraint, const double* __restrict__ tmpl_param,
                                                size_t v, uint32_t e) {
    const uint32_t c = raw_param ? __ldg(expr_constraint + e) : 0xFFFFFFFFu;
    return c != 0xFFFFFFFFu ? __ldg(raw_param + v * n_constraints + c) : __ldg(tmpl_param + e);
}

// RMS scale of one sketch: every variable left to right, then the distance parameters in expression order, summed
// sequentially (fiksi/src/utils.rs:12-19).  param(e) returns the raw parameter of expression e.
template <class Param>
__device__ __forceinline__ double prepare_scale(const double* __restrict__ rv, uint32_t n_vars, uint32_t n_expr,
                                                const uint8_t* __restrict__ kinds, const Param& param) {
    double sum = 0.0;
    uint32_t cnt = n_vars;
    uint32_t i = 0;
    for (; i + 8 <= n_vars; i += 8) {  // eight loads in flight, the additions stay in order
        double v[8];
#pragma unroll
        for (int u = 0; u < 8; u++) v[u] = __ldg(rv + i + u);
#pragma unroll
        for (int u = 0; u < 8; u++) sum = sum + v[u] * v[u];
    }
    for (; i < n_vars; i++) {
        const double v = __ldg(rv + i);
        sum = sum + v * v;
    }
    for (uint32_t e = 0; e < n_expr; e++) {
        if (prepare_is_distance(__ldg(kinds + e))) {
            const double q = param(e);
            sum = sum + q * q;
            cnt++;
        }
    }
    return sqrt(sum / (double)cnt);
}

// The seeded perturbation of one scaled free variable with its two draws (assemble/mod.rs:113-124).
__device__ __forceinline__ double prepare_perturb(double col, double r1, double r2) {
    return col + (col * (1.0 / 8196.0) * r1 + (1.0 / 65568.0) * r2);
}

}  // namespace fk
