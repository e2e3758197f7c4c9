// Kernels of fk_system_batch_solve (System::solve over n variants of one drawing): the scale, perturbation and gather of
// every component's input rows into its structure's batch buffers, and the write-back of the solved components into the
// variants' variable rows.  The arithmetic of the pre-processing is prepare.cuh's, shared with fk_batch_prepare_kernel.
#include <cuda_runtime.h>

#include <algorithm>

#include "prepare.cuh"
#include "system_batch.cuh"

namespace fk {

namespace {
constexpr uint32_t kPrepVariants = 128;  // variants per CTA of the prepare kernel, one thread each for the sequential scale sum
}

// One CTA per kPrepVariants variants.  First every thread computes its variant's scale (the reference's sequential sums,
// so one thread per variant), then the CTA writes the input rows of its variants structure by structure: the rows of
// variants [v0, v0 + nb) are contiguous in every structure's buffers (sketch = variant * mult + member), so consecutive
// threads write consecutive doubles.
__global__ void __launch_bounds__(kPrepVariants)
fk_system_batch_prepare_kernel(uint32_t n, uint32_t n_vars, uint32_t n_expr, uint32_t n_constraints, const uint8_t* __restrict__ kinds,
                               const uint32_t* __restrict__ expr_constraint, const double* __restrict__ draws, uint32_t perturb,
                               const double* __restrict__ raw_vars, uint32_t raw_vars_stride, const double* __restrict__ raw_param,
                               const double* __restrict__ tmpl_param, uint32_t n_structures, const SbStructure* __restrict__ structures,
                               double* __restrict__ scales) {
    __shared__ double s_recip[kPrepVariants];
    const uint32_t v0 = blockIdx.x * kPrepVariants;
    const uint32_t nb = min(kPrepVariants, n - v0);
    // raw parameter of expression e in variant v
    auto param_of = [&](uint32_t v, uint32_t e) -> double {
        const uint32_t c = raw_param ? __ldg(expr_constraint + e) : kSbNone;
        return c != kSbNone ? __ldg(raw_param + (size_t)v * n_constraints + c) : __ldg(tmpl_param + e);
    };
    if (threadIdx.x < nb) {
        const uint32_t v = v0 + threadIdx.x;
        const double scale =
            prepare_scale(raw_vars + (size_t)v * raw_vars_stride, n_vars, n_expr, kinds, [&](uint32_t e) { return param_of(v, e); });
        s_recip[threadIdx.x] = 1.0 / scale;
        scales[v] = scale;
    }
    __syncthreads();
    for (uint32_t s = 0; s < n_structures; s++) {
        const SbStructure S = structures[s];
        const uint32_t vrow = S.mult * S.nv, prow = S.mult * S.ne;
        double* ov = S.vars + (size_t)v0 * vrow;
        for (uint32_t i = threadIdx.x; i < nb * vrow; i += kPrepVariants) {
            const uint32_t b = i / vrow, r = i - b * vrow;
            const uint32_t g = __ldg(S.slot_var + r), d = __ldg(S.slot_draw + r);
            double col = __ldg(raw_vars + (size_t)(v0 + b) * raw_vars_stride + g) * s_recip[b];
            if (perturb && d != kSbNone) col = prepare_perturb(col, __ldg(draws + 2 * (size_t)d), __ldg(draws + 2 * (size_t)d + 1));
            ov[i] = col;
        }
        double* op = S.params + (size_t)v0 * prow;
        for (uint32_t i = threadIdx.x; i < nb * prow; i += kPrepVariants) {
            const uint32_t b = i / prow, r = i - b * prow;
            const uint32_t e = __ldg(S.expr + r);
            const double q = param_of(v0 + b, e);
            op[i] = prepare_is_distance(__ldg(kinds + e)) ? s_recip[b] * q : q;
        }
    }
}

// system.variables after the solve (assemble/mod.rs:161-166): solved free variables scale * x, everything else as it came in.
__global__ void __launch_bounds__(256)
fk_system_batch_scatter_kernel(uint32_t n, uint32_t n_vars, const double* __restrict__ raw_vars, uint32_t raw_vars_stride,
                               const double* __restrict__ scales, const uint32_t* __restrict__ var_struct, const uint32_t* __restrict__ var_off,
                               uint32_t n_reports, const uint32_t* __restrict__ comp_struct, const uint32_t* __restrict__ comp_member,
                               const SbStructure* __restrict__ structures, double* __restrict__ vars_out, uint64_t* __restrict__ reports_out) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t total = (uint64_t)n * n_vars;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < total; i += stride) {
        const uint64_t v = i / n_vars;
        const uint32_t g = (uint32_t)(i - v * n_vars);
        const uint32_t s = __ldg(var_struct + g);
        double x;
        if (s == kSbNone) {
            x = __ldg(raw_vars + v * raw_vars_stride + g);
        } else {
            const SbStructure& S = structures[s];
            x = __ldg(scales + v) * __ldg(S.out + v * S.mult * S.nf + __ldg(var_off + g));
        }
        vars_out[i] = x;
    }
    constexpr uint32_t W = sizeof(fk_report) / 8;
    const uint64_t words = (uint64_t)n * n_reports * W;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < words; i += stride) {
        const uint64_t vk = i / W;
        const uint32_t w = (uint32_t)(i - vk * W);
        const uint64_t v = vk / n_reports;
        const uint32_t k = (uint32_t)(vk - v * n_reports);
        const SbStructure& S = structures[__ldg(comp_struct + k)];
        reports_out[i] = __ldg((const unsigned long long*)(S.reps + v * S.mult + __ldg(comp_member + k)) + w);
    }
}

int launch_system_batch_prepare(uint32_t n, uint32_t n_vars, uint32_t n_expr, uint32_t n_constraints, const uint8_t* kinds,
                                const uint32_t* expr_constraint, const double* draws, int perturb, const double* raw_vars,
                                uint32_t raw_vars_stride, const double* raw_param, const double* tmpl_param, uint32_t n_structures,
                                const SbStructure* structures, double* scales, void* stream) {
    if (n == 0) return 0;
    fk_system_batch_prepare_kernel<<<(n + kPrepVariants - 1) / kPrepVariants, kPrepVariants, 0, (cudaStream_t)stream>>>(
        n, n_vars, n_expr, n_constraints, kinds, expr_constraint, draws, perturb ? 1u : 0u, raw_vars, raw_vars_stride, raw_param, tmpl_param,
        n_structures, structures, scales);
    return (int)cudaGetLastError();
}

int launch_system_batch_scatter(uint32_t n, uint32_t n_vars, const double* raw_vars, uint32_t raw_vars_stride, const double* scales,
                                const uint32_t* var_struct, const uint32_t* var_off, uint32_t n_reports, const uint32_t* comp_struct,
                                const uint32_t* comp_member, const SbStructure* structures, double* vars_out, fk_report* reports_out,
                                void* stream) {
    static_assert(sizeof(fk_report) % 8 == 0, "fk_report is moved as 64-bit words");
    const uint64_t total = std::max<uint64_t>((uint64_t)n * n_vars, (uint64_t)n * n_reports * (sizeof(fk_report) / 8));
    if (total == 0) return 0;
    const uint32_t grid = (uint32_t)std::min<uint64_t>((total + 255) / 256, 148u * 16u);
    fk_system_batch_scatter_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(n, n_vars, raw_vars, raw_vars_stride, scales, var_struct, var_off,
                                                                          n_reports, comp_struct, comp_member, structures, vars_out,
                                                                          (uint64_t*)reports_out);
    return (int)cudaGetLastError();
}

}  // namespace fk
