// Kernels of fk_system_batch_solve (System::solve over n variants of one drawing): the scale, perturbation and gather of
// every component's input rows into its structure's batch buffers, and the write-back of the solved components into the
// variants' variable rows.  The arithmetic of the pre-processing is prepare.cuh's, shared with fk_batch_prepare_kernel.
// fk_system_batch_solve_single_pass and _recursive_assembly reuse the prepare kernel (one identity structure: the resident
// scaled rows) and move values between the waves of sets or steps with fk_system_sp_gather_scatter_kernel.
// fk_system_batch_analyze and fk_system_batch_residuals expand the variants' parameter rows, then reduce the analyze flags
// per constraint or evaluate every constraint's residual.  fk_systems_solve (n different drawings) has its own prepare and
// scatter kernels over ragged rows: every drawing its own size, every component its own destination.
#include <cuda_runtime.h>

#include <algorithm>

#include "expressions.cuh"
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
    auto param_of = [&](uint32_t v, uint32_t e) { return variant_param(raw_param, n_constraints, expr_constraint, tmpl_param, v, e); };
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

// Between two waves of fk_system_batch_solve_single_pass / _recursive_assembly.  One CTA per `vb` consecutive variants, so
// that the phases (scatter, moves and reports, perturbations, gather, write-back) of a variant are ordered by __syncthreads
// alone.  A group's rows of variants [v0, v0 + nb) are contiguous in its batch buffers (sketch = variant * mult + member):
// consecutive threads read the solved values and write the gathered rows at consecutive addresses; the resident rows vt / pt
// are read and written by index.  Steps of one wave move disjoint points (the waves order every step after the steps that
// read or write what it writes), so one thread per (variant, step) applies that step's moves in their recorded order.
__global__ void __launch_bounds__(256)
fk_system_sp_gather_scatter_kernel(uint32_t n, uint32_t vb, uint32_t n_vars, uint32_t n_expr, double* __restrict__ vt,
                                   const double* __restrict__ pt, uint32_t n_scatter, const SpGroup* __restrict__ scatter,
                                   uint32_t n_reports, uint64_t* __restrict__ reports_out, uint32_t n_perturb,
                                   const uint32_t* __restrict__ perturb_var, const uint32_t* __restrict__ perturb_draw,
                                   const double* __restrict__ draws, uint32_t n_gather, const SpGroup* __restrict__ gather,
                                   const uint8_t* __restrict__ solved, const double* __restrict__ raw_vars, uint32_t raw_vars_stride,
                                   const double* __restrict__ scales, double* __restrict__ vars_out) {
    const uint32_t v0 = blockIdx.x * vb;
    const uint32_t nb = min(vb, n - v0);
    double* vrow = vt + (size_t)v0 * n_vars;
    for (uint32_t g = 0; g < n_scatter; g++) {  // assemble/mod.rs:201-208 (:226-233): the solution replaces its free variables
        const SpGroup G = scatter[g];
        const uint32_t row = G.s.mult * G.s.nf;
        const double* src = G.s.out + (size_t)v0 * row;
        for (uint32_t i = threadIdx.x; i < nb * row; i += blockDim.x) {
            const uint32_t b = i / row, r = i - b * row;
            const uint32_t f = __ldg(G.free_var + r);
            if (f != kSbNone) vrow[(size_t)b * n_vars + f] = src[i];
        }
    }
    __syncthreads();
    for (uint32_t g = 0; g < n_scatter; g++) {
        const SpGroup G = scatter[g];
        const uint32_t row = G.s.mult * G.s.nf;
        for (uint32_t i = threadIdx.x; i < nb * G.s.mult; i += blockDim.x) {  // assemble/mod.rs:235-273: owned points follow the pose
            const uint32_t b = i / G.s.mult, m = i - b * G.s.mult;
            const double* x = G.s.out + (size_t)(v0 + b) * row + (size_t)m * G.s.nf;
            double* p = vrow + (size_t)b * n_vars;
            for (uint32_t k = __ldg(G.move_off + m), end = __ldg(G.move_off + m + 1); k < end; k++) {
                const uint32_t pv = __ldg(G.moves + 2 * (size_t)k), col = __ldg(G.moves + 2 * (size_t)k + 1);
                const double tx = x[col + 1], ty = x[col + 2];
                double sn, cs;
                sincos(x[col], &sn, &cs);
                const double u = p[pv], w = p[pv + 1];  // Pose2D::transform_point, expressions.rs:1122-1136
                const double uc = u * cs, us = u * sn, vc = w * cs, vs = w * sn;
                p[pv] = tx + uc - vs;
                p[pv + 1] = ty + us + vc;
            }
        }
        constexpr uint32_t W = sizeof(fk_report) / 8;
        const uint32_t words = G.s.mult * W;
        const unsigned long long* rsrc = (const unsigned long long*)(G.s.reps + (size_t)v0 * G.s.mult);
        for (uint32_t i = threadIdx.x; i < nb * words; i += blockDim.x) {
            const uint32_t b = i / words, r = i - b * words, m = r / W, w = r - m * W;
            const uint32_t k = __ldg(G.step + m);
            if (k < n_reports) reports_out[((size_t)(v0 + b) * n_reports + k) * W + w] = rsrc[i];
        }
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < nb * n_perturb; i += blockDim.x) {  // assemble/mod.rs:113-124, this component's turn
        const uint32_t b = i / n_perturb, k = i - b * n_perturb;
        const uint32_t d = __ldg(perturb_draw + k);
        double& x = vrow[(size_t)b * n_vars + __ldg(perturb_var + k)];
        x = prepare_perturb(x, __ldg(draws + 2 * (size_t)d), __ldg(draws + 2 * (size_t)d + 1));
    }
    __syncthreads();
    for (uint32_t g = 0; g < n_gather; g++) {
        const SpGroup G = gather[g];
        const uint32_t row = G.s.mult * G.s.nv, prow = G.s.mult * G.s.ne;
        double* ov = G.s.vars + (size_t)v0 * row;
        for (uint32_t i = threadIdx.x; i < nb * row; i += blockDim.x) {
            const uint32_t b = i / row, r = i - b * row;
            const uint32_t sv = __ldg(G.s.slot_var + r);
            ov[i] = sv == kSbNone ? 0.0 : vrow[(size_t)b * n_vars + sv];  // (a pose column starts at the identity)
        }
        double* op = G.s.params + (size_t)v0 * prow;
        const double* prow_src = pt + (size_t)v0 * n_expr;
        for (uint32_t i = threadIdx.x; i < nb * prow; i += blockDim.x) {
            const uint32_t b = i / prow, r = i - b * prow;
            const uint32_t e = __ldg(G.s.expr + r);
            op[i] = e == kSbNone ? 0.0 : __ldg(prow_src + (size_t)b * n_expr + e);
        }
    }
    if (!vars_out) return;
    for (uint32_t i = threadIdx.x; i < nb * n_vars; i += blockDim.x) {  // assemble/mod.rs:201-208: system.variables
        const uint32_t b = i / n_vars, g = i - b * n_vars;
        const size_t v = v0 + b;
        vars_out[v * n_vars + g] = __ldg(solved + g) ? __ldg(scales + v) * vrow[i] : __ldg(raw_vars + v * raw_vars_stride + g);
    }
}

// ---- fk_systems_solve: n different drawings ----------------------------------------------------------------------------
namespace {
// Drawings per CTA of the two kernels of fk_systems_solve.  One thread owns a drawing's scale (the reference's sequential
// sum); 32 keeps a call of a thousand mid-size drawings on 32 CTAs rather than 8.
constexpr uint32_t kSysDrawings = 32, kSysThreads = 128;
}  // namespace

// One CTA per kSysDrawings consecutive drawings.  The first warp computes their scales, then the CTA's warps take the drawings'
// instances (consecutive: [inst_off[d0], inst_off[d0 + nb])) one each, the lanes over its local variables and expressions.
__global__ void __launch_bounds__(kSysThreads)
fk_systems_prepare_kernel(uint32_t n, const uint64_t* __restrict__ var_off, const uint64_t* __restrict__ expr_off,
                          const uint32_t* __restrict__ inst_off, const uint8_t* __restrict__ kinds, const double* __restrict__ raw_vars,
                          const double* __restrict__ raw_param, const double* __restrict__ draws, uint32_t perturb,
                          const SysInst* __restrict__ inst, const uint32_t* __restrict__ tabs, double* __restrict__ scales) {
    __shared__ double s_recip[kSysDrawings];
    const uint32_t d0 = blockIdx.x * kSysDrawings;
    const uint32_t nb = min(kSysDrawings, n - d0);
    if (threadIdx.x < nb) {
        const uint32_t d = d0 + threadIdx.x;
        const uint64_t v0 = __ldg(var_off + d), e0 = __ldg(expr_off + d);
        const double* q = raw_param + e0;
        const double scale = prepare_scale(raw_vars + v0, (uint32_t)(__ldg(var_off + d + 1) - v0), (uint32_t)(__ldg(expr_off + d + 1) - e0),
                                           kinds + e0, [&](uint32_t e) { return __ldg(q + e); });
        s_recip[threadIdx.x] = 1.0 / scale;
        scales[d] = scale;
    }
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    for (uint32_t k = __ldg(inst_off + d0) + warp, end = __ldg(inst_off + d0 + nb); k < end; k += kSysThreads / 32) {
        const SysInst I = inst[k];
        const double recip = s_recip[I.drawing - d0];
        const double* rv = raw_vars + __ldg(var_off + I.drawing);
        const uint64_t e0 = __ldg(expr_off + I.drawing);
        const uint32_t* slot_var = tabs + I.tab;
        const uint32_t* slot_draw = slot_var + I.nv;
        const uint32_t* expr = slot_draw + I.nv;
        for (uint32_t j = lane; j < I.nv; j += 32) {
            const uint32_t dr = __ldg(slot_draw + j);
            double col = __ldg(rv + __ldg(slot_var + j)) * recip;
            if (perturb && dr != kSbNone) col = prepare_perturb(col, __ldg(draws + 2 * (size_t)dr), __ldg(draws + 2 * (size_t)dr + 1));
            I.vars[j] = col;
        }
        for (uint32_t j = lane; j < I.ne; j += 32) {
            const uint64_t e = e0 + __ldg(expr + j);
            const double q = __ldg(raw_param + e);
            I.params[j] = prepare_is_distance(__ldg(kinds + e)) ? recip * q : q;
        }
    }
}

// system.variables after the solve (assemble/mod.rs:161-166), per drawing: every variable as it came in, then (after the
// CTA's barrier, so the raw copy never lands on a solved value) scale * x for the solved free variables.  The reports go to
// the instance's slot.
__global__ void __launch_bounds__(kSysThreads)
fk_systems_scatter_kernel(uint32_t n, const uint64_t* __restrict__ var_off, const uint32_t* __restrict__ inst_off,
                          const double* __restrict__ raw_vars, const double* __restrict__ scales, const SysInst* __restrict__ inst,
                          const uint32_t* __restrict__ tabs, double* __restrict__ vars_out, uint64_t* __restrict__ reports_out) {
    const uint32_t d0 = blockIdx.x * kSysDrawings;
    const uint32_t nb = min(kSysDrawings, n - d0);
    for (uint64_t i = __ldg(var_off + d0) + threadIdx.x, end = __ldg(var_off + d0 + nb); i < end; i += kSysThreads) vars_out[i] = __ldg(raw_vars + i);
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    constexpr uint32_t W = sizeof(fk_report) / 8;
    for (uint32_t k = __ldg(inst_off + d0) + warp, end = __ldg(inst_off + d0 + nb); k < end; k += kSysThreads / 32) {
        const SysInst I = inst[k];
        const double scale = __ldg(scales + I.drawing);
        double* row = vars_out + __ldg(var_off + I.drawing);
        const uint32_t* free_var = tabs + I.tab + 2 * (uint64_t)I.nv + I.ne;
        for (uint32_t j = lane; j < I.nf; j += 32) row[__ldg(free_var + j)] = scale * __ldg(I.out + j);
        if (lane < W) reports_out[(uint64_t)k * W + lane] = __ldg((const unsigned long long*)I.rep + lane);
    }
}

int launch_systems_prepare(uint32_t n, const uint64_t* var_off, const uint64_t* expr_off, const uint32_t* inst_off, const uint8_t* kinds,
                           const double* raw_vars, const double* raw_param, const double* draws, int perturb, const SysInst* inst,
                           const uint32_t* tabs, double* scales, void* stream) {
    if (n == 0) return 0;
    fk_systems_prepare_kernel<<<(n + kSysDrawings - 1) / kSysDrawings, kSysThreads, 0, (cudaStream_t)stream>>>(
        n, var_off, expr_off, inst_off, kinds, raw_vars, raw_param, draws, perturb ? 1u : 0u, inst, tabs, scales);
    return (int)cudaGetLastError();
}

int launch_systems_scatter(uint32_t n, const uint64_t* var_off, const uint32_t* inst_off, const double* raw_vars, const double* scales,
                           const SysInst* inst, const uint32_t* tabs, double* vars_out, fk_report* reports_out, void* stream) {
    static_assert(sizeof(fk_report) % 8 == 0 && sizeof(fk_report) / 8 <= 32, "fk_report is moved as 64-bit words by one warp");
    if (n == 0) return 0;
    fk_systems_scatter_kernel<<<(n + kSysDrawings - 1) / kSysDrawings, kSysThreads, 0, (cudaStream_t)stream>>>(
        n, var_off, inst_off, raw_vars, scales, inst, tabs, vars_out, (uint64_t*)reports_out);
    return (int)cudaGetLastError();
}

// ---- fk_system_batch_analyze / fk_system_batch_residuals ---------------------------------------------------------------
namespace {
uint32_t grid_for(uint64_t total) { return (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((total + 255) / 256, 148u * 16u)); }
}  // namespace

// The variants' rows as the analyze kernels and fk_system_residuals_kernel read them: pt[v][e] = variant_param, and, given
// tmpl_vars (the call passed no variables), vt[v] = tmpl_vars.
__global__ void __launch_bounds__(256)
fk_system_an_expand_kernel(uint32_t n, uint32_t n_vars, uint32_t n_expr, uint32_t n_constraints, const double* __restrict__ tmpl_vars,
                           double* __restrict__ vt, const uint32_t* __restrict__ expr_constraint, const double* __restrict__ raw_param,
                           const double* __restrict__ tmpl_param, double* __restrict__ pt) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t first = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (tmpl_vars)
        for (uint64_t i = first; i < (uint64_t)n * n_vars; i += stride) vt[i] = __ldg(tmpl_vars + i % n_vars);
    for (uint64_t i = first; i < (uint64_t)n * n_expr; i += stride) {
        const uint64_t v = i / n_expr;
        pt[i] = variant_param(raw_param, n_constraints, expr_constraint, tmpl_param, v, (uint32_t)(i - v * n_expr));
    }
}

// dependent[v][c] = the expressions [con_off[c], con_off[c + 1]) of constraint c that analyze found dependent.
__global__ void __launch_bounds__(256)
fk_system_an_reduce_kernel(uint32_t n, uint32_t n_expr, uint32_t n_constraints, const uint8_t* __restrict__ independent,
                           const uint32_t* __restrict__ con_off, uint8_t* __restrict__ dependent) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < (uint64_t)n * n_constraints; i += stride) {
        const uint64_t v = i / n_constraints;
        const uint32_t c = (uint32_t)(i - v * n_constraints);
        uint32_t d = 0;
        for (uint32_t e = __ldg(con_off + c), end = __ldg(con_off + c + 1); e < end; e++) d += independent[v * n_expr + e] ? 0u : 1u;
        dependent[i] = (uint8_t)d;
    }
}

// out[v][c] = calculate_residual (constraints/mod.rs:88-110) of constraint c in variant v, as fk_system_residuals combines the
// expression residuals: a one-expression constraint its residual, otherwise q += r * r in expression order, then sqrt(q).
// The slots are read as the analyze kernels read them (slot_var[e][8], arity_of), the residual is eval_expression's.
__global__ void __launch_bounds__(256)
fk_system_residuals_kernel(uint32_t n, uint32_t n_vars, uint32_t n_expr, uint32_t n_constraints, const uint8_t* __restrict__ kinds,
                           const uint32_t* __restrict__ slot_var, const uint32_t* __restrict__ con_off, const double* __restrict__ vt,
                           const double* __restrict__ pt, double* __restrict__ out) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < (uint64_t)n * n_constraints; i += stride) {
        const uint64_t v = i / n_constraints;
        const uint32_t c = (uint32_t)(i - v * n_constraints);
        const double* vars = vt + v * n_vars;
        const uint32_t e0 = __ldg(con_off + c), e1 = __ldg(con_off + c + 1);
        double q = 0.0, r = 0.0;
        for (uint32_t e = e0; e < e1; e++) {
            const int kind = (int)__ldg(kinds + e);
            const int ar = dev::arity_of(kind);
            double x[8], g[8];
#pragma unroll
            for (int sl = 0; sl < 8; sl++) x[sl] = sl < ar ? __ldg(vars + __ldg(slot_var + (size_t)e * 8 + sl)) : 0.0;
            r = dev::eval_expression(kind, x, __ldg(pt + v * n_expr + e), g);
            q += r * r;
        }
        out[i] = e1 - e0 > 1 ? sqrt(q) : r;
    }
}

int launch_system_an_expand(uint32_t n, uint32_t n_vars, uint32_t n_expr, uint32_t n_constraints, const double* tmpl_vars, double* vt,
                            const uint32_t* expr_constraint, const double* raw_param, const double* tmpl_param, double* pt, void* stream) {
    const uint64_t total = (uint64_t)n * std::max(tmpl_vars ? n_vars : 0u, n_expr);
    if (total == 0) return 0;
    fk_system_an_expand_kernel<<<grid_for(total), 256, 0, (cudaStream_t)stream>>>(n, n_vars, n_expr, n_constraints, tmpl_vars, vt,
                                                                                  expr_constraint, raw_param, tmpl_param, pt);
    return (int)cudaGetLastError();
}

int launch_system_an_reduce(uint32_t n, uint32_t n_expr, uint32_t n_constraints, const uint8_t* independent, const uint32_t* con_off,
                            uint8_t* dependent, void* stream) {
    const uint64_t total = (uint64_t)n * n_constraints;
    if (total == 0) return 0;
    fk_system_an_reduce_kernel<<<grid_for(total), 256, 0, (cudaStream_t)stream>>>(n, n_expr, n_constraints, independent, con_off, dependent);
    return (int)cudaGetLastError();
}

int launch_system_residuals(uint32_t n, uint32_t n_vars, uint32_t n_expr, uint32_t n_constraints, const uint8_t* kinds, const uint32_t* slot_var,
                            const uint32_t* con_off, const double* vt, const double* pt, double* out, void* stream) {
    const uint64_t total = (uint64_t)n * n_constraints;
    if (total == 0) return 0;
    fk_system_residuals_kernel<<<grid_for(total), 256, 0, (cudaStream_t)stream>>>(n, n_vars, n_expr, n_constraints, kinds, slot_var, con_off,
                                                                                  vt, pt, out);
    return (int)cudaGetLastError();
}

int launch_system_sp_gather_scatter(uint32_t n, uint32_t n_vars, uint32_t n_expr, double* vt, const double* pt, uint32_t n_scatter,
                                    const SpGroup* scatter, uint32_t n_reports, fk_report* reports_out, uint32_t n_perturb,
                                    const uint32_t* perturb_var, const uint32_t* perturb_draw, const double* draws, uint32_t n_gather,
                                    const SpGroup* gather, const uint8_t* solved, const double* raw_vars, uint32_t raw_vars_stride,
                                    const double* scales, double* vars_out, void* stream) {
    static_assert(sizeof(fk_report) % 8 == 0, "fk_report is moved as 64-bit words");
    if (n == 0) return 0;
    // up to 32 variants per CTA, fewer while that leaves under four CTAs per SM
    const uint32_t vb = std::max<uint32_t>(1, std::min<uint32_t>(32, n / (148u * 4u)));
    fk_system_sp_gather_scatter_kernel<<<(n + vb - 1) / vb, 256, 0, (cudaStream_t)stream>>>(
        n, vb, n_vars, n_expr, vt, pt, n_scatter, scatter, n_reports, (uint64_t*)reports_out, n_perturb, perturb_var, perturb_draw, draws,
        n_gather, gather, solved, raw_vars, raw_vars_stride, scales, vars_out);
    return (int)cudaGetLastError();
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
