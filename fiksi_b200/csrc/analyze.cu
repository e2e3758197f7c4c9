// System::analyze with the matrix in global memory: one CTA per sketch, or a cooperative group of CTAs per sketch
// (analyze.cuh).  Every floating-point operation is the reference's, in the reference's order
// (incremental_gauss_jordan_elimination, fiksi/src/analyze/numerical/mod.rs:33-117, restated in oracle/fiksi_ref.hpp):
// multiply, then subtract (this file is built with -fmad=false), one IEEE reciprocal per pivot row, so the flags are
// bit-for-bit those of the CPU restatement.
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "../../include/fiksi_b200.h"
#include "analyze.cuh"
#include "expressions.cuh"
#include "lm_kernels.cuh"

namespace fk {

namespace cg = cooperative_groups;

namespace {

constexpr uint32_t kAnWarpsCta = kAnThreads / 32;

struct AnArgs {
    uint32_t n_vars, n_expr, nsteps, ld, group, n_sketches;
    uint64_t slot_doubles;
    const uint8_t* kinds;
    const uint32_t* slot_var;
    const double* vars_all;
    const double* params_all;
    uint8_t* out;
    double* ws;        // slots * slot_doubles
    unsigned* next;    // sketch counter of the persistent grid (group == 1)
};

// The matrix rows are written by one CTA and read by others (group) or by the same CTA after a barrier: every access to the
// workspace goes through L2 (.cg), so that no SM reads a stale L1 line after grid.sync().
__device__ __forceinline__ double ld2(const double* p) { return __ldcg(p); }
__device__ __forceinline__ void st2(double* p, double v) { __stcg(p, v); }
__device__ __forceinline__ uint32_t ldu(const uint32_t* p) { return __ldcg(p); }

__device__ __forceinline__ void an_sync(uint32_t group) {
    if (group > 1)
        cg::this_grid().sync();
    else
        __syncthreads();
}

}  // namespace

// Workspace of one sketch: M[nsteps][ld] (only rows 0 .. min(m, n) - 1 are ever examined or modified, mod.rs:64), then
// ci[n] (column_indices), inc[nsteps] (constraint_increases_rank) and hdr[2] (pivot column, pivot found) of the current row.

__global__ void __launch_bounds__(kAnThreads, 2)
fk_analyze_cta_kernel(AnArgs a) {
    extern __shared__ __align__(16) double R[];  // the row being reduced, then the normalised pivot row [n_vars]
    __shared__ double s_f[32];
    __shared__ uint32_t s_u[kAnWarpsCta];
    __shared__ uint32_t s_sketch;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t G = a.group, g = blockIdx.x % G, slot = blockIdx.x / G, n_slots = gridDim.x / G;
    const uint32_t n = a.n_vars, m = a.n_expr, ns = a.nsteps, ld = a.ld;
    double* M = a.ws + (size_t)slot * a.slot_doubles;
    uint32_t* ci = reinterpret_cast<uint32_t*>(M + (size_t)ns * ld);
    uint32_t* inc = ci + n;
    uint32_t* hdr = inc + ns;
    for (uint32_t round = 0;; round++) {
        uint32_t sketch;
        if (G == 1) {
            if (tid == 0) s_sketch = atomicAdd(a.next, 1u);
            __syncthreads();
            sketch = s_sketch;
            __syncthreads();
            if (sketch >= a.n_sketches) break;
        } else {
            // every group runs the same number of rounds and reaches every grid.sync(): the rows of all sketches of one
            // topology are the same, so the groups go through them in lockstep (an idle group in the last round too)
            if ((uint64_t)round * n_slots >= a.n_sketches) break;
            sketch = round * n_slots + slot;
        }
        const bool active = sketch < a.n_sketches;
        // Jacobian (mod.rs:123-147): dense over ALL variables, gradient entries ASSIGNED per slot; this CTA's row range
        {
            const uint32_t lo = (uint32_t)((uint64_t)ns * g / G), hi = (uint32_t)((uint64_t)ns * (g + 1) / G);
            if (active) {
                for (uint32_t r = lo; r < hi; r++)
                    for (uint32_t c = tid; c < n; c += kAnThreads) st2(M + (size_t)r * ld + c, 0.0);
                if (g == 0) {
                    for (uint32_t c = tid; c < n; c += kAnThreads) ci[c] = c;
                    for (uint32_t r = tid; r < ns; r += kAnThreads) inc[r] = 0;
                }
                __syncthreads();
                const double* vars = a.vars_all + (size_t)sketch * n;
                const double* params = a.params_all + (size_t)sketch * m;
                for (uint32_t row = lo + tid; row < hi; row += kAnThreads) {
                    const int kind = (int)__ldg(a.kinds + row);
                    const int ar = dev::arity_of(kind);
                    double v[8], gr[8];
                    uint32_t var[8];
#pragma unroll
                    for (int sl = 0; sl < 8; sl++) {
                        var[sl] = sl < ar ? __ldg(a.slot_var + row * 8 + sl) : 0u;
                        v[sl] = sl < ar ? __ldg(vars + var[sl]) : 0.0;
                    }
                    dev::eval_expression(kind, v, __ldg(params + row), gr);
#pragma unroll
                    for (int sl = 0; sl < 8; sl++)
                        if (sl < ar) st2(M + (size_t)row * ld + var[sl], gr[sl]);
                }
            }
            an_sync(G);
        }
        uint32_t current_col = 0;  // (CTA 0 of the group; uniform over its threads)
        for (uint32_t i = 0; i < ns; i++) {
            double* Mi = M + (size_t)i * ld;
            if (active && g == 0) {
                for (uint32_t c = tid; c < n; c += kAnThreads) R[c] = ld2(Mi + c);
                __syncthreads();
                // Elimination (mod.rs:66-77) in blocks of 32 earlier rows k.  Warp 0 forms the block's 32 factors
                // f_k = R[ci[rank_k]] from the at most 32 distinct columns they read, applying the block's earlier
                // updates to those columns in ascending k; then the whole CTA applies the 32 updates to every column,
                // again in ascending k.  Per entry that is the reference's sequence of subtractions.
                uint32_t rank = 0;  // (warp 0)
                for (uint32_t k0 = 0; k0 < i; k0 += 32) {
                    const uint32_t cnt = min(32u, i - k0);
                    if (warp == 0) {
                        const unsigned incbits = __ballot_sync(0xFFFFFFFFu, lane < cnt && ldu(inc + k0 + lane) != 0u);
                        const uint32_t col = rank + lane < n ? ldu(ci + rank + lane) : 0u;
                        double mk[32];
#pragma unroll
                        for (uint32_t j = 0; j < 32; j++) mk[j] = j < cnt ? ld2(M + (size_t)(k0 + j) * ld + col) : 0.0;
                        double v = R[col];
#pragma unroll
                        for (uint32_t j = 0; j < 32; j++) {
                            if (j < cnt) {
                                const double f = __shfl_sync(0xFFFFFFFFu, v, __popc(incbits & ((1u << j) - 1u)));
                                if (lane == 0) s_f[j] = f;
                                v = v - f * mk[j];
                            }
                        }
                        rank += __popc(incbits);
                    }
                    __syncthreads();
                    for (uint32_t c = tid; c < n; c += kAnThreads) {
                        double x = R[c];
                        if (cnt == 32) {
                            double mk[32];
#pragma unroll
                            for (uint32_t j = 0; j < 32; j++) mk[j] = ld2(M + (size_t)(k0 + j) * ld + c);
#pragma unroll
                            for (uint32_t j = 0; j < 32; j++) x = x - s_f[j] * mk[j];
                        } else {
                            for (uint32_t j = 0; j < cnt; j++) x = x - s_f[j] * ld2(M + (size_t)(k0 + j) * ld + c);
                        }
                        R[c] = x;
                    }
                    __syncthreads();
                }
                // Pivot (mod.rs:81-90): the first position p >= current_col in ci order with |R[ci[p]]| > 1e-8
                uint32_t found = 0xFFFFFFFFu;
                for (uint32_t base = current_col; base < n; base += kAnThreads) {
                    const uint32_t idx = base + tid;
                    const bool ok = idx < n && fabs(R[ldu(ci + idx)]) > 1e-8;
                    const unsigned b = __ballot_sync(0xFFFFFFFFu, ok);
                    if (lane == 0) s_u[warp] = b ? base + warp * 32u + (uint32_t)__ffs(b) - 1u : 0xFFFFFFFFu;
                    __syncthreads();
#pragma unroll
                    for (uint32_t w = 0; w < kAnWarpsCta; w++) found = min(found, s_u[w]);
                    __syncthreads();
                    if (found != 0xFFFFFFFFu) break;
                }
                if (found != 0xFFFFFFFFu) {
                    // swap ci[current_col] and ci[found] only; normalise with one IEEE reciprocal (mod.rs:93-100)
                    const uint32_t pc = ldu(ci + found);
                    const double inv = 1.0 / R[pc];
                    __syncthreads();
                    if (tid == 0) {
                        ci[found] = ldu(ci + current_col);
                        ci[current_col] = pc;
                        inc[i] = 1u;
                        hdr[0] = pc;
                        hdr[1] = 1u;
                    }
                    for (uint32_t c = tid; c < n; c += kAnThreads) R[c] = R[c] * inv;
                    current_col++;
                } else if (tid == 0) {
                    hdr[1] = 0u;
                }
                for (uint32_t c = tid; c < n; c += kAnThreads) st2(Mi + c, R[c]);  // dependent rows are kept reduced
                __syncthreads();
            }
            an_sync(G);
            // Jordan step (mod.rs:104-110): rows k < i split over the group's CTAs by ranges, one warp per row;
            // f2 = M[k][pc] is read by every lane before any lane updates row k
            if (active && ldu(hdr + 1) != 0u) {
                const uint32_t pc = ldu(hdr);
                if (g != 0) {
                    for (uint32_t c = tid; c < n; c += kAnThreads) R[c] = ld2(Mi + c);
                    __syncthreads();
                }
                const uint32_t lo = (uint32_t)((uint64_t)i * g / G), hi = (uint32_t)((uint64_t)i * (g + 1) / G);
                for (uint32_t k = lo + warp; k < hi; k += kAnWarpsCta) {
                    double* Mk = M + (size_t)k * ld;
                    const double f2 = ld2(Mk + pc);
                    __syncwarp();
                    for (uint32_t c = lane; c < n; c += 32) st2(Mk + c, ld2(Mk + c) - f2 * R[c]);
                }
            }
            an_sync(G);
        }
        if (active && g == 0) {
            uint8_t* out = a.out + (size_t)sketch * m;
            for (uint32_t r = tid; r < m; r += kAnThreads) out[r] = r < ns ? (uint8_t)ldu(inc + r) : (uint8_t)0;
        }
        __syncthreads();
    }
}

namespace {

int forced_analyze_kernel() {
    const char* e = std::getenv("FK_ANALYZE_KERNEL");
    if (!e) return -1;
    if (!std::strcmp(e, "warp")) return kAnWarp;
    if (!std::strcmp(e, "cta")) return kAnCta;
    if (!std::strcmp(e, "group")) return kAnGroup;
    return -1;
}

}  // namespace

int choose_analyze(uint32_t n_vars, uint32_t n_expr, uint32_t n_sketches, int device, AnalyzePlan* plan, std::string* err) {
    AnalyzePlan p;
    const int forced = forced_analyze_kernel();
    const bool warp_fits = batch_analyze_warp_fits(n_vars, n_expr);
    if (forced == kAnWarp || (forced < 0 && warp_fits)) {
        if (!warp_fits) {
            if (err) *err = "fk_batch_analyze: FK_ANALYZE_KERNEL=warp, but the " + std::to_string(n_expr) + " x " + std::to_string(n_vars) +
                            " matrix of one sketch does not fit a warp's 200 KiB of shared memory";
            return FK_ERR_TOO_LARGE;
        }
        *plan = p;
        return FK_OK;
    }
    p.nsteps = std::min(n_vars, n_expr);
    p.ld = (n_vars + 31u) & ~31u;
    // matrix, then ci[n] / inc[nsteps] / hdr[2] as 32-bit words, rounded to whole 256-byte lines
    const uint64_t words = (uint64_t)n_vars + p.nsteps + 2;
    p.slot_doubles = (((uint64_t)p.nsteps * p.ld + (words + 1) / 2) + 31) & ~(uint64_t)31;
    const uint64_t bytes = sizeof(double) * p.slot_doubles;
    if (n_vars > kAnMaxVars || bytes > kAnWorkspaceBytes) {
        if (err)
            *err = "fk_batch_analyze: one sketch needs " + std::to_string(bytes) + " bytes of workspace (" + std::to_string(p.nsteps) + " x " +
                   std::to_string(n_vars) + " doubles), the limit is " + std::to_string(kAnWorkspaceBytes) + " bytes; n_vars = " +
                   std::to_string(n_vars) + " against the shared-memory row cap of " + std::to_string(kAnMaxVars);
        return FK_ERR_TOO_LARGE;
    }
    int per_sm = 0, sms = 0;
    cudaError_t e = cudaFuncSetAttribute(fk_analyze_cta_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kAnMaxVars * sizeof(double)));
    if (e == cudaSuccess)
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fk_analyze_cta_kernel, kAnThreads, std::max<size_t>(8, n_vars * sizeof(double)));
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    if (e != cudaSuccess) {
        cudaGetLastError();
        if (err) *err = std::string("fk_batch_analyze: occupancy query: ") + cudaGetErrorString(e);
        return e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? FK_ERR_NO_DEVICE : FK_ERR_CUDA;
    }
    const uint64_t resident = (uint64_t)std::max(1, per_sm) * (uint64_t)sms;
    const uint64_t budget = kAnWorkspaceBytes / bytes;  // >= 1 by the limit rule
    const uint64_t slots = std::max<uint64_t>(1, std::min<uint64_t>({(uint64_t)std::max(1u, n_sketches), resident, budget}));
    uint64_t group = resident / slots;
    if (forced == kAnCta || (forced < 0 && group < 2)) {
        p.kernel = kAnCta;
        p.slots = (uint32_t)slots;
        p.group = 1;
    } else {
        p.kernel = kAnGroup;
        group = std::max<uint64_t>(2, group);
        p.group = (uint32_t)std::min<uint64_t>(group, resident);
        p.slots = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(slots, resident / p.group));
    }
    *plan = p;
    return FK_OK;
}

int launch_analyze(const AnalyzePlan& plan, uint32_t n_vars, uint32_t n_expr, const uint8_t* kinds, const uint32_t* slot_var,
                   uint32_t n_sketches, const double* vars, const double* params, uint8_t* out, double* ws, void* stream) {
    if (n_sketches == 0 || n_expr == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    AnArgs a{};
    a.n_vars = n_vars; a.n_expr = n_expr; a.nsteps = plan.nsteps; a.ld = plan.ld; a.group = plan.group; a.n_sketches = n_sketches;
    a.slot_doubles = plan.slot_doubles; a.kinds = kinds; a.slot_var = slot_var; a.vars_all = vars; a.params_all = params; a.out = out;
    a.ws = ws + kAnHeadDoubles;
    a.next = reinterpret_cast<unsigned*>(ws);
    const size_t smem = std::max<size_t>(8, (size_t)n_vars * sizeof(double));
    cudaError_t e = cudaFuncSetAttribute(fk_analyze_cta_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kAnMaxVars * sizeof(double)));
    if (e != cudaSuccess) return (int)e;
    if (plan.kernel == kAnCta) {
        e = cudaMemsetAsync(ws, 0, sizeof(unsigned), st);
        if (e != cudaSuccess) return (int)e;
        const uint32_t grid = std::min(n_sketches, plan.slots);
        fk_analyze_cta_kernel<<<grid, kAnThreads, smem, st>>>(a);
        return (int)cudaGetLastError();
    }
    void* args[] = {&a};
    e = cudaLaunchCooperativeKernel((const void*)fk_analyze_cta_kernel, dim3(plan.slots * plan.group), dim3(kAnThreads), args, smem, st);
    return (int)e;
}

}  // namespace fk
