// Batched Levenberg–Marquardt on sm_100a: K1 (residual + Jacobian into a precomputed pattern),
// K2 (residual only), K3 (H = JᵀJ + lambda I, g = Jᵀ(-r) through contribution lists, no atomics)
// and K4 (the whole LM loop with an LDLᵀ factorisation in shared memory) — SURVEY §2 "new
// kernels".  Control flow follows fiksi/src/solve/lm.rs:21-193 line by line (SURVEY App. A); the
// linear solve is the normal-equation form north_star asks for instead of the reference's sparse
// Householder QR of [J; sqrt(lambda) I] (solvi/src/decomposition/sparse/qr.rs:281-356).
//
// Compiled with -fmad=false: every a*b+c below is two roundings unless it is an explicit fma().
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>

#include "expressions.cuh"
#include "lbfgs_core.cuh"
#include "lm_kernels.cuh"
#include "lm_sketch.cuh"
#include "prepare.cuh"

namespace fk {

template <int TILE>
struct TileOps {
    static constexpr bool kWholeCta = TILE > 32;
    __device__ static __forceinline__ unsigned mask() {
        if constexpr (TILE >= 32) {
            return 0xFFFFFFFFu;
        } else {
            const unsigned lane_in_warp = threadIdx.x & 31u;
            return ((1u << TILE) - 1u) << (lane_in_warp & ~(unsigned)(TILE - 1));
        }
    }
    __device__ static __forceinline__ void sync(unsigned m) {
        if (kWholeCta) __syncthreads();
        else __syncwarp(m);
    }
};

// One expression row: gather the slot values (free ones from `xfree`, fixed ones from the
// sketch's `vars`, fiksi/src/variable_map.rs:57-72), evaluate, store the residual and scatter
// the gradient into the precomputed CSC slots (duplicates of a column inside a row are summed, as
// SparseColMat::from_triplet_mat does).  == one iteration of the loop at
// fiksi/src/subsystem.rs:143-165.  KIND >= 0: every row of the topology has this kind.
template <int KIND, bool WITH_JACOBIAN>
__device__ __forceinline__ void eval_row(const DevProgram& P, uint32_t row, const double* xfree,
                                         const double* __restrict__ vars, const double* __restrict__ params,
                                         double* rdst, double* jdst) {
    const uint32_t hdr = __ldg(P.row_hdr + row);
    if (hdr == kNop) return;
    const int kind = KIND >= 0 ? KIND : (int)(hdr & 0xFFu);
    const int a = dev::arity_of(kind);
    uint2 sl[8];
    double v[8], g[8];
#pragma unroll
    for (int s = 0; s < 8; s++) {
        v[s] = 0.0;
        sl[s] = make_uint2(kNop, kNop);
        if (s < a) {
            sl[s] = __ldg(P.row_slots + row * 8 + s);
            v[s] = (int32_t)sl[s].x >= 0 ? xfree[sl[s].x] : __ldg(vars + (sl[s].x & 0x7FFFFFFFu));
        }
    }
    const double param = __ldg(params + (hdr >> 8));
    rdst[row] = dev::eval_expression(kind, v, param, g);
    if (WITH_JACOBIAN) {
#pragma unroll
        for (int s = 0; s < 8; s++) {
            if (s < a && sl[s].y != kNop) {
                const uint32_t pos = sl[s].y & 0xFFFFFFu;
                if (sl[s].y & 0x40000000u) jdst[pos] += g[s];
                else jdst[pos] = g[s];
            }
        }
    }
}

// Sequential left-to-right sum of squares, as fiksi/src/solve/lm.rs:195-197 (every lane computes
// the same value, which keeps the LM control flow uniform across the tile without a broadcast).
__device__ __forceinline__ double sum_squares_seq(const double* v, uint32_t n) {
    double s = 0.0;
#pragma unroll 4
    for (uint32_t i = 0; i < n; i++) s += v[i] * v[i];
    return s;
}

// 1/d for a positive finite pivot: hardware seed + two Newton steps (relative error ~1e-16; the
// LDLt is not compared bit-wise with anything, it only has to be deterministic).
__device__ __forceinline__ double fast_rcp(double d) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    double e = fma(-d, r, 1.0);
    r = fma(r, e, r);
    e = fma(-d, r, 1.0);
    r = fma(r, e, r);
    return r;
}

constexpr uint32_t kFirst = 1u << 16, kLast = 1u << 17;

// K3: L storage := JᵀJ (permuted, lower; the damping is added when a pivot is read) and
// g = -Jᵀ r (permuted).  Each output entry is the sum of its precomputed contribution list in
// row order — a segmented reduction without atomics.  The lists are laid out as flat steps (one
// packed op per lane per step, longest lists first); step s+1 is prefetched while step s runs.
template <int TILE, bool NEGATE>
__device__ __forceinline__ void accumulate_steps(uint32_t nsteps, const uint32_t* __restrict__ flags,
                                                 const uint32_t* __restrict__ ops, const uint32_t* __restrict__ dsts,
                                                 int lane, const double* A, const double* B, double* out) {
    uint32_t fl = __ldg(flags), op = __ldg(ops + lane), dst = __ldg(dsts + lane);
    double acc = 0.0;
    for (uint32_t s = 0; s < nsteps; s++) {
        const uint32_t nfl = __ldg(flags + s + 1);
        const uint32_t nop = __ldg(ops + (s + 1) * TILE + lane);
        const uint32_t ndst = __ldg(dsts + (s + 1) * TILE + lane);
        if (fl & kFirst) acc = 0.0;
        if (op != kNop) acc = fma(A[op & 0xFFFFu], B[op >> 16], acc);
        if ((fl & kLast) && dst != kNop) out[dst] = NEGATE ? -acc : acc;
        fl = nfl; op = nop; dst = ndst;
    }
}

// LDLᵀ of (L + lam2 I) in place: column k keeps the unscaled entries (L D)(i,k) and 1/D(k) on
// its diagonal slot.  Right-looking; per step every lane applies at most one packed update.
// Returns 0 ok, 1 non-positive pivot, 2 NaN pivot.
template <int TILE>
__device__ __forceinline__ int factor_tile(const DevProgram& P, int lane, unsigned msk, double lam2, double* L) {
    uint32_t hdr = __ldg(P.f_steps);
    uint2 op = __ldg(P.f_ops + lane);
    uint32_t prev_dpos = 0;
    double inv = 0.0;
    bool have_prev = false;
    // First bad pivot in column order (kNop if none): its kind decides between "not solved" and NaN.
    // A bad pivot only poisons later columns, so checking after the fact finds the same first one.
    uint32_t bad_col = kNop;
    bool bad_nan = false;
    uint32_t col = 0;
    for (uint32_t s = 0; s < P.f_nsteps; s++) {
        const uint32_t nhdr = __ldg(P.f_steps + s + 1);
        const uint2 nop = __ldg(P.f_ops + (s + 1) * TILE + lane);
        if (hdr & kFirst) {
            const uint32_t dpos = hdr & 0xFFFFu;
            const double d = L[dpos] + lam2;
            // the previous pivot slot is free now (every lane passed the barrier that ended its column)
            if (have_prev && lane == 0) L[prev_dpos] = inv;
            if (!(d > 0.0 && d < INFINITY) && bad_col == kNop) {
                bad_col = col;
                bad_nan = d != d;
            }
            inv = fast_rcp(d);
            prev_dpos = dpos;
            have_prev = true;
            col++;
        }
        if (op.x != kNop) {
            const uint32_t dst = op.x & 0xFFFFu;
            L[dst] = fma(-(L[op.x >> 16] * inv), L[op.y], L[dst]);
        }
        if (TILE > 1 && (hdr & kLast)) TileOps<TILE>::sync(msk);
        hdr = nhdr; op = nop;
    }
    if (have_prev && lane == 0) L[prev_dpos] = inv;
    if (TILE > 1) TileOps<TILE>::sync(msk);
    return bad_col == kNop ? 0 : (bad_nan ? 2 : 1);
}

// Solve (L D Lᵀ) z = g.  w holds g on entry (permuted order); the solution is written in
// variable order (delta[perm[k]] = z[k], the P_c z of qr.rs:354) into `delta`.
template <int TILE>
__device__ __forceinline__ void solve_tile(const DevProgram& P, int lane, unsigned msk, const double* L,
                                           double* w, double* delta) {
    // (the forward substitution has already been applied to w by the factorisation steps)
    {   // backward: D Lᵀ z = y column by column over R = Lᵀ: z_k = y_k / d_k, then y_j -= (L D)(k,j) z_k
        uint2 hdr = __ldg(P.b_steps);
        uint32_t op = __ldg(P.b_ops + lane);
        double zk = 0.0;
        for (uint32_t s = 0; s < P.b_nsteps; s++) {
            const uint2 nhdr = __ldg(P.b_steps + s + 1);
            const uint32_t nop = __ldg(P.b_ops + (s + 1) * TILE + lane);
            if (hdr.x & kFirst) {
                zk = w[hdr.y & 0xFFFFu] * L[hdr.x & 0xFFFFu];
                if (lane == 0) delta[hdr.y >> 16] = zk;
            }
            if (op != kNop) {
                const uint32_t j = op & 0xFFFFu;
                w[j] = fma(-L[op >> 16], zk, w[j]);
            }
            if (TILE > 1 && (hdr.x & kLast)) TileOps<TILE>::sync(msk);
            hdr = nhdr; op = nop;
        }
    }
}

__device__ __forceinline__ uint64_t trace_push(uint64_t h, uint32_t code) { return h * 3ull + code + 1ull; }

// The whole LM solve of one sketch by one tile.  The reference's nested loops (outer <= 100,
// unbounded damping loop) are flattened into one loop over damping iterations with the outer
// bookkeeping done at accept time, so that sketches sharing a warp (TILE < 32) stay in step.
// The LM solve of ONE sketch by one tile: `x` = the tile's shared-memory block, vars / params / out / rep = the sketch's rows.
template <int TILE, int KIND>
__device__ __forceinline__ void lm_tile_solve(const DevProgram& P, int lane, unsigned msk, double* x, const double* __restrict__ vars,
                                              const double* __restrict__ params, double* __restrict__ out, fk_report* __restrict__ rep_out) {
    const uint32_t n = P.n, m = P.m;
    double* xs = x + n;
    double* g = xs + n;
    double* J = g + n;          // Jacobian values at the accepted point (CSC order)
    double* L = J + P.jnnz;     // LDLt factor; receives the trial Jacobian after the solve
    double* w = L + (P.lnnz > P.jnnz ? P.lnnz : P.jnnz);  // right-hand side / solve vector, addressed
    double* rs = w;                                        // as L[wbase + i] by the factor steps; the
                                                           // trial residuals live here outside the solve

    for (uint32_t i = lane; i < n; i += TILE) x[i] = __ldg(vars + __ldg(P.free_vars + i));
    if (TILE > 1) TileOps<TILE>::sync(msk);

    // lm.rs:80-106: initial residuals + Jacobian, ssr, g = J^T(-r)
    for (uint32_t rd = 0; rd < P.eval_rounds; rd++) eval_row<KIND, true>(P, rd * TILE + lane, x, vars, params, rs, J);
    if (TILE > 1) TileOps<TILE>::sync(msk);
    double ssr = sum_squares_seq(rs, m);
    accumulate_steps<TILE, true>(P.g_nsteps, P.g_flags, P.g_ops, P.g_dst, lane, J, rs, g);
    if (TILE > 1) TileOps<TILE>::sync(msk);

    double lambda = 0.5;  // lm.rs:108
    uint32_t exit_reason = FK_EXIT_MAX_OUTER, outer_iters = 0, factorizations = 0, accepted = 0;
    uint64_t trace = 0;
    bool active = true;
    if (ssr < 1e-8) {  // lm.rs:110-112 on the first outer iteration
        exit_reason = FK_EXIT_CONVERGED_RESIDUAL;
        active = false;
    } else {
        outer_iters = 1;
    }

    while (active) {  // one pass == one iteration of the damping loop, lm.rs:115-191
        if (!isfinite(lambda)) {
            exit_reason = FK_EXIT_LAMBDA_OVERFLOW;
            break;
        }
        // lm.rs:119-125: the damping entries are sqrt(lambda); their square lands on diag(H)
        const double sl = sqrt(lambda);
        const double lam2 = sl * sl;
        accumulate_steps<TILE, false>(P.a_nsteps, P.a_flags, P.a_ops, P.a_dst, lane, J, J, L);
        for (uint32_t k = lane; k < n; k += TILE) w[k] = g[k];
        if (TILE > 1) TileOps<TILE>::sync(msk);

        const int fstat = factor_tile<TILE>(P, lane, msk, lam2, L);  // replaces lm.rs:128
        factorizations++;
        if (fstat == 1) {  // lm.rs:134-137 (`!solved`)
            lambda *= 8.0;
            trace = trace_push(trace, 0);
            if (TILE > 1) TileOps<TILE>::sync(msk);
            continue;
        }
        double ssr_s = NAN;
        if (fstat == 0) {
            solve_tile<TILE>(P, lane, msk, L, w, xs);  // replaces lm.rs:130-132
            if (sum_squares_seq(xs, n) < 1e-12) {      // lm.rs:139-142
                exit_reason = FK_EXIT_SMALL_STEP;
                break;
            }
            if (TILE > 1) TileOps<TILE>::sync(msk);
            for (uint32_t i = lane; i < n; i += TILE) xs[i] = x[i] + xs[i];  // lm.rs:144-146
            if (TILE > 1) TileOps<TILE>::sync(msk);
            // lm.rs:148-149 (+ the Jacobian the accept branch would recompute at lm.rs:173-185)
            for (uint32_t rd = 0; rd < P.eval_rounds; rd++)
                eval_row<KIND, true>(P, rd * TILE + lane, xs, vars, params, rs, L);
            if (TILE > 1) TileOps<TILE>::sync(msk);
            ssr_s = sum_squares_seq(rs, m);
        }
        if (ssr_s < ssr) {  // lm.rs:151 (strict; NaN rejects)
            lambda *= 0.125;
            if (lambda < 1e-50) lambda = 1e-50;
            accepted++;
            trace = trace_push(trace, 1);
            for (uint32_t i = lane; i < n; i += TILE) x[i] = xs[i];
            const bool stalled = (ssr - ssr_s) / ssr <= 1e-6;  // lm.rs:164-168
            ssr = ssr_s;
            if (stalled) {
                exit_reason = FK_EXIT_STALLED;
                break;
            }
            for (uint32_t i = lane; i < P.jnnz; i += TILE) J[i] = L[i];
            if (TILE > 1) TileOps<TILE>::sync(msk);
            accumulate_steps<TILE, true>(P.g_nsteps, P.g_flags, P.g_ops, P.g_dst, lane, J, rs, g);
            if (TILE > 1) TileOps<TILE>::sync(msk);
            // next outer iteration, lm.rs:109-112
            if (outer_iters == 100) break;  // FK_EXIT_MAX_OUTER: the 100th outer iteration has ended
            if (ssr < 1e-8) {
                exit_reason = FK_EXIT_CONVERGED_RESIDUAL;
                break;
            }
            outer_iters++;
        } else {  // lm.rs:187-190
            lambda *= 2.0;
            trace = trace_push(trace, 2);
            if (TILE > 1) TileOps<TILE>::sync(msk);
        }
    }

    if (TILE > 1) TileOps<TILE>::sync(msk);
    for (uint32_t i = lane; i < n; i += TILE) out[i] = x[i];
    if (lane == 0) {
        fk_report rep;
        rep.exit_reason = exit_reason;
        rep.outer_iters = outer_iters;
        rep.factorizations = factorizations;
        rep.accepted = accepted;
        rep.ssr = ssr;
        rep.lambda = lambda;
        rep.trace_hash = trace;
        *rep_out = rep;
    }
}

// Uniform batch: every sketch shares the topology P (kernel parameter: constant bank).
template <int TILE, int KIND>
__global__ void __launch_bounds__(TILE > 128 ? TILE : 128)
fk_batch_lm_kernel(const DevProgram P, uint32_t n_sketches, uint32_t stride_doubles,
                   const double* __restrict__ vars_all, const double* __restrict__ params_all,
                   double* __restrict__ free_out, fk_report* __restrict__ reports) {
    extern __shared__ double smem[];
    const int tiles_per_cta = blockDim.x / TILE;
    const int tile_id = threadIdx.x / TILE;
    const int lane = threadIdx.x % TILE;
    const uint32_t sketch = blockIdx.x * tiles_per_cta + tile_id;
    if (sketch >= n_sketches) return;
    // per-sketch shared arrays; the stride is odd so that tiles of one warp touching the same
    // element index land in different banks
    lm_tile_solve<TILE, KIND>(P, lane, TileOps<TILE>::mask(), smem + (size_t)tile_id * stride_doubles, vars_all + (size_t)sketch * P.n_vars,
                              params_all + (size_t)sketch * P.n_expr, free_out + (size_t)sketch * P.n, reports + sketch);
}

// Heterogeneous batch: every system has its own topology.  One warp per system; the warp reads its job (program index and
// the offsets of its rows in the call's input / output buffers) and then runs the same LM solve with the program's tables
// (32-lane tables, in device memory).  One launch for any mix of small systems: the reference's unit of work is "each
// connected component" (fiksi/src/assemble/mod.rs:81), and a drawing is many different small components.
__global__ void __launch_bounds__(128)
fk_hetero_lm_kernel(const DevProgram* __restrict__ progs, const HeteroJob* __restrict__ jobs, uint32_t n_jobs, uint32_t stride_doubles,
                    const double* __restrict__ in, double* __restrict__ out, fk_report* __restrict__ reports) {
    extern __shared__ double smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t job = blockIdx.x * (blockDim.x >> 5) + warp;
    if (job >= n_jobs) return;
    const HeteroJob j = jobs[job];
    lm_tile_solve<32, -1>(progs[j.prog], lane, 0xFFFFFFFFu, smem + (size_t)warp * stride_doubles, in + j.vars_off, in + j.param_off,
                          out + j.out_off, reports + job);
}

int launch_hetero_lm(const DevProgram* d_progs, const HeteroJob* d_jobs, uint32_t n_jobs, uint32_t max_state_doubles, const double* d_in,
                     double* d_out, fk_report* d_reports, void* stream) {
    if (n_jobs == 0) return 0;
    const uint32_t stride = max_state_doubles | 1u;
    const size_t per_warp = (size_t)stride * sizeof(double);
    int warps = 4;
    while (warps > 1 && per_warp * warps > 100 * 1024) warps >>= 1;
    const size_t smem = per_warp * warps;
    if (smem > 220 * 1024) return (int)cudaErrorInvalidConfiguration;
    cudaError_t e = cudaFuncSetAttribute(fk_hetero_lm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    fk_hetero_lm_kernel<<<(n_jobs + warps - 1) / warps, 32 * warps, smem, (cudaStream_t)stream>>>(d_progs, d_jobs, n_jobs, stride, d_in, d_out, d_reports);
    return (int)cudaGetLastError();
}

// K1 / K2 on their own: one thread per (sketch, row), used for the assembly-bandwidth metric and
// for per-entry parity tests.  mode 0: residual + Jacobian, mode 1: residual only.
template <bool WITH_JACOBIAN>
__global__ void __launch_bounds__(256)
fk_batch_eval_kernel(const DevProgram P, uint32_t n_sketches, const double* __restrict__ vars_all,
                     const double* __restrict__ params_all, double* __restrict__ out_r, double* __restrict__ out_j) {
    const uint64_t total = (uint64_t)n_sketches * P.m;
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t sketch = (uint32_t)(t / P.m), row = (uint32_t)(t % P.m);
        const double* vars = vars_all + (size_t)sketch * P.n_vars;
        // no free-value overlay here: free variables are read from the sketch's vars as well
        const uint32_t hdr = __ldg(P.row_hdr + row);
        const int kind = (int)(hdr & 0xFFu);
        const int a = dev::arity_of(kind);
        uint2 sl[8];
        double v[8], g[8];
#pragma unroll
        for (int s = 0; s < 8; s++) {
            v[s] = 0.0;
            sl[s] = make_uint2(kNop, kNop);
            if (s < a) {
                sl[s] = __ldg(P.row_slots + row * 8 + s);
                const uint32_t var = (int32_t)sl[s].x >= 0 ? __ldg(P.free_vars + sl[s].x) : (sl[s].x & 0x7FFFFFFFu);
                v[s] = __ldg(vars + var);
            }
        }
        const double param = __ldg(params_all + (size_t)sketch * P.n_expr + (hdr >> 8));
        out_r[(size_t)sketch * P.m + row] = dev::eval_expression(kind, v, param, g);
        if (WITH_JACOBIAN) {
            double* jdst = out_j + (size_t)sketch * P.jnnz;
#pragma unroll
            for (int s = 0; s < 8; s++) {
                if (s < a && sl[s].y != kNop) {
                    const uint32_t pos = sl[s].y & 0xFFFFFFu;
                    if (sl[s].y & 0x40000000u) jdst[pos] += g[s];
                    else jdst[pos] = g[s];
                }
            }
        }
    }
}

// K1 / K2, tile-staged: a CTA owns S consecutive sketches at a time.  Their variables and
// parameters are one contiguous chunk of the caller's [sketch][var] arrays; the CTA reads the chunk
// with fully coalesced loads and transposes it on the fly into shared memory as [var][sketch]
// (row stride S+1 doubles: odd, so both the transposing writes and the per-sketch reads are
// bank-conflict free).  Work items are (row, sketch) pairs with the sketch index fastest, so a warp
// evaluates ONE row for 32 sketches: the slot table entries are warp-uniform broadcasts, there is
// no divergence between expression kinds, and every gather / scatter is a conflict-free shared
// memory access.  Residuals and Jacobian values are collected in shared memory ([pos][sketch]) and
// leave as contiguous, coalesced stores.  HBM sees each input and output byte exactly once.

// Row table decoded once per CTA into shared memory: all offsets are premultiplied by the tile's
// leading dimension, so the inner loop is `value = sv[voff + sketch]`.
struct alignas(16) EvalRow {
    uint32_t kind;      // bit 8: the row has a fixed or a duplicated slot (slow scatter path)
    uint32_t poff;      // parameter offset
    uint32_t pad0, pad1;
    uint32_t voff[8];   // variable offsets
    uint32_t joff[8];   // Jacobian offsets; kNop: no entry (fixed variable); bit 31: add (duplicate column)
};

template <int KIND, bool WITH_JACOBIAN, bool SPECIAL>
__device__ __forceinline__ void eval_tiled_row(const EvalRow& T, uint32_t sk, uint32_t roff, const double* sv,
                                               const double* sp, double* sr, double* sj) {
    constexpr int A = (int)((0x6678888566642ull >> (4 * KIND)) & 0xF);
    double v[8], g[8];
#pragma unroll
    for (int s = 0; s < 8; s++) v[s] = s < A ? sv[T.voff[s] + sk] : 0.0;
    sr[roff + sk] = dev::eval_expression(KIND, v, sp[T.poff + sk], g);
    if (WITH_JACOBIAN) {
#pragma unroll
        for (int s = 0; s < A; s++) {
            if (SPECIAL) {
                const uint32_t j = T.joff[s];
                if (j != kNop) {
                    const uint32_t pos = (j & 0x7FFFFFFFu) + sk;
                    if (j >> 31) sj[pos] += g[s];
                    else sj[pos] = g[s];
                }
            } else {
                sj[T.joff[s] + sk] = g[s];
            }
        }
    }
}

// 8-byte asynchronous copy global -> shared (no register staging: the copy is in flight while the thread computes)
__device__ __forceinline__ void eval_cp_async8(double* smem_dst, const double* gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gsrc) : "memory");
}

// PREFETCH: the inputs of a CTA's NEXT tile are copied into a second input buffer with cp.async while the current tile is
// evaluated and stored (ncu on the version without it: 27 % of the warp samples sit on the stores of the load phase waiting
// for their global loads, 9 % at the barriers between the phases).
template <int S, bool WITH_JACOBIAN, int kEvalThreads, bool PREFETCH = false>
__global__ void __launch_bounds__(kEvalThreads, 1024 / kEvalThreads)
fk_batch_eval_tiled_kernel(const DevProgram P, uint32_t n_sketches, const double* __restrict__ vars_all,
                           const double* __restrict__ params_all, double* __restrict__ out_r, double* __restrict__ out_j) {
    extern __shared__ __align__(16) double smem_eval[];
    double* smem = smem_eval;
    constexpr uint32_t LD = S + 1;
    const uint32_t nv = P.n_vars, ne = P.n_expr, m = P.m, jn = P.jnnz;
    const size_t in_doubles = (size_t)(nv + ne) * LD;
    double* sv = smem;                 // [nv][LD]
    double* sp = sv + (size_t)nv * LD;  // [ne][LD]   (PREFETCH: a second [nv + ne][LD] input buffer follows)
    double* sr = smem + (PREFETCH ? 2 : 1) * in_doubles;  // [m][LD]
    double* sj = sr + (size_t)m * LD;   // [jn][LD]
    EvalRow* tab = reinterpret_cast<EvalRow*>(sj + (WITH_JACOBIAN ? (size_t)jn * LD : 0) +
                                              (((PREFETCH ? 2 : 1) * (nv + ne) + m + (WITH_JACOBIAN ? jn : 0)) & 1u));
    const uint32_t tid = threadIdx.x;
    const uint32_t n_tiles = (n_sketches + S - 1) / S;

    for (uint32_t row = tid; row < m; row += kEvalThreads) {
        const uint32_t hdr = __ldg(P.row_hdr + row);
        const int kind = (int)(hdr & 0xFFu);
        const int a = dev::arity_of(kind);
        EvalRow t;
        bool special = false;
        for (int s = 0; s < 8; s++) {
            t.voff[s] = 0;
            t.joff[s] = kNop;
            if (s < a) {
                const uint2 sl = __ldg(P.row_slots + row * 8 + s);
                const uint32_t var = (int32_t)sl.x >= 0 ? __ldg(P.free_vars + sl.x) : (sl.x & 0x7FFFFFFFu);
                t.voff[s] = var * LD;
                if (sl.y == kNop) special = true;
                else {
                    t.joff[s] = (sl.y & 0xFFFFFFu) * LD;
                    if (sl.y & 0x40000000u) { t.joff[s] |= 0x80000000u; special = true; }
                }
            }
        }
        t.kind = (uint32_t)kind | (special ? 0x100u : 0u);
        t.poff = (hdr >> 8) * LD;
        t.pad0 = t.pad1 = 0;
        tab[row] = t;
    }

    // Flat element i of a [count][width] chunk lives at [i % width][i / width] of the transposed tile;
    // the division is a multiply-high by ceil(2^32 / width) (exact while i * width < 2^32, which the
    // launcher checks), so the loops carry no dependency and unroll four deep.
    auto transpose_in = [&](const double* __restrict__ src, double* dst, uint32_t width, uint32_t total) {
        if (width == 0) return;
        const uint32_t M = width == 1 ? 0u : 0xFFFFFFFFu / width + 1u;
        uint32_t i = tid;
        for (; i + 3 * kEvalThreads < total; i += 4 * kEvalThreads) {
            double v[4];
#pragma unroll
            for (int u = 0; u < 4; u++) v[u] = __ldcs(src + i + u * kEvalThreads);
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const uint32_t e = i + u * kEvalThreads, q = width == 1 ? e : __umulhi(e, M);
                dst[(e - q * width) * LD + q] = v[u];
            }
        }
        for (; i < total; i += kEvalThreads) {
            const uint32_t q = width == 1 ? i : __umulhi(i, M);
            dst[(i - q * width) * LD + q] = __ldcs(src + i);
        }
    };
    auto transpose_out = [&](const double* src, double* __restrict__ dst, uint32_t width, uint32_t total) {
        if (width == 0) return;
        const uint32_t M = width == 1 ? 0u : 0xFFFFFFFFu / width + 1u;
        uint32_t i = tid;
        for (; i + 3 * kEvalThreads < total; i += 4 * kEvalThreads) {
            double v[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const uint32_t e = i + u * kEvalThreads, q = width == 1 ? e : __umulhi(e, M);
                v[u] = src[(e - q * width) * LD + q];
            }
#pragma unroll
            for (int u = 0; u < 4; u++) __stcs(dst + i + u * kEvalThreads, v[u]);
        }
        for (; i < total; i += kEvalThreads) {
            const uint32_t q = width == 1 ? i : __umulhi(i, M);
            __stcs(dst + i, src[(i - q * width) * LD + q]);
        }
    };

    auto transpose_in_async = [&](const double* __restrict__ src, double* dst, uint32_t width, uint32_t total) {
        if (width == 0) return;
        const uint32_t M = width == 1 ? 0u : 0xFFFFFFFFu / width + 1u;
        for (uint32_t i = tid; i < total; i += kEvalThreads) {
            const uint32_t q = width == 1 ? i : __umulhi(i, M);
            eval_cp_async8(dst + (i - q * width) * LD + q, src + i);
        }
    };
    auto prefetch = [&](uint32_t tile, uint32_t buf) {
        const uint32_t first = tile * S;
        const uint32_t count = min((uint32_t)S, n_sketches - first);
        transpose_in_async(vars_all + (size_t)first * nv, smem + buf * in_doubles, nv, count * nv);
        transpose_in_async(params_all + (size_t)first * ne, smem + buf * in_doubles + (size_t)nv * LD, ne, count * ne);
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    if (PREFETCH && blockIdx.x < n_tiles) prefetch(blockIdx.x, 0);
    uint32_t it = 0;
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, it++) {
        const uint32_t first = tile * S;
        const uint32_t count = min((uint32_t)S, n_sketches - first);
        if (PREFETCH) {
            const uint32_t b = it & 1u;
            if (tile + gridDim.x < n_tiles) {  // the other buffer's readers finished before the barrier that ended the last tile
                prefetch(tile + gridDim.x, b ^ 1u);
                asm volatile("cp.async.wait_group 1;" ::: "memory");
            } else {
                asm volatile("cp.async.wait_group 0;" ::: "memory");
            }
            sv = smem + b * in_doubles;
            sp = sv + (size_t)nv * LD;
        } else {
            transpose_in(vars_all + (size_t)first * nv, sv, nv, count * nv);
            transpose_in(params_all + (size_t)first * ne, sp, ne, count * ne);
        }
        __syncthreads();
        for (uint32_t item = tid; item < m * S; item += kEvalThreads) {
            const uint32_t row = item / S, sk = item % S;  // S is a power of two >= 32: row is warp-uniform
            if (sk >= count) continue;
            const EvalRow& T = tab[row];
            const uint32_t roff = row * LD;
#define FK_ROW(K)                                                                                   \
    case K:                                                                                         \
        eval_tiled_row<K, WITH_JACOBIAN, false>(T, sk, roff, sv, sp, sr, sj);                       \
        break;                                                                                      \
    case 0x100 | K:                                                                                 \
        eval_tiled_row<K, WITH_JACOBIAN, true>(T, sk, roff, sv, sp, sr, sj);                        \
        break;
            switch (T.kind) {
                FK_ROW(0) FK_ROW(1) FK_ROW(2) FK_ROW(3) FK_ROW(4) FK_ROW(5)
                FK_ROW(6) FK_ROW(7) FK_ROW(8) FK_ROW(9) FK_ROW(10) FK_ROW(11) FK_ROW(12)
                default: break;
            }
#undef FK_ROW
        }
        __syncthreads();
        transpose_out(sr, out_r + (size_t)first * m, m, count * m);
        if (WITH_JACOBIAN) transpose_out(sj, out_j + (size_t)first * jn, jn, count * jn);
        // (no barrier here: the next tile's evaluation only starts behind the barrier that follows its inputs, which every
        // thread reaches after these stores; the inputs read by this tile's evaluation were released by the barrier above)
    }
}

// System::analyze on a batch (SURVEY 8f-2): per sketch the dense Jacobian over ALL variables
// (find_overconstraints, fiksi/src/analyze/numerical/mod.rs:123-147; gradient entries are ASSIGNED
// per slot, expressions.rs:1003-1007) followed by the row-by-row Gauss-Jordan elimination with
// tracked column swaps (incremental_gauss_jordan_elimination, :33-117).  One warp per sketch, the
// matrix in shared memory, lanes across the columns; every floating-point operation is the
// reference's (multiply, then subtract; one IEEE reciprocal per pivot row), so the flags are
// bit-for-bit those of the CPU restatement.  out[sketch][row] = 1 iff the row increased the rank.
// The body of both analyze warp kernels, so that their flags agree by construction: sketch `sketch` of the rows vars_all / params_all
// (n_vars / n_expr per sketch) in the warp's slice of smem_an, its flags to out[sketch][n_expr].  The parameters keep the uniform
// kernel's own names and arithmetic: taking pre-offset row pointers instead changes fk_batch_analyze_kernel's SASS.
__device__ __forceinline__ void analyze_warp(uint32_t n_vars, uint32_t n_expr, const uint8_t* __restrict__ kinds,
                                             const uint32_t* __restrict__ slot_var, uint32_t sketch, const double* __restrict__ vars_all,
                                             const double* __restrict__ params_all, uint8_t* __restrict__ out, double* smem_an,
                                             uint32_t warp_doubles, uint32_t warp, uint32_t lane) {
    const uint32_t m = n_expr, n = n_vars;
    double* M = smem_an + (size_t)warp * warp_doubles;
    uint32_t* ci = reinterpret_cast<uint32_t*>(M + (size_t)m * n);
    uint32_t* inc = ci + n;
    const double* vars = vars_all + (size_t)sketch * n_vars;
    const double* params = params_all + (size_t)sketch * n_expr;
    for (uint32_t e = lane; e < m * n; e += 32) M[e] = 0.0;
    for (uint32_t k = lane; k < n; k += 32) ci[k] = k;
    for (uint32_t r = lane; r < m; r += 32) inc[r] = 0;
    __syncwarp();
    for (uint32_t row = lane; row < m; row += 32) {
        const int kind = (int)__ldg(kinds + row);
        const int a = dev::arity_of(kind);
        double v[8], g[8];
        uint32_t var[8];
#pragma unroll
        for (int sl = 0; sl < 8; sl++) {
            var[sl] = sl < a ? __ldg(slot_var + row * 8 + sl) : 0u;
            v[sl] = sl < a ? __ldg(vars + var[sl]) : 0.0;
        }
        dev::eval_expression(kind, v, __ldg(params + row), g);
#pragma unroll
        for (int sl = 0; sl < 8; sl++)
            if (sl < a) M[(size_t)row * n + var[sl]] = g[sl];
    }
    __syncwarp();
    uint32_t current_col = 0;
    const uint32_t nsteps = m < n ? m : n;
    for (uint32_t row = 0; row < nsteps; row++) {
        double* Mr = M + (size_t)row * n;
        uint32_t rank = 0;
        for (uint32_t row_idx = 0; row_idx < row; row_idx++) {
            const double factor = Mr[ci[rank]];
            __syncwarp();
            const double* Mi = M + (size_t)row_idx * n;
            for (uint32_t col = lane; col < n; col += 32) Mr[col] -= factor * Mi[col];
            __syncwarp();
            if (inc[row_idx]) rank++;
        }
        uint32_t found = 0xFFFFFFFFu;
        for (uint32_t base = current_col; base < n; base += 32) {
            const uint32_t idx = base + lane;
            const bool ok = idx < n && fabs(Mr[ci[idx]]) > 1e-8;
            const unsigned b = __ballot_sync(0xFFFFFFFFu, ok);
            if (b) {
                found = base + (uint32_t)__ffs(b) - 1u;
                break;
            }
        }
        if (found == 0xFFFFFFFFu) continue;
        if (lane == 0) {
            const uint32_t tmp = ci[current_col];
            ci[current_col] = ci[found];
            ci[found] = tmp;
        }
        __syncwarp();
        const uint32_t column_idx = ci[current_col];
        const double inv = 1.0 / Mr[column_idx];
        __syncwarp();
        for (uint32_t col = lane; col < n; col += 32) Mr[col] *= inv;
        __syncwarp();
        for (uint32_t row_idx = 0; row_idx < row; row_idx++) {
            double* Mi = M + (size_t)row_idx * n;
            const double f2 = Mi[column_idx];
            __syncwarp();
            for (uint32_t col = lane; col < n; col += 32) Mi[col] -= f2 * Mr[col];
            __syncwarp();
        }
        current_col++;
        if (lane == 0) inc[row] = 1;
        __syncwarp();
    }
    for (uint32_t r = lane; r < m; r += 32) out[(size_t)sketch * m + r] = (uint8_t)inc[r];
}

constexpr int kAnalyzeWarps = 4;
__global__ void __launch_bounds__(kAnalyzeWarps * 32)
fk_batch_analyze_kernel(uint32_t n_vars, uint32_t n_expr, const uint8_t* __restrict__ kinds, const uint32_t* __restrict__ slot_var,
                        uint32_t n_sketches, const double* __restrict__ vars_all, const double* __restrict__ params_all,
                        uint8_t* __restrict__ out, uint32_t warp_doubles, uint32_t warps_per_cta) {
    extern __shared__ __align__(16) double smem_an[];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t sketch = blockIdx.x * warps_per_cta + warp;
    if (warp >= warps_per_cta || sketch >= n_sketches) return;
    analyze_warp(n_vars, n_expr, kinds, slot_var, sketch, vars_all, params_all, out, smem_an, warp_doubles, warp, lane);
}

// fk_systems_analyze: one warp per job, every job its own drawing (sizes, tables, rows); one footprint class per launch.
__global__ void __launch_bounds__(kAnalyzeWarps * 32)
fk_systems_analyze_kernel(const SysAnJob* __restrict__ jobs, uint32_t n_jobs, const uint32_t* __restrict__ tabs,
                          const double* __restrict__ vars, const double* __restrict__ params, uint8_t* __restrict__ flags,
                          uint32_t warp_doubles, uint32_t warps_per_cta) {
    extern __shared__ __align__(16) double smem_an[];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t j = blockIdx.x * warps_per_cta + warp;
    if (warp >= warps_per_cta || j >= n_jobs) return;
    const SysAnJob J = jobs[j];
    const uint32_t* slot_var = tabs + J.tab;
    analyze_warp(J.n_vars, J.n_expr, sys_an_kinds(slot_var, J.n_expr), slot_var, 0, vars + J.vars, params + J.exprs, flags + J.exprs,
                 smem_an, warp_doubles, warp, lane);
}

size_t batch_analyze_warp_bytes(uint32_t n_vars, uint32_t n_expr) {
    return (((size_t)n_expr * n_vars * sizeof(double) + ((size_t)n_vars + n_expr) * sizeof(uint32_t)) + 15) & ~(size_t)15;
}
bool batch_analyze_warp_fits(uint32_t n_vars, uint32_t n_expr) { return batch_analyze_warp_bytes(n_vars, n_expr) <= 200 * 1024; }

int launch_batch_analyze(uint32_t n_vars, uint32_t n_expr, const uint8_t* kinds, const uint32_t* slot_var, uint32_t n_sketches,
                         const double* vars, const double* params, uint8_t* out, void* stream) {
    if (n_sketches == 0 || n_expr == 0) return 0;
    if (!batch_analyze_warp_fits(n_vars, n_expr)) return (int)cudaErrorInvalidConfiguration;
    const size_t per_warp = batch_analyze_warp_bytes(n_vars, n_expr);
    const uint32_t wpc = (uint32_t)std::max<size_t>(1, std::min<size_t>(kAnalyzeWarps, (200 * 1024) / per_warp));
    const size_t smem = per_warp * wpc;
    cudaError_t e = cudaFuncSetAttribute(fk_batch_analyze_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const uint32_t grid = (n_sketches + wpc - 1) / wpc;
    fk_batch_analyze_kernel<<<grid, kAnalyzeWarps * 32, smem, (cudaStream_t)stream>>>(n_vars, n_expr, kinds, slot_var, n_sketches, vars, params, out,
                                                                                       (uint32_t)(per_warp / sizeof(double)), wpc);
    return (int)cudaGetLastError();
}

int launch_systems_analyze(const SysAnJob* jobs, uint32_t n_jobs, size_t warp_bytes, const uint32_t* tabs, const double* vars,
                           const double* params, uint8_t* flags, void* stream) {
    if (n_jobs == 0) return 0;
    if (warp_bytes > 200 * 1024 || warp_bytes % 16) return (int)cudaErrorInvalidConfiguration;
    const uint32_t wpc = (uint32_t)std::max<size_t>(1, std::min<size_t>(kAnalyzeWarps, (200 * 1024) / warp_bytes));
    const size_t smem = warp_bytes * wpc;
    cudaError_t e = cudaFuncSetAttribute(fk_systems_analyze_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    fk_systems_analyze_kernel<<<(n_jobs + wpc - 1) / wpc, kAnalyzeWarps * 32, smem, (cudaStream_t)stream>>>(
        jobs, n_jobs, tabs, vars, params, flags, (uint32_t)(warp_bytes / sizeof(double)), wpc);
    return (int)cudaGetLastError();
}

// ---- L-BFGS (SURVEY 8f-3): fiksi/src/solve/lbfgs.rs on one tile per sketch -------------------------------
// Same tile layout as the LM kernel (TILE lanes per sketch, state in shared memory); the control flow is
// lbfgs_solve (lbfgs_core.cuh).  Every lane computes each sequential sum itself, which keeps the control flow
// uniform across the tile without a broadcast.
__device__ __forceinline__ double dot_seq(const double* a, const double* b, uint32_t n) {
    double s = 0.0;
#pragma unroll 4
    for (uint32_t i = 0; i < n; i++) s += a[i] * b[i];
    return s;
}

template <int TILE, int KIND>
struct TileLbfgsOps {
    const DevProgram& P;
    const LbfgsTables& T;
    const double* vars;
    const double* params;
    int lane;
    unsigned msk;
    __device__ void sync() const { if (TILE > 1) TileOps<TILE>::sync(msk); }
    __device__ bool leader() const { return lane == 0; }
    template <class F>
    __device__ void each(uint32_t cnt, F f) const {
        for (uint32_t i = lane; i < cnt; i += TILE) f(i);
    }
    __device__ double dot(const double* a, const double* b, uint32_t k) const { return dot_seq(a, b, k); }
    __device__ void dot2(const double* a1, const double* b1, uint32_t k1, const double* a2, const double* b2, uint32_t k2, double* o1,
                         double* o2) const {
        *o1 = dot_seq(a1, b1, k1);
        *o2 = dot_seq(a2, b2, k2);
    }
    // residuals + Jacobian + gradient at `pt` (== Eval::calculate_phi without the phi / dphi sums)
    __device__ void evaluate(const double* pt, const LbfgsVecs& s) const {
        for (uint32_t rd = 0; rd < P.eval_rounds; rd++) eval_row_assign<KIND>(P, rd * TILE + lane, pt, vars, params, s.r, s.J);
        sync();
        for (uint32_t c = lane; c < P.n; c += TILE) s.g[c] = lbfgs_grad_col(T, s.J, s.r, c);
        sync();
    }
};

template <int TILE, int KIND>
__global__ void __launch_bounds__(128)
fk_batch_lbfgs_kernel(const DevProgram P, const LbfgsTables T, uint32_t n_sketches, uint32_t stride_doubles,
                      const double* __restrict__ vars_all, const double* __restrict__ params_all, double* __restrict__ free_out,
                      fk_report* __restrict__ reports) {
    extern __shared__ double smem[];
    const int tiles_per_cta = blockDim.x / TILE;
    const int tile_id = threadIdx.x / TILE;
    const int lane = threadIdx.x % TILE;
    const uint32_t sketch = blockIdx.x * tiles_per_cta + tile_id;
    if (sketch >= n_sketches) return;
    const uint32_t n = P.n, m = P.m;
    LbfgsVecs s;
    s.x = smem + (size_t)tile_id * stride_doubles;
    s.xs = s.x + n;
    s.g = s.xs + n;
    s.dir = s.g + n;
    s.sh = s.dir + n;        // [5][n]
    s.yh = s.sh + 5 * n;     // [5][n]
    s.r = s.yh + 5 * n;      // [m]
    s.J = s.r + m;           // [jnnz]
    s.rho = s.J + P.jnnz;    // [5]
    s.alpha = s.rho + 5;     // [5]
    const double* vars = vars_all + (size_t)sketch * P.n_vars;
    TileLbfgsOps<TILE, KIND> ops{P, T, vars, params_all + (size_t)sketch * P.n_expr, lane, TileOps<TILE>::mask()};
    lbfgs_solve(ops, P, vars, s, free_out + (size_t)sketch * n, reports + sketch);
}

// Shared memory of one CTA of the tile kernel, and how many sketches it holds; 0 when the topology does not take the
// tile kernel (lanes other than 4 / 8 / 16 / 32, or the state of a warp's sketches above 220 KiB).
static size_t lbfgs_tile_smem(uint32_t n, uint32_t m, uint32_t jnnz, uint32_t tile, int* tiles_per_cta) {
    if (tile != 4 && tile != 8 && tile != 16 && tile != 32) return 0;
    const uint32_t stride = lbfgs_smem_doubles(n, m, jnnz) | 1u;
    const size_t bytes_per_sketch = (size_t)stride * sizeof(double);
    const int tiles_per_warp = 32 / (int)tile;
    int warps = 4;
    while (warps > 1 && bytes_per_sketch * tiles_per_warp * warps > 72 * 1024) warps >>= 1;
    *tiles_per_cta = tiles_per_warp * warps;
    const size_t smem = bytes_per_sketch * *tiles_per_cta;
    return smem > 220 * 1024 ? 0 : smem;
}

bool batch_lbfgs_tile_fits(uint32_t n, uint32_t m, uint32_t jnnz, uint32_t tile) {
    int tiles_per_cta = 0;
    return lbfgs_tile_smem(n, m, jnnz, tile, &tiles_per_cta) != 0;
}

template <int TILE, int KIND>
static int launch_lbfgs_t(const DevProgram& prog, const LbfgsTables& T, uint32_t n_sketches, const double* vars, const double* params,
                          double* free_out, fk_report* reports, cudaStream_t stream) {
    int tiles_per_cta = 0;
    const size_t smem = lbfgs_tile_smem(prog.n, prog.m, prog.jnnz, TILE, &tiles_per_cta);
    if (smem == 0) return (int)cudaErrorInvalidConfiguration;
    const uint32_t stride = lbfgs_smem_doubles(prog.n, prog.m, prog.jnnz) | 1u;
    cudaError_t e = cudaFuncSetAttribute(fk_batch_lbfgs_kernel<TILE, KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const uint32_t grid = (n_sketches + tiles_per_cta - 1) / tiles_per_cta;
    fk_batch_lbfgs_kernel<TILE, KIND><<<grid, TILE * tiles_per_cta, smem, stream>>>(prog, T, n_sketches, stride, vars, params, free_out, reports);
    return (int)cudaGetLastError();
}

int launch_batch_lbfgs(const DevProgram& prog, const uint32_t* d_jcolptr, const uint32_t* d_jrow, uint32_t n_sketches, const double* vars,
                       const double* params, double* free_out, fk_report* reports, void* stream) {
    if (n_sketches == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    LbfgsTables T{d_jcolptr, d_jrow};
#define FK_LBFGS(TL)                                                                                          \
    case TL:                                                                                                  \
        return prog.uniform_kind == 1 ? launch_lbfgs_t<TL, 1>(prog, T, n_sketches, vars, params, free_out, reports, s) \
                                      : launch_lbfgs_t<TL, -1>(prog, T, n_sketches, vars, params, free_out, reports, s);
    switch (prog.tile) {
        FK_LBFGS(4) FK_LBFGS(8) FK_LBFGS(16) FK_LBFGS(32)
        default: return (int)cudaErrorInvalidConfiguration;
    }
#undef FK_LBFGS
}

const char* lm_kernel_name() { return "fk_batch_lm_kernel"; }

// FP64 roofline denominator: 8 independent DFMA chains per thread, enough warps to fill every SMSP.
__global__ void __launch_bounds__(256) fk_fp64_peak_kernel(double* out, int iters, double a, double b) {
    double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; i++) {
        x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
        x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}

int measure_fp64_peak(double* tflops) {
    const int blocks = 148 * 8, threads = 256, iters = 1 << 14;
    double* d = nullptr;
    cudaError_t e = cudaMalloc(&d, sizeof(double) * blocks * threads);
    if (e != cudaSuccess) return (int)e;
    cudaEvent_t t0, t1;
    cudaEventCreate(&t0);
    cudaEventCreate(&t1);
    float best = 1e30f;
    for (int rep = 0; rep < 5; rep++) {
        cudaEventRecord(t0);
        fk_fp64_peak_kernel<<<blocks, threads>>>(d, iters, 0.999999, 1e-9);
        cudaEventRecord(t1);
        e = cudaEventSynchronize(t1);
        if (e != cudaSuccess) break;
        float ms = 0;
        cudaEventElapsedTime(&ms, t0, t1);
        if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(t0);
    cudaEventDestroy(t1);
    cudaFree(d);
    if (e != cudaSuccess) return (int)e;
    *tflops = 2.0 * 8.0 * (double)iters * blocks * threads / (best * 1e-3) / 1e12;
    return 0;
}

template <int TILE, int KIND>
static int launch_lm_t(const DevProgram& prog, uint32_t n_sketches, const double* vars, const double* params,
                       double* free_out, fk_report* reports, cudaStream_t stream) {
    const uint32_t stride = lm_smem_doubles(prog.n, prog.m, prog.jnnz, prog.lnnz) | 1u;  // odd: see kernel
    const size_t bytes_per_sketch = (size_t)stride * sizeof(double);
    int tiles_per_cta;
    if (TILE > 32) {
        tiles_per_cta = 1;
    } else {
        // whole warps; as many as fit in ~1/3 of an SM's shared memory, at most 4 warps
        const int tiles_per_warp = 32 / TILE;
        int warps = 4;
        while (warps > 1 && bytes_per_sketch * tiles_per_warp * warps > 72 * 1024) warps >>= 1;
        if (const char* e = std::getenv("FK_LM_WARPS")) {  // tuning knob: warps per CTA (1..4)
            const int v = std::atoi(e);
            if (v >= 1 && v <= 4) warps = v;
        }
        tiles_per_cta = tiles_per_warp * warps;
        if (bytes_per_sketch * tiles_per_cta > 220 * 1024) return (int)cudaErrorInvalidConfiguration;
    }
    const size_t smem = bytes_per_sketch * tiles_per_cta;
    cudaError_t e = cudaFuncSetAttribute(fk_batch_lm_kernel<TILE, KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const uint32_t grid = (n_sketches + tiles_per_cta - 1) / tiles_per_cta;
    fk_batch_lm_kernel<TILE, KIND><<<grid, TILE * tiles_per_cta, smem, stream>>>(prog, n_sketches, stride, vars, params, free_out, reports);
    return (int)cudaGetLastError();
}

template <int TILE>
static int launch_lm_k(const DevProgram& prog, uint32_t n_sketches, const double* vars, const double* params,
                       double* free_out, fk_report* reports, cudaStream_t s) {
    if (prog.uniform_kind == 1) return launch_lm_t<TILE, 1>(prog, n_sketches, vars, params, free_out, reports, s);
    return launch_lm_t<TILE, -1>(prog, n_sketches, vars, params, free_out, reports, s);
}

std::atomic<int>& lm_kernel_choice() {
    static std::atomic<int> choice{[] {
        const char* e = std::getenv("FK_LM_KERNEL");
        if (!e) return -1;
        return e[0] == 's' ? 1 : (e[0] == 't' ? 0 : -1);
    }()};
    return choice;
}

// The sketch-per-thread kernel runs one warp per 32 sketches: it needs a batch that fills the machine.  Below
// that the tile kernel (4-32 lanes per sketch) has more parallelism to offer.  FK_LM_KERNEL=tile|sketch forces one.
int batch_lm_uses_sketch_kernel(const DevProgram& prog, uint32_t n_sketches) {
    if (!prog.sketch_prog) return 0;
    const int forced = lm_kernel_choice().load(std::memory_order_relaxed);
    if (forced >= 0) return forced >= 1 ? 1 : 0;
    static const uint32_t min_batch = [] {
        const char* e = std::getenv("FK_LM_SKETCH_MIN");
        // measured (tools/lm_ab_small.py): the sketch kernel is ahead of the tile kernel from 256 sketches up on every topology
        // tried, also in latency per batch (20-point truss, 256 sketches: 143 vs 165 us); below a warp's worth of sketches the
        // tile kernel's lanes-per-sketch parallelism wins
        return (uint32_t)(e ? std::max(1, std::atoi(e)) : 64);
    }();
    return n_sketches >= min_batch ? 1 : 0;
}

int launch_batch_lm(const DevProgram& prog, uint32_t n_sketches, const double* vars, const double* params,
                    double* free_out, fk_report* reports, void* stream) {
    if (n_sketches == 0) return 0;
    if (batch_lm_uses_sketch_kernel(prog, n_sketches))
        return launch_batch_lm_sketch(*prog.sketch_prog, n_sketches, vars, params, free_out, reports, stream);
    cudaStream_t s = (cudaStream_t)stream;
    switch (prog.tile) {
        case 1: return launch_lm_k<1>(prog, n_sketches, vars, params, free_out, reports, s);
        case 2: return launch_lm_k<2>(prog, n_sketches, vars, params, free_out, reports, s);
        case 4: return launch_lm_k<4>(prog, n_sketches, vars, params, free_out, reports, s);
        case 8: return launch_lm_k<8>(prog, n_sketches, vars, params, free_out, reports, s);
        case 16: return launch_lm_k<16>(prog, n_sketches, vars, params, free_out, reports, s);
        case 32: return launch_lm_k<32>(prog, n_sketches, vars, params, free_out, reports, s);
        case 256: return launch_lm_k<256>(prog, n_sketches, vars, params, free_out, reports, s);
        default: return (int)cudaErrorInvalidValue;
    }
}

__global__ void fk_scatter_free_kernel(const uint32_t* __restrict__ free_vars, uint32_t n_free, uint32_t n_vars, uint64_t total,
                                       const double* __restrict__ free_out, double* __restrict__ vars) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t k = i / n_free;
        const uint32_t f = (uint32_t)(i - k * n_free);
        vars[k * n_vars + free_vars[f]] = free_out[i];
    }
}

int launch_scatter_free(const uint32_t* d_free_vars, uint32_t n_free, uint32_t n_vars, uint32_t n_sketches, const double* free_out,
                        double* vars, void* stream) {
    const uint64_t total = (uint64_t)n_sketches * n_free;
    if (total == 0) return 0;
    const uint32_t grid = (uint32_t)std::min<uint64_t>((total + 255) / 256, 148u * 8u);
    fk_scatter_free_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_free_vars, n_free, n_vars, total, free_out, vars);
    return (int)cudaGetLastError();
}

__global__ void fk_transpose_reports_kernel(const uint64_t* __restrict__ in, uint64_t* __restrict__ out, uint32_t n, uint32_t steps) {
    constexpr uint32_t W = sizeof(fk_report) / 8;
    const uint64_t total = (uint64_t)n * steps * W;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t w = (uint32_t)(i % W);
        const uint64_t ks = i / W;  // k * steps + st
        const uint64_t k = ks / steps;
        const uint32_t st = (uint32_t)(ks - k * steps);
        out[i] = in[((uint64_t)st * n + k) * W + w];
    }
}

int launch_transpose_reports(const fk_report* in, fk_report* out, uint32_t n_sketches, uint32_t steps, void* stream) {
    static_assert(sizeof(fk_report) % 8 == 0, "fk_report is moved as 64-bit words");
    const uint64_t total = (uint64_t)n_sketches * steps * (sizeof(fk_report) / 8);
    if (total == 0) return 0;
    const uint32_t grid = (uint32_t)std::min<uint64_t>((total + 255) / 256, 148u * 16u);
    fk_transpose_reports_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const uint64_t*)in, (uint64_t*)out, n_sketches, steps);
    return (int)cudaGetLastError();
}

// ---- assemble::solve's pre- and post-processing on the device (SURVEY a19) -------------------------------------
// One thread per sketch, every sum in the reference's order (fiksi/src/utils.rs:12-19 via assemble/mod.rs:32-44:
// all variables left to right, then the distance parameters in expression order), one IEEE reciprocal, then
// variables * recip, recip * distance (expressions.rs:195-211) and the seeded perturbation of the listed variables
// (assemble/mod.rs:113-124; the generator is re-seeded per solve, so all sketches share one vector of draws).
// Bit-identical to fiksi_b200.workloads.Workload.prepare / fk_system_solve's host loop (no FMA contraction here).
__global__ void __launch_bounds__(32)
fk_batch_prepare_kernel(uint32_t n_sketches, uint32_t n_vars, uint32_t n_expr, const uint8_t* __restrict__ kinds, uint32_t shared_param,
                        uint32_t n_perturb, const uint32_t* __restrict__ perturb_vars, const double* __restrict__ draws,
                        const double* __restrict__ raw_vars, const double* __restrict__ raw_param, double* __restrict__ vars,
                        double* __restrict__ params, double* __restrict__ scales) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_sketches) return;
    const double* rv = raw_vars + (size_t)k * n_vars;
    const double* rp = raw_param + (shared_param ? 0 : (size_t)k * n_expr);
    const double scale = prepare_scale(rv, n_vars, n_expr, kinds, [&](uint32_t e) { return __ldg(rp + e); });
    const double recip = 1.0 / scale;
    double* ov = vars + (size_t)k * n_vars;
    double* op = params + (size_t)k * n_expr;
    // the perturbation list is ascending (a BTreeSet in the reference): one merge walk, every value is written once
    uint32_t j = 0, next = n_perturb ? __ldg(perturb_vars) : 0xFFFFFFFFu;
    for (uint32_t i = 0; i < n_vars; i++) {
        double col = __ldg(rv + i) * recip;
        if (i == next) {
            col = prepare_perturb(col, __ldg(draws + 2 * j), __ldg(draws + 2 * j + 1));
            j++;
            next = j < n_perturb ? __ldg(perturb_vars + j) : 0xFFFFFFFFu;
        }
        ov[i] = col;
    }
    for (uint32_t e = 0; e < n_expr; e++) {
        const double q = __ldg(rp + e);
        op[e] = prepare_is_distance(__ldg(kinds + e)) ? recip * q : q;
    }
    scales[k] = scale;
}

// system.variables[var] = system_scale * x[k] (assemble/mod.rs:161-166), in place on the solved free values.
__global__ void __launch_bounds__(256)
fk_batch_unscale_kernel(uint32_t n_sketches, uint32_t n_free, const double* __restrict__ scales, double* __restrict__ free_values) {
    const uint64_t total = (uint64_t)n_sketches * n_free;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x)
        free_values[i] = __ldg(scales + i / n_free) * free_values[i];
}

int launch_batch_prepare(uint32_t n_sketches, uint32_t n_vars, uint32_t n_expr, const uint8_t* kinds, int shared_param, uint32_t n_perturb,
                         const uint32_t* perturb_vars, const double* draws, const double* raw_vars, const double* raw_param, double* vars,
                         double* params, double* scales, void* stream) {
    if (n_sketches == 0) return 0;
    // one warp per CTA: a chunk of a few thousand sketches still spreads over every SM, and each thread's dependent chain
    // (the sequential sums) is short against the launch
    fk_batch_prepare_kernel<<<(n_sketches + 31) / 32, 32, 0, (cudaStream_t)stream>>>(n_sketches, n_vars, n_expr, kinds, shared_param ? 1u : 0u, n_perturb,
                                                                                        perturb_vars, draws, raw_vars, raw_param, vars, params, scales);
    return (int)cudaGetLastError();
}

int launch_batch_unscale(uint32_t n_sketches, uint32_t n_free, const double* scales, double* free_values, void* stream) {
    const uint64_t total = (uint64_t)n_sketches * n_free;
    if (total == 0) return 0;
    const uint32_t grid = (uint32_t)std::min<uint64_t>((total + 255) / 256, 148u * 16u);
    fk_batch_unscale_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(n_sketches, n_free, scales, free_values);
    return (int)cudaGetLastError();
}

int launch_batch_eval(const DevProgram& prog, uint32_t n_sketches, const double* vars, const double* params,
                      double* out_r, double* out_j, int mode, void* stream) {
    if (n_sketches == 0 || prog.m == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    // tile-staged kernel whenever S >= 32 sketches fit in shared memory with >= 2 CTAs per SM
    {
        const size_t per_sketch_rows = (size_t)prog.n_vars + prog.n_expr + prog.m + (mode == 0 ? prog.jnnz : 0);
        auto bytes_for = [&](int S) { return (per_sketch_rows * (size_t)(S + 1) + 1) * sizeof(double) + (size_t)prog.m * sizeof(EvalRow); };
        // 256-thread CTAs, largest tile that keeps three of them (24 warps) on an SM: measured on B200 (tools/bench_assembly.py,
        // residual + Jacobian, M sketches of the config-4 topology / 262,144 trusses): 128 threads S=64 0.185 / 0.216 ms,
        // 256 threads S=128 0.173 ms, S=32 (truss: the largest that fits) 0.163 ms; with the input prefetch S=64 0.161 ms
        // (S=128 0.165) and truss S=32 0.139 ms.  What remains is instruction issue (IEEE divide / sqrt / atan2 sequences and
        // index arithmetic: ~3,000 thread instructions per config-4 sketch, a quarter of them IMAD), not bytes in flight.
        // Input prefetch (second input buffer, cp.async): default on; FK_EVAL_PF=0 keeps the load phase in front of every tile.
        static const bool want_pf = [] {
            const char* e = std::getenv("FK_EVAL_PF");
            return !(e && std::atoi(e) == 0);
        }();
        auto bytes_pf = [&](int S) { return bytes_for(S) + ((size_t)prog.n_vars + prog.n_expr) * (size_t)(S + 1) * sizeof(double); };
        int S = 0;
        bool pf = false;
        if (want_pf) {  // largest tile that keeps four CTAs on an SM, else three
            for (int cand : {32, 64, 128})
                if (bytes_pf(cand) <= 55 * 1024) S = cand;
            if (S == 0)
                for (int cand : {32, 64, 128})
                    if (bytes_pf(cand) <= 74 * 1024) S = cand;
            if (S == 0)
                for (int cand : {32, 64, 128})
                    if (bytes_pf(cand) <= 110 * 1024) S = cand;  // two CTAs: still ahead (truss, S = 32: 0.139 ms against 0.163)
            pf = S != 0;
        }
        if (S == 0)
            for (int cand : {32, 64, 128})
                if (bytes_for(cand) <= 76 * 1024) S = cand;
        if (S == 0)
            for (int cand : {128, 64, 32})
                if (bytes_for(cand) <= 110 * 1024) { S = cand; break; }
        if (const char* e = std::getenv("FK_EVAL_S")) {
            const int f = std::atoi(e);
            if ((f == 32 || f == 64 || f == 128) && (want_pf ? bytes_pf(f) : bytes_for(f)) <= 200 * 1024) { S = f; pf = want_pf; }
        }
        {   // exactness bound of the multiply-high division in the transposes
            const uint64_t wmax = std::max<uint64_t>(std::max(prog.n_vars, prog.n_expr), std::max(prog.m, prog.jnnz));
            if (S != 0 && wmax * wmax * (uint64_t)S >= (1ull << 32)) S = 0;
        }
        if (S != 0) {
            static const int threads = [] {  // CTA size of the tile-staged kernel (A/B knob; see DESIGN.md K1)
                const char* e = std::getenv("FK_EVAL_THREADS");
                return (e && std::atoi(e) == 128) ? 128 : 256;
            }();
            if (threads != 256) pf = false;  // (the prefetching variant exists for 256-thread CTAs)
            const size_t smem = pf ? bytes_pf(S) : bytes_for(S);
            const int ctas_per_sm = (int)std::min<size_t>(16, (226 * 1024) / (smem + 1024));
            const uint32_t tiles = (n_sketches + S - 1) / S;
            const uint32_t grid = std::min<uint32_t>(tiles, 148u * (uint32_t)ctas_per_sm);
            cudaError_t e = cudaSuccess;
#define FK_EVAL_TILED_T(SV, JV, TH, PF)                                                                                    \
    do {                                                                                                               \
        e = cudaFuncSetAttribute(fk_batch_eval_tiled_kernel<SV, JV, TH, PF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        if (e == cudaSuccess)                                                                                          \
            fk_batch_eval_tiled_kernel<SV, JV, TH, PF><<<grid, TH, smem, s>>>(prog, n_sketches, vars, params, out_r, out_j); \
    } while (0)
#define FK_EVAL_TILED(SV, JV)                                   \
    do {                                                        \
        if (pf) FK_EVAL_TILED_T(SV, JV, 256, true);             \
        else if (threads == 256) FK_EVAL_TILED_T(SV, JV, 256, false); \
        else FK_EVAL_TILED_T(SV, JV, 128, false);               \
    } while (0)
            if (S == 128) { if (mode == 0) FK_EVAL_TILED(128, true); else FK_EVAL_TILED(128, false); }
            else if (S == 64) { if (mode == 0) FK_EVAL_TILED(64, true); else FK_EVAL_TILED(64, false); }
            else { if (mode == 0) FK_EVAL_TILED(32, true); else FK_EVAL_TILED(32, false); }
#undef FK_EVAL_TILED_T
#undef FK_EVAL_TILED
            if (e != cudaSuccess) return (int)e;
            return (int)cudaGetLastError();
        }
    }
    const uint64_t total = (uint64_t)n_sketches * prog.m;
    uint64_t blocks = (total + 255) / 256;
    const uint64_t cap = 148ull * 8 * 4;  // a few waves of resident CTAs, grid-stride beyond that
    if (blocks > cap) blocks = cap;
    if (mode == 0) fk_batch_eval_kernel<true><<<(unsigned)blocks, 256, 0, s>>>(prog, n_sketches, vars, params, out_r, out_j);
    else fk_batch_eval_kernel<false><<<(unsigned)blocks, 256, 0, s>>>(prog, n_sketches, vars, params, out_r, out_j);
    return (int)cudaGetLastError();
}

}  // namespace fk
