// See sparse_batch.cuh.  Compiled with -fmad=false like the rest of the library (the evaluators must not contract); the
// linear algebra uses explicit fma().
#include "sparse_batch.cuh"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <utility>

#include "expressions.cuh"
#include "lm_kernels.cuh"
#include "lm_rules.cuh"
#include "multifrontal.cuh"
#include "symbolic.hpp"

namespace fk {

namespace {

constexpr int kSbThreads = 256;
constexpr int kSbWarps = kSbThreads / 32;
constexpr uint32_t kNop = 0xFFFFFFFFu;
constexpr size_t kSbMaxSmem = (size_t)kSbMaxFront * (kSbMaxFront + 1) / 2 * sizeof(double);  // front of order kSbMaxFront
static_assert(kSbMaxFront < (uint32_t)kSbThreads, "the elimination gives every row of a front its own thread");

// Packed lower triangle of order f, column-major: entry (i, j), i >= j, at tri_col(j, f) + i - j.  Consecutive rows of a
// column are consecutive doubles, so a warp working on 32 rows of one column touches 32 distinct banks.
__device__ __forceinline__ uint32_t tri_col(uint32_t j, uint32_t f) { return j * f - (j * (j - 1)) / 2; }

// Sum of one value per thread over the CTA; every thread gets the same bits (butterfly pairs add the same two values,
// the warp totals are added in warp order by every thread).
__device__ __forceinline__ double cta_sum(double s, double* red) {
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < kSbWarps; w++) t += red[w];
    __syncthreads();
    return t;
}
__device__ __forceinline__ double cta_sumsq(const double* v, uint32_t len, double* red) {
    double s = 0.0;
    for (uint32_t i = threadIdx.x; i < len; i += kSbThreads) s = fma(v[i], v[i], s);
    return cta_sum(s, red);
}
// The reference's norm_squared: squares rounded on their own, added left to right (lm_rules.cuh says when).
__device__ __forceinline__ double seq_sumsq(const double* v, uint32_t len, double* red) {
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (uint32_t i = 0; i < len; i++) s = __dadd_rn(s, __dmul_rn(v[i], v[i]));
        red[kSbWarps] = s;
    }
    __syncthreads();
    const double t = red[kSbWarps];
    __syncthreads();
    return t;
}

// K1/K2: residuals and Jacobian (CSC order) at x, one thread per row (the row body of sparse_eval_kernel).
__device__ void sb_eval(const SbDev& D, const double* x, const double* vars, const double* params, double* r, double* J) {
    for (uint32_t row = threadIdx.x; row < D.m; row += kSbThreads) {
        const uint32_t hdr = __ldg(D.row_hdr + row);
        const int kind = (int)(hdr & 0xFFu);
        const int a = dev::arity_of(kind);
        uint2 sl[8];
        double v[8], g[8];
#pragma unroll
        for (int s = 0; s < 8; s++) {
            v[s] = 0.0;
            sl[s] = make_uint2(kNop, kNop);
            if (s < a) {
                sl[s] = __ldg(D.row_slots + (size_t)row * 8 + s);
                v[s] = (int32_t)sl[s].x >= 0 ? x[sl[s].x] : vars[sl[s].x & 0x7FFFFFFFu];
            }
        }
        r[row] = dev::eval_expression(kind, v, params[hdr >> 8], g);
#pragma unroll
        for (int s = 0; s < 8; s++) {
            if (s < a && sl[s].y != kNop) {
                const uint32_t pos = sl[s].y & 0xFFFFFFu;
                if (sl[s].y & 0x40000000u) J[pos] += g[s];
                else J[pos] = g[s];
            }
        }
    }
}

// g = -Jᵀr in permuted order, every entry summed in list order (sparse_gradient_kernel).
__device__ void sb_gradient(const SbDev& D, const double* J, const double* r, double* g) {
    for (uint32_t k = threadIdx.x; k < D.n; k += kSbThreads) {
        double s = 0.0;
        for (uint32_t q = __ldg(D.g_ptr + k); q < __ldg(D.g_ptr + k + 1); q++) s = fma(J[__ldg(D.g_pairs + 2 * q)], r[__ldg(D.g_pairs + 2 * q + 1)], s);
        g[k] = -s;
    }
}

// Multifrontal LDLᵀ of JᵀJ + lam2 I.  Per supernode in postorder: the front's panel columns are summed from the H lists
// (sparse_assemble_kernel's order, lam2 added to the diagonal afterwards as sparse_arm_kernel does), the children's update
// matrices are taken from the top of the update stack and extend-added in ascending child order, the ns pivot columns are
// eliminated right-looking, the panel goes to `pan` and the update matrix onto the stack where the first child's began.
// Fronts of up to 32 rows are worked by warp 0 alone (warp barriers instead of CTA barriers).  Returns the status of
// flag_pivot: 0 all pivots positive, 1 a non-positive or infinite pivot, 2 a NaN pivot.
__device__ int sb_factor(const SbDev& D, const double* J, double lam2, double* pan, double* stk, double* F, int* s_status) {
    const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int status = 0;  // (thread 0)
    for (uint32_t q = 0; q < D.S; q++) {
        const uint32_t s = __ldg(D.post + q);
        const uint4 a = __ldg(D.sn + s), b = __ldg(D.sn2 + s);
        const uint32_t c0 = a.x, ns = a.y, f = a.z;
        const bool solo = f <= 32;
        if (!solo || warp == 0) {
            const uint32_t nw = solo ? 1u : (uint32_t)kSbWarps, nt = solo ? 32u : (uint32_t)kSbThreads, t = solo ? lane : tid;
            auto sync = [&] {
                if (solo) __syncwarp();
                else __syncthreads();
            };
            for (uint32_t j = warp; j < f; j += nw) {
                const uint32_t cs = tri_col(j, f);
                for (uint32_t i = j + lane; i < f; i += 32) {
                    double v = 0.0;
                    if (j < ns) {
                        const uint32_t p = __ldg(D.l_colptr + c0 + j) + (i - j);
                        for (uint32_t h = __ldg(D.h_ptr + p); h < __ldg(D.h_ptr + p + 1); h++)
                            v = fma(J[__ldg(D.h_pairs + 2 * h)], J[__ldg(D.h_pairs + 2 * h + 1)], v);
                        if (i == j) v += lam2;
                    }
                    F[cs + i - j] = v;
                }
            }
            sync();
            for (uint32_t cq = __ldg(D.child_ptr + s); cq < __ldg(D.child_ptr + s + 1); cq++) {
                const uint32_t c = __ldg(D.child + cq);
                const uint4 ca = __ldg(D.sn + c), cb = __ldg(D.sn2 + c);
                const uint32_t rc = ca.z - ca.y;
                const uint32_t* relc = D.rel + cb.x;
                const double* U = stk + cb.w;
                for (uint32_t bb = warp; bb < rc; bb += nw) {
                    const uint32_t tb = __ldg(relc + bb), ucs = tri_col(bb, rc), fcs = tri_col(tb, f);
                    for (uint32_t aa = bb + lane; aa < rc; aa += 32) F[fcs + __ldg(relc + aa) - tb] += U[ucs + aa - bb];
                }
                sync();  // (children may add to the same entries)
            }
            // one barrier per pivot column: column k is scaled after the barrier, and the update with column k + 1
            // reads nothing of column k
            for (uint32_t k = 0; k < ns; k++) {
                const uint32_t ck = tri_col(k, f);
                const double d = F[ck];
                if (tid == 0) {
                    if (d != d) status = 2;
                    else if (!(d > 0.0) || d == INFINITY) status = max(status, 1);
                }
                const double inv = 1.0 / d;
                for (uint32_t i = k + 1 + t; i < f; i += nt) {
                    const double li = F[ck + i - k] * inv;
                    uint32_t cj = ck + (f - k);  // tri_col(k + 1, f)
                    uint32_t j = k + 1;
                    for (; j + 3 <= i; j += 4) {  // four independent entries in flight
                        uint32_t at[4];
                        double c[4], v[4];
#pragma unroll
                        for (int u = 0; u < 4; u++) {
                            at[u] = cj + i - (j + u);
                            cj += f - (j + u);
                            c[u] = F[ck + j + u - k];
                            v[u] = F[at[u]];
                        }
#pragma unroll
                        for (int u = 0; u < 4; u++) F[at[u]] = fma(-li, c[u], v[u]);
                    }
                    for (; j <= i; j++) {
                        F[cj + i - j] = fma(-li, F[ck + j - k], F[cj + i - j]);
                        cj += f - j;
                    }
                }
                sync();
                for (uint32_t i = k + 1 + t; i < f; i += nt) F[ck + i - k] *= inv;
            }
            sync();
            const uint32_t r = f - ns;
            double* P = pan + b.z;
            double* Us = stk + b.w;
            for (uint32_t j = warp; j < f; j += nw) {
                const uint32_t cs = tri_col(j, f);
                if (j < ns) {
                    for (uint32_t i = j + lane; i < f; i += 32) P[(size_t)j * f + i] = F[cs + i - j];
                } else {
                    const uint32_t ucs = tri_col(j - ns, r);
                    for (uint32_t i = j + lane; i < f; i += 32) Us[ucs + i - j] = F[cs + i - j];
                }
            }
        }
        __syncthreads();  // (the next front overwrites F)
    }
    if (tid == 0) *s_status = status;
    __syncthreads();
    const int st = *s_status;
    __syncthreads();
    return st;
}

// w (g in permuted order) -> the step: forward substitution with the unit factor in postorder, the diagonal, backward
// substitution in reverse postorder; delta[perm[k]] = z[k].
__device__ void sb_solve(const SbDev& D, const double* pan, double* w, double* delta) {
    const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (uint32_t q = 0; q < D.S; q++) {
        const uint32_t s = __ldg(D.post + q);
        const uint4 a = __ldg(D.sn + s);
        const uint32_t c0 = a.x, ns = a.y, f = a.z;
        const double* P = pan + __ldg(D.sn2 + s).z;
        const uint32_t* rws = D.rows + a.w;
        if (warp == 0) {
            for (uint32_t j = 0; j < ns; j++) {
                const double yj = w[c0 + j];
                for (uint32_t i = j + 1 + lane; i < ns; i += 32) w[c0 + i] = fma(-P[(size_t)j * f + i], yj, w[c0 + i]);
                __syncwarp();
            }
        }
        __syncthreads();
        if (f > ns) {
            for (uint32_t i = ns + tid; i < f; i += kSbThreads) {
                double acc = 0.0;
                for (uint32_t j = 0; j < ns; j++) acc = fma(P[(size_t)j * f + i], w[c0 + j], acc);
                const uint32_t row = __ldg(rws + i);
                w[row] -= acc;
            }
            __syncthreads();
        }
    }
    for (uint32_t q = D.S; q-- > 0;) {
        const uint32_t s = __ldg(D.post + q);
        const uint4 a = __ldg(D.sn + s);
        const uint32_t c0 = a.x, ns = a.y, f = a.z;
        const double* P = pan + __ldg(D.sn2 + s).z;
        const uint32_t* rws = D.rows + a.w;
        for (uint32_t j = tid; j < ns; j += kSbThreads) {
            double acc = 0.0;
            for (uint32_t i = ns; i < f; i++) acc = fma(P[(size_t)j * f + i], w[__ldg(rws + i)], acc);
            w[c0 + j] = w[c0 + j] / P[(size_t)j * f + j] - acc;
        }
        __syncthreads();
        if (warp == 0) {
            for (uint32_t j = ns; j-- > 0;) {
                const double zj = w[c0 + j];
                for (uint32_t i = lane; i < j; i += 32) w[c0 + i] = fma(-P[(size_t)i * f + j], zj, w[c0 + i]);
                __syncwarp();
            }
        }
        __syncthreads();
    }
    for (uint32_t k = tid; k < D.n; k += kSbThreads) delta[__ldg(D.perm + k)] = w[k];
    __syncthreads();
}

__global__ void __launch_bounds__(kSbThreads, 2)
fk_sparse_batch_lm_kernel(SbDev D, uint32_t n_sketches, const double* __restrict__ vars_all, const double* __restrict__ params_all,
                          double* __restrict__ free_out, fk_report* __restrict__ reports, double* __restrict__ ws, unsigned* __restrict__ next) {
    extern __shared__ double F[];
    __shared__ double red[kSbWarps + 1];
    __shared__ int s_int;
    const uint32_t tid = threadIdx.x, n = D.n, m = D.m;
    double* W = ws + (size_t)blockIdx.x * D.ws_doubles;
    double* const g = W + D.o_g;
    double* const w = W + D.o_w;
    double* const dl = W + D.o_d;
    double* const pan = W + D.o_pan;
    double* const stk = W + D.o_stk;
    for (;;) {
        if (tid == 0) s_int = (int)atomicAdd(next, 1u);
        __syncthreads();
        const uint32_t k = (uint32_t)s_int;
        __syncthreads();
        if (k >= n_sketches) break;
        const double* vars = vars_all + (size_t)k * D.n_vars;
        const double* params = params_all + (size_t)k * D.n_expr;
        double *x = W + D.o_x, *xs = W + D.o_xs, *r = W + D.o_r, *rs = W + D.o_rs, *J = W + D.o_J, *Jt = W + D.o_Jt;
        for (uint32_t c = tid; c < n; c += kSbThreads) x[c] = vars[__ldg(D.free_vars + c)];
        __syncthreads();
        // lm.rs:80-106
        sb_eval(D, x, vars, params, r, J);
        __syncthreads();
        double ssr = cta_sumsq(r, m, red);
        if (lm_initial_ssr_needs_exact(ssr, m)) ssr = seq_sumsq(r, m, red);
        sb_gradient(D, J, r, g);
        __syncthreads();
        double lambda = 0.5;
        uint32_t exit_reason = FK_EXIT_MAX_OUTER, outer_iters = 0, factorizations = 0, accepted = 0;
        uint64_t trace = 0;
        bool active = true;
        if (ssr < 1e-8) {
            exit_reason = FK_EXIT_CONVERGED_RESIDUAL;
            active = false;
        } else {
            outer_iters = 1;
        }
        // every value below is CTA-uniform: the same decisions in every thread
        while (active) {
            if (!isfinite(lambda)) {
                exit_reason = FK_EXIT_LAMBDA_OVERFLOW;
                break;
            }
            const double sl = sqrt(lambda);
            const double lam2 = sl * sl;
            const int fstat = sb_factor(D, J, lam2, pan, stk, F, &s_int);
            factorizations++;
            double dn = 0.0, ssr_s = NAN;
            if (fstat == 0) {  // (a failed factorisation decides without its step: the single-system path discards it)
                for (uint32_t c = tid; c < n; c += kSbThreads) w[c] = g[c];
                __syncthreads();
                sb_solve(D, pan, w, dl);
                dn = cta_sumsq(dl, n, red);
                for (uint32_t c = tid; c < n; c += kSbThreads) xs[c] = x[c] + dl[c];
                __syncthreads();
                sb_eval(D, xs, vars, params, rs, Jt);
                __syncthreads();
                ssr_s = cta_sumsq(rs, m, red);
                if (lm_step_needs_exact(fstat, dn, ssr_s, ssr, n, m)) {
                    dn = seq_sumsq(dl, n, red);
                    ssr_s = seq_sumsq(rs, m, red);
                    ssr = seq_sumsq(r, m, red);
                }
            }
            if (fstat == 1) {  // non-positive pivot == the reference's `!solved` (lm.rs:134-137)
                lambda *= 8.0;
                trace = trace * 3ull + 1ull;
                continue;
            }
            if (fstat == 0 && dn < 1e-12) {  // lm.rs:139-142
                exit_reason = FK_EXIT_SMALL_STEP;
                break;
            }
            if (ssr_s < ssr) {
                lambda *= 0.125;
                if (lambda < 1e-50) lambda = 1e-50;
                accepted++;
                trace = trace * 3ull + 2ull;
                double* tmp = x; x = xs; xs = tmp;
                tmp = r; r = rs; rs = tmp;
                tmp = J; J = Jt; Jt = tmp;
                const bool stalled = (ssr - ssr_s) / ssr <= 1e-6;
                ssr = ssr_s;
                if (stalled) {
                    exit_reason = FK_EXIT_STALLED;
                    break;
                }
                sb_gradient(D, J, r, g);
                __syncthreads();
                if (outer_iters == 100) break;
                if (ssr < 1e-8) {
                    exit_reason = FK_EXIT_CONVERGED_RESIDUAL;
                    break;
                }
                outer_iters++;
            } else {
                lambda *= 2.0;
                trace = trace * 3ull + 3ull;
            }
        }
        for (uint32_t c = tid; c < n; c += kSbThreads) free_out[(size_t)k * n + c] = x[c];
        if (tid == 0) {
            fk_report rep;
            rep.exit_reason = exit_reason;
            rep.outer_iters = outer_iters;
            rep.factorizations = factorizations;
            rep.accepted = accepted;
            rep.ssr = ssr;
            rep.lambda = lambda;
            rep.trace_hash = trace;
            reports[k] = rep;
        }
        __syncthreads();  // (the next sketch overwrites the workspace)
    }
}

template <class T>
cudaError_t upload_vec(const std::vector<T>& v, const T** out, std::vector<void*>& owned) {
    void* d = nullptr;
    cudaError_t e = cudaMalloc(&d, std::max<size_t>(1, v.size()) * sizeof(T));
    if (e != cudaSuccess) return e;
    owned.push_back(d);
    if (!v.empty()) e = cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
    *out = (const T*)d;
    return e;
}

int analyse(const Topology& t, Multifrontal& mf, std::string* err) {
    std::string merr;
    if (mf.build_symbolic(t, &merr) != cudaSuccess) {
        if (err) *err = merr;
        return FK_ERR_TOO_LARGE;
    }
    if (mf.sym.max_front > kSbMaxFront) {
        if (err)
            *err = "largest supernodal front has order " + std::to_string(mf.sym.max_front) + "; the batched sparse kernel holds fronts of up to " +
                   std::to_string(kSbMaxFront) + " rows in shared memory (solve such systems one at a time with fk_topology_lm_solve)";
        return FK_ERR_TOO_LARGE;
    }
    return FK_OK;
}

}  // namespace

int sparse_batch_fits(const Topology& t, uint32_t* max_front, std::string* err) {
    Multifrontal mf;
    const int rc = analyse(t, mf, err);
    if (max_front) *max_front = mf.sym.max_front;
    return rc;
}

SparseBatchProgram::~SparseBatchProgram() {
    if (device_ >= 0) cudaSetDevice(device_);
    for (void* p : owned_) cudaFree(p);
}

#define SB_CU(call)                                                              \
    do {                                                                         \
        cudaError_t e_ = (call);                                                 \
        if (e_ != cudaSuccess) {                                                 \
            if (err) *err = std::string(#call) + ": " + cudaGetErrorString(e_);  \
            return e_ == cudaErrorMemoryAllocation ? FK_ERR_OOM : FK_ERR_CUDA;   \
        }                                                                        \
    } while (0)

int SparseBatchProgram::init(const Topology& t, const DevProgram& prog, int device, std::string* err) {
    Multifrontal mf;
    int rc = analyse(t, mf, err);
    if (rc != FK_OK) return rc;
    const MfSymbolic& y = mf.sym;
    const uint32_t S = y.S;
    // postorder of the supernodal forest, children in ascending order
    std::vector<uint32_t> post;
    post.reserve(S);
    {
        std::vector<std::pair<uint32_t, uint32_t>> st;  // (supernode, next child slot)
        for (uint32_t root = 0; root < S; root++) {
            if (y.sparent[root] >= 0) continue;
            st.push_back({root, y.child_ptr[root]});
            while (!st.empty()) {
                const uint32_t s = st.back().first, cq = st.back().second;
                if (cq < y.child_ptr[s + 1]) {
                    st.back().second++;
                    st.push_back({y.child[cq], y.child_ptr[y.child[cq]]});
                } else {
                    post.push_back(s);
                    st.pop_back();
                }
            }
        }
    }
    if (post.size() != S) {
        if (err) *err = "sparse batch: the supernodal tree is not a forest";
        return FK_ERR_INTERNAL;
    }
    // update stack: in postorder the children's update matrices are the topmost entries, in child order; the parent
    // reads them, then pushes its own where the first child's began
    auto upd_size = [&](uint32_t s) { const uint64_t r = y.f[s] - y.ns[s]; return r * (r + 1) / 2; };
    std::vector<uint64_t> stk(S, 0);
    uint64_t top = 0, peak = 0;
    for (uint32_t s : post) {
        for (uint32_t cq = y.child_ptr[s]; cq < y.child_ptr[s + 1]; cq++) top -= upd_size(y.child[cq]);
        if (y.child_ptr[s + 1] > y.child_ptr[s] && stk[y.child[y.child_ptr[s]]] != top) {
            if (err) *err = "sparse batch: children's update matrices are not on top of the stack";
            return FK_ERR_INTERNAL;
        }
        stk[s] = top;
        top += upd_size(s);
        peak = std::max(peak, top);
    }
    // per-CTA workspace (doubles), every array on a 256-byte boundary
    const uint32_t n = t.n_free, m = t.n_rows;
    uint64_t off = 0;
    auto take = [&](uint64_t count) {
        const uint64_t at = off;
        off += (std::max<uint64_t>(count, 1) + 31) & ~uint64_t(31);
        return at;
    };
    SbDev& D = dev_;
    const uint64_t o_x = take(n), o_xs = take(n), o_g = take(n), o_w = take(n), o_d = take(n), o_r = take(m), o_rs = take(m),
                   o_J = take(t.jac_nnz), o_Jt = take(t.jac_nnz), o_pan = take(y.pan_total), o_stk = take(peak);
    if (off >= (1ull << 32) || t.l_rowidx.size() >= (1ull << 32)) {
        if (err) *err = "sparse batch: the workspace of one sketch exceeds 32-bit offsets";
        return FK_ERR_TOO_LARGE;
    }
    D.o_x = (uint32_t)o_x; D.o_xs = (uint32_t)o_xs; D.o_g = (uint32_t)o_g; D.o_w = (uint32_t)o_w; D.o_d = (uint32_t)o_d;
    D.o_r = (uint32_t)o_r; D.o_rs = (uint32_t)o_rs; D.o_J = (uint32_t)o_J; D.o_Jt = (uint32_t)o_Jt; D.o_pan = (uint32_t)o_pan;
    D.o_stk = (uint32_t)o_stk;
    D.ws_doubles = off;
    D.n = n; D.m = m; D.n_vars = t.n_vars; D.n_expr = t.n_expr; D.S = S;
    D.row_hdr = prog.row_hdr; D.row_slots = prog.row_slots; D.free_vars = prog.free_vars;
    std::vector<uint4> sn(S), sn2(S);
    for (uint32_t s = 0; s < S; s++) {
        sn[s] = make_uint4(y.c0[s], y.ns[s], y.f[s], y.rows_off[s]);
        sn2[s] = make_uint4(y.rel_off[s], 0u, (uint32_t)y.pan_off[s], (uint32_t)stk[s]);  // (.y: padding)
    }
    device_ = device;
    SB_CU(cudaSetDevice(device));
    SB_CU(upload_vec(t.g_ptr, &D.g_ptr, owned_));
    SB_CU(upload_vec(t.g_pairs, &D.g_pairs, owned_));
    SB_CU(upload_vec(t.perm, &D.perm, owned_));
    SB_CU(upload_vec(t.l_colptr, &D.l_colptr, owned_));
    SB_CU(upload_vec(t.h_ptr, &D.h_ptr, owned_));
    SB_CU(upload_vec(t.h_pairs, &D.h_pairs, owned_));
    SB_CU(upload_vec(post, &D.post, owned_));
    SB_CU(upload_vec(sn, &D.sn, owned_));
    SB_CU(upload_vec(sn2, &D.sn2, owned_));
    SB_CU(upload_vec(y.child_ptr, &D.child_ptr, owned_));
    SB_CU(upload_vec(y.child, &D.child, owned_));
    SB_CU(upload_vec(y.rows, &D.rows, owned_));
    SB_CU(upload_vec(y.rel, &D.rel, owned_));
    smem_ = (uint32_t)(std::max<uint64_t>(1, (uint64_t)y.max_front * (y.max_front + 1) / 2) * sizeof(double));
    // The attribute belongs to the kernel on the device, not to this topology: every topology sets the same value, the
    // largest front the kernel takes, so that no topology's setting can refuse another's launch, whatever the order
    // (or the threads) in which they are set up.  Each launch asks for its own front's size.
    SB_CU(cudaFuncSetAttribute(fk_sparse_batch_lm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSbMaxSmem));
    int per_sm = 0, sms = 0;
    SB_CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fk_sparse_batch_lm_kernel, kSbThreads, smem_));
    SB_CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    if (per_sm < 1) {
        if (err) *err = "sparse batch: the kernel does not fit an SM with a front of order " + std::to_string(y.max_front);
        return FK_ERR_TOO_LARGE;
    }
    resident_ = (uint32_t)(per_sm * sms);
    return FK_OK;
}

int SparseBatchProgram::launch(uint32_t n, const double* vars, const double* params, double* free_out, fk_report* reports, double* workspace,
                               uint32_t ctas, void* stream) const {
    if (n == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(workspace, 0, sizeof(unsigned), st);
    if (e != cudaSuccess) return (int)e;
    const uint32_t grid = std::min(n, std::min(ctas, resident_));
    fk_sparse_batch_lm_kernel<<<grid, kSbThreads, smem_, st>>>(dev_, n, vars, params, free_out, reports, workspace + kHeadDoubles,
                                                                 (unsigned*)workspace);
    return (int)cudaGetLastError();
}

}  // namespace fk
