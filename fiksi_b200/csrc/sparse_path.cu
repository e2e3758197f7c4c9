// See sparse_path.cuh.  Compiled with -fmad=false (the evaluators must not contract); the linear
// algebra uses explicit fma().
#include "sparse_path.cuh"

#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "expressions.cuh"
#include "lm_rules.cuh"
#include "multifrontal.cuh"

namespace fk {

namespace {

constexpr uint32_t kNop = 0xFFFFFFFFu;

struct SparseDev {
    uint32_t n, m, jnnz, n_vars, n_expr, n_hent;
    // evaluation tables (Topology::Tables layout with tile == 1)
    const uint32_t* row_hdr;
    const uint2* row_slots;
    // Jacobian CSC without damping rows (g = -J^T r): column c = entries jcolptr[c]..jcolptr[c+1]
    const uint32_t* jcolptr;
    const uint32_t* jrow;
    const int32_t* perm;      // perm[k] = original column at position k
    // H = JtJ contribution lists, only entries that receive contributions
    const uint32_t* he_pos;   // [n_hent] offset in the supernodal panel storage
    const uint32_t* he_ptr;   // [n_hent+1]
    const uint32_t* he_pairs; // 2 per contribution
    const uint32_t* diag_pos; // [n] panel offset of the diagonal entry of permuted column k
    double* pan;              // supernodal panels (multifrontal.cuh)
    int* status;              // factorisation status word
};

// ---- K1 / K2 -----------------------------------------------------------------------------------
template <bool WITH_JACOBIAN>
__global__ void __launch_bounds__(256)
sparse_eval_kernel(SparseDev S, const double* __restrict__ x, const double* __restrict__ vars,
                   const double* __restrict__ params, double* __restrict__ r, double* __restrict__ J) {
    for (uint32_t row = blockIdx.x * blockDim.x + threadIdx.x; row < S.m; row += gridDim.x * blockDim.x) {
        const uint32_t hdr = __ldg(S.row_hdr + row);
        const int kind = (int)(hdr & 0xFFu);
        const int a = dev::arity_of(kind);
        uint2 sl[8];
        double v[8], g[8];
#pragma unroll
        for (int s = 0; s < 8; s++) {
            v[s] = 0.0;
            sl[s] = make_uint2(kNop, kNop);
            if (s < a) {
                sl[s] = __ldg(S.row_slots + (size_t)row * 8 + s);
                v[s] = (int32_t)sl[s].x >= 0 ? x[sl[s].x] : __ldg(vars + (sl[s].x & 0x7FFFFFFFu));
            }
        }
        r[row] = dev::eval_expression(kind, v, __ldg(params + (hdr >> 8)), g);
        if (WITH_JACOBIAN) {
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
}

// ---- K3 ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
sparse_assemble_kernel(SparseDev S, const double* __restrict__ J) {
    for (uint32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < S.n_hent; e += gridDim.x * blockDim.x) {
        const uint32_t b = __ldg(S.he_ptr + e), en = __ldg(S.he_ptr + e + 1);
        double s = 0.0;
        for (uint32_t q = b; q < en; q++) s = fma(J[__ldg(S.he_pairs + 2 * q)], J[__ldg(S.he_pairs + 2 * q + 1)], s);
        S.pan[__ldg(S.he_pos + e)] = s;
    }
}
// Damping (sqrt(lambda))^2 on the diagonal (lm.rs:119-125); clears the factorisation status.
__global__ void __launch_bounds__(256) sparse_arm_kernel(SparseDev S, double lam2) {
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < S.n; k += gridDim.x * blockDim.x)
        S.pan[__ldg(S.diag_pos + k)] += lam2;
    if (blockIdx.x == 0 && threadIdx.x == 0) *S.status = 0;
}

__global__ void __launch_bounds__(256)
sparse_gradient_kernel(SparseDev S, const double* __restrict__ J, const double* __restrict__ r, double* __restrict__ g) {
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < S.n; k += gridDim.x * blockDim.x) {
        const uint32_t c = (uint32_t)__ldg(S.perm + k);
        double s = 0.0;
        for (uint32_t q = __ldg(S.jcolptr + c); q < __ldg(S.jcolptr + c + 1); q++) s = fma(J[q], r[__ldg(S.jrow + q)], s);
        g[k] = -s;  // r := -r of lm.rs:86-88 folded into the sign
    }
}

// ---- deterministic reductions and vector helpers -----------------------------------------------------
constexpr int kRedBlocks = 592, kRedThreads = 256;
__global__ void __launch_bounds__(kRedThreads)
sumsq_partial_kernel(const double* __restrict__ v, uint32_t n, double* __restrict__ partial) {
    __shared__ double sh[kRedThreads];
    double s = 0.0;
    for (uint32_t i = blockIdx.x * kRedThreads + threadIdx.x; i < n; i += kRedBlocks * kRedThreads) s = fma(v[i], v[i], s);
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int o = kRedThreads / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[blockIdx.x] = sh[0];
}
__global__ void __launch_bounds__(1024)
sumsq_final_kernel(const double* __restrict__ partial, double* __restrict__ out) {
    __shared__ double sh[1024];
    sh[threadIdx.x] = threadIdx.x < kRedBlocks ? partial[threadIdx.x] : 0.0;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = sh[0];
}
// The reference's norm_squared (fiksi/src/solve/lm.rs:195-197) is a sequential, non-fused sum.  The tree
// reduction above rounds differently in the last bits; whenever one of the LM decisions lies within the
// distance the two can differ by, the host asks for this kernel: the squares are formed by all threads
// (a product is rounded the same way wherever it is computed), the additions are done by thread 0 alone,
// left to right, from shared memory.  ~1.4 ms for 300,000 values; used only near a threshold.
constexpr int kSeqChunk = 2048;
__global__ void __launch_bounds__(256)
sumsq_sequential_kernel(const double* __restrict__ v, uint32_t n, double* __restrict__ out) {
    __shared__ double sq[2][kSeqChunk];
    double s = 0.0;
    const uint32_t nchunks = (n + kSeqChunk - 1) / kSeqChunk;
    auto stage = [&](uint32_t ch) {
        for (uint32_t i = threadIdx.x; i < kSeqChunk; i += 256) {
            const uint32_t k = ch * kSeqChunk + i;
            const double x = k < n ? v[k] : 0.0;
            sq[ch & 1][i] = __dmul_rn(x, x);
        }
    };
    if (nchunks) stage(0);
    __syncthreads();
    for (uint32_t ch = 0; ch < nchunks; ch++) {
        if (threadIdx.x == 0) {
            const uint32_t cnt = min((uint32_t)kSeqChunk, n - ch * kSeqChunk);
            const double* q = sq[ch & 1];
#pragma unroll 8
            for (uint32_t i = 0; i < cnt; i++) s = __dadd_rn(s, q[i]);
        } else if (ch + 1 < nchunks) {
            stage(ch + 1);  // threads 1..255 fill the other buffer meanwhile (thread 0's share below)
        }
        if (threadIdx.x == 0 && ch + 1 < nchunks) {
            for (uint32_t i = 0; i < kSeqChunk; i += 256) {
                const uint32_t k = (ch + 1) * kSeqChunk + i;
                const double x = k < n ? v[k] : 0.0;
                sq[(ch + 1) & 1][i] = __dmul_rn(x, x);
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = s;
}
__global__ void __launch_bounds__(256)
add_kernel(const double* __restrict__ a, const double* __restrict__ b, double* __restrict__ out, uint32_t n) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = a[i] + b[i];
}
__global__ void fetch_flag_kernel(const int* status, double* scalars) { scalars[2] = (double)*status; }

template <class T>
cudaError_t upload(const std::vector<T>& v, const T** out, std::vector<void*>& owned) {
    void* d = nullptr;
    cudaError_t e = cudaMalloc(&d, std::max<size_t>(1, v.size()) * sizeof(T));
    if (e != cudaSuccess) return e;
    owned.push_back(d);
    if (!v.empty()) e = cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
    *out = (const T*)d;
    return e;
}

}  // namespace

struct SparseSolver::Impl {
    const Topology* t = nullptr;
    int device = 0;
    SparseDev S{};
    std::vector<void*> owned;
    double *d_x = nullptr, *d_xs = nullptr, *d_vars = nullptr, *d_params = nullptr;
    double *d_r = nullptr, *d_rs = nullptr, *d_J = nullptr, *d_Jt = nullptr, *d_g = nullptr, *d_w = nullptr;
    double *d_delta = nullptr, *d_partial = nullptr, *d_scalars = nullptr;
    double* h_scalars = nullptr;  // pinned: [0] dn, [1] ssr, [2] factor status
    int sm_count = 0;
    Multifrontal mf;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[2] = {nullptr, nullptr};

    template <class T>
    cudaError_t alloc(T** p, size_t count) {
        void* d = nullptr;
        cudaError_t e = cudaMalloc(&d, std::max<size_t>(1, count) * sizeof(T));
        if (e == cudaSuccess) {
            owned.push_back(d);
            *p = (T*)d;
        }
        return e;
    }
    int grid_for(uint32_t items) const {
        uint32_t b = (items + 255) / 256;
        return (int)std::max<uint32_t>(1, std::min<uint32_t>(b, (uint32_t)sm_count * 8));
    }
    cudaError_t sumsq(const double* v, uint32_t n, double* out) {
        sumsq_partial_kernel<<<kRedBlocks, kRedThreads, 0, stream>>>(v, n, d_partial);
        sumsq_final_kernel<<<1, 1024, 0, stream>>>(d_partial, out);
        return cudaGetLastError();
    }
    cudaError_t sumsq_exact(const double* v, uint32_t n, double* out) {
        sumsq_sequential_kernel<<<1, 256, 0, stream>>>(v, n, out);
        return cudaGetLastError();
    }
    void eval(const double* x, double* r, double* J) {
        sparse_eval_kernel<true><<<grid_for(S.m), 256, 0, stream>>>(S, x, d_vars, d_params, r, J);
    }
};

SparseSolver::~SparseSolver() {
    if (!impl_) return;
    cudaSetDevice(impl_->device);
    for (void* p : impl_->owned) cudaFree(p);
    if (impl_->h_scalars) cudaFreeHost(impl_->h_scalars);
    if (impl_->stream) cudaStreamDestroy(impl_->stream);
    for (auto& e : impl_->ev)
        if (e) cudaEventDestroy(e);
    delete impl_;
}

#define SP_CU(call)                                                              \
    do {                                                                         \
        cudaError_t e_ = (call);                                                 \
        if (e_ != cudaSuccess) {                                                 \
            if (err) *err = std::string(#call) + ": " + cudaGetErrorString(e_);  \
            return e_ == cudaErrorMemoryAllocation ? FK_ERR_OOM : FK_ERR_CUDA;   \
        }                                                                        \
    } while (0)

int SparseSolver::init(const Topology& t, int device, std::string* err) {
    impl_ = new Impl();
    Impl& I = *impl_;
    I.t = &t;
    I.device = device;
    static const bool sym_timing = std::getenv("FK_SYM_TIMING") != nullptr;
    auto lap_t0 = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (!sym_timing) return;
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[sparse init] %-26s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(now - lap_t0).count());
        lap_t0 = now;
    };
    SP_CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    SP_CU(cudaGetDeviceProperties(&prop, device));
    I.sm_count = prop.multiProcessorCount;
    const uint32_t n = t.n_free, m = t.n_rows, lnnz = (uint32_t)t.l_rowidx.size();
    if (t.jac_nnz >= (1u << 24) || t.n_expr >= (1u << 24)) {
        if (err) *err = "problem exceeds the 24-bit position fields of the evaluation tables";
        return FK_ERR_TOO_LARGE;
    }
    SparseDev& S = I.S;
    S.n = n; S.m = m; S.jnnz = t.jac_nnz; S.n_vars = t.n_vars; S.n_expr = t.n_expr;

    // evaluation tables
    SP_CU(upload(t.tab.row_hdr, &S.row_hdr, I.owned));
    {
        const uint32_t* p = nullptr;
        SP_CU(upload(t.tab.row_slots, &p, I.owned));
        S.row_slots = (const uint2*)p;
    }
    // CSC Jacobian without the damping rows
    std::vector<uint32_t> jcolptr(n + 1), jrow(t.jac_nnz);
    for (uint32_t c = 0; c <= n; c++) jcolptr[c] = t.aug_colptr[c] - c;
    for (uint32_t c = 0; c < n; c++)
        for (uint32_t q = t.aug_colptr[c]; q + 1 < t.aug_colptr[c + 1]; q++) jrow[q - c] = t.aug_rowidx[q];
    SP_CU(upload(jcolptr, &S.jcolptr, I.owned));
    SP_CU(upload(jrow, &S.jrow, I.owned));
    SP_CU(upload(t.perm, &S.perm, I.owned));
    lap("context, evaluation tables");
    // supernodal multifrontal factorisation (K5): symbolic structures, panel storage
    {
        std::string merr;
        cudaError_t me = I.mf.init(t, nullptr, &merr);
        if (me != cudaSuccess) {
            if (err) *err = merr + ": " + cudaGetErrorString(me);
            return me == cudaErrorMemoryAllocation ? FK_ERR_OOM : (me == cudaErrorInvalidValue ? FK_ERR_TOO_LARGE : FK_ERR_CUDA);
        }
    }
    if (I.mf.panel_doubles() >= (1ull << 32)) {
        if (err) *err = "panel storage exceeds the 32-bit offsets of the assembly lists";
        return FK_ERR_TOO_LARGE;
    }
    lap("multifrontal init");
    S.pan = I.mf.panels();
    S.status = I.mf.status();
    // compacted H contribution lists, addressed by panel offset
    const std::vector<uint64_t>& dmap = I.mf.diag_panel();
    std::vector<uint32_t> he_pos, he_ptr, diag_pos(n);
    for (uint32_t j = 0; j < n; j++)
        for (uint32_t p = t.l_colptr[j]; p < t.l_colptr[j + 1]; p++)
            if (t.h_ptr[p + 1] > t.h_ptr[p]) {
                he_pos.push_back((uint32_t)(dmap[j] + (p - t.l_colptr[j])));
                he_ptr.push_back(t.h_ptr[p]);  // h_pairs is ordered by L position: lists stay contiguous
            }
    he_ptr.push_back(t.h_ptr[lnnz]);
    for (uint32_t k = 0; k < n; k++) diag_pos[k] = (uint32_t)I.mf.diag_panel()[k];
    S.n_hent = (uint32_t)he_pos.size();
    SP_CU(upload(he_pos, &S.he_pos, I.owned));
    SP_CU(upload(he_ptr, &S.he_ptr, I.owned));
    SP_CU(upload(t.h_pairs, &S.he_pairs, I.owned));
    SP_CU(upload(diag_pos, &S.diag_pos, I.owned));
    lap("assembly lists");
    SP_CU(I.alloc(&I.d_x, n));
    SP_CU(I.alloc(&I.d_xs, n));
    SP_CU(I.alloc(&I.d_vars, t.n_vars));
    SP_CU(I.alloc(&I.d_params, t.n_expr));
    SP_CU(I.alloc(&I.d_r, m));
    SP_CU(I.alloc(&I.d_rs, m));
    SP_CU(I.alloc(&I.d_J, t.jac_nnz));
    SP_CU(I.alloc(&I.d_Jt, t.jac_nnz));
    SP_CU(I.alloc(&I.d_g, n));
    SP_CU(I.alloc(&I.d_w, n));
    SP_CU(I.alloc(&I.d_delta, n));
    SP_CU(I.alloc(&I.d_partial, kRedBlocks));
    SP_CU(I.alloc(&I.d_scalars, 4));
    SP_CU(cudaMallocHost((void**)&I.h_scalars, 4 * sizeof(double)));
    SP_CU(cudaStreamCreateWithFlags(&I.stream, cudaStreamNonBlocking));
    SP_CU(cudaEventCreate(&I.ev[0]));
    SP_CU(cudaEventCreate(&I.ev[1]));
    lap("work vectors, stream");
    return FK_OK;
}

int SparseSolver::eval_once(const double* vars, const double* param, const double* free_values, double* out_r,
                            double* out_j, int repeats, float* ms_per_eval, std::string* err) {
    Impl& I = *impl_;
    const Topology& t = *I.t;
    SP_CU(cudaSetDevice(I.device));
    SP_CU(cudaMemcpyAsync(I.d_vars, vars, sizeof(double) * t.n_vars, cudaMemcpyHostToDevice, I.stream));
    if (t.n_expr) SP_CU(cudaMemcpyAsync(I.d_params, param, sizeof(double) * t.n_expr, cudaMemcpyHostToDevice, I.stream));
    SP_CU(cudaMemcpyAsync(I.d_x, free_values, sizeof(double) * t.n_free, cudaMemcpyHostToDevice, I.stream));
    I.eval(I.d_x, I.d_r, I.d_J);
    SP_CU(cudaEventRecord(I.ev[0], I.stream));
    for (int k = 0; k < repeats; k++) I.eval(I.d_x, I.d_r, I.d_J);
    SP_CU(cudaEventRecord(I.ev[1], I.stream));
    if (out_r) SP_CU(cudaMemcpyAsync(out_r, I.d_r, sizeof(double) * t.n_rows, cudaMemcpyDeviceToHost, I.stream));
    if (out_j) SP_CU(cudaMemcpyAsync(out_j, I.d_J, sizeof(double) * t.jac_nnz, cudaMemcpyDeviceToHost, I.stream));
    SP_CU(cudaStreamSynchronize(I.stream));
    if (ms_per_eval && repeats > 0) {
        float ms = 0;
        cudaEventElapsedTime(&ms, I.ev[0], I.ev[1]);
        *ms_per_eval = ms / repeats;
    }
    return FK_OK;
}

int SparseSolver::solve(const double* vars, const double* param, double* free_values, fk_report* report, std::string* err) {
    Impl& I = *impl_;
    const Topology& t = *I.t;
    SparseDev& S = I.S;
    const uint32_t n = t.n_free, m = t.n_rows;
    SP_CU(cudaSetDevice(I.device));
    cudaStream_t st = I.stream;
    last = Timing();
    SP_CU(cudaMemcpyAsync(I.d_vars, vars, sizeof(double) * t.n_vars, cudaMemcpyHostToDevice, st));
    if (t.n_expr) SP_CU(cudaMemcpyAsync(I.d_params, param, sizeof(double) * t.n_expr, cudaMemcpyHostToDevice, st));
    SP_CU(cudaMemcpyAsync(I.d_x, free_values, sizeof(double) * n, cudaMemcpyHostToDevice, st));

    double* x = I.d_x;
    double* xs = I.d_xs;
    double* r = I.d_r;
    double* rs = I.d_rs;
    double* J = I.d_J;
    double* Jt = I.d_Jt;

    auto phase = [&](float& acc, auto&& body) -> cudaError_t {
        cudaEventRecord(I.ev[0], st);
        body();
        cudaEventRecord(I.ev[1], st);
        cudaError_t e = cudaEventSynchronize(I.ev[1]);
        if (e != cudaSuccess) return e;
        float ms = 0;
        cudaEventElapsedTime(&ms, I.ev[0], I.ev[1]);
        acc += ms;
        return cudaGetLastError();
    };

    // lm.rs:80-106
    SP_CU(phase(last.eval_ms, [&] { I.eval(x, r, J); }));
    last.evals++;
    SP_CU(I.sumsq(r, m, I.d_scalars + 1));
    sparse_gradient_kernel<<<I.grid_for(n), 256, 0, st>>>(S, J, r, I.d_g);
    SP_CU(cudaMemcpyAsync(I.h_scalars, I.d_scalars, 4 * sizeof(double), cudaMemcpyDeviceToHost, st));
    SP_CU(cudaStreamSynchronize(st));
    double ssr = I.h_scalars[1];
    if (lm_initial_ssr_needs_exact(ssr, m)) {
        SP_CU(I.sumsq_exact(r, m, I.d_scalars + 1));  // the first lm.rs:110 test sits on its threshold: decide on the reference's sum
        SP_CU(cudaMemcpyAsync(I.h_scalars, I.d_scalars, 4 * sizeof(double), cudaMemcpyDeviceToHost, st));
        SP_CU(cudaStreamSynchronize(st));
        ssr = I.h_scalars[1];
        last.exact_sums++;
    }

    double lambda = 0.5;
    uint32_t exit_reason = FK_EXIT_MAX_OUTER, outer_iters = 0, factorizations = 0, accepted = 0;
    uint64_t trace = 0;
    auto push = [&](uint32_t code) { trace = trace * 3ull + code + 1ull; };
    bool active = true;
    if (ssr < 1e-8) {
        exit_reason = FK_EXIT_CONVERGED_RESIDUAL;
        active = false;
    } else {
        outer_iters = 1;
    }
    while (active) {
        if (!std::isfinite(lambda)) {
            exit_reason = FK_EXIT_LAMBDA_OVERFLOW;
            break;
        }
        const double sl = std::sqrt(lambda);
        const double lam2 = sl * sl;
        SP_CU(phase(last.assemble_ms, [&] {
            cudaMemsetAsync(S.pan, 0, sizeof(double) * I.mf.panel_doubles(), st);
            sparse_assemble_kernel<<<I.grid_for(S.n_hent), 256, 0, st>>>(S, J);
            sparse_arm_kernel<<<I.grid_for(n), 256, 0, st>>>(S, lam2);
        }));
        SP_CU(phase(last.factor_ms, [&] { I.mf.factor(st); }));
        factorizations++;
        last.factors++;
        SP_CU(phase(last.tri_ms, [&] {
            cudaMemcpyAsync(I.d_w, I.d_g, sizeof(double) * n, cudaMemcpyDeviceToDevice, st);
            I.mf.solve(I.d_w, I.d_delta, S.perm, st);
        }));
        SP_CU(I.sumsq(I.d_delta, n, I.d_scalars + 0));
        add_kernel<<<I.grid_for(n), 256, 0, st>>>(x, I.d_delta, xs, n);
        SP_CU(phase(last.eval_ms, [&] { I.eval(xs, rs, Jt); }));
        last.evals++;
        SP_CU(I.sumsq(rs, m, I.d_scalars + 1));
        fetch_flag_kernel<<<1, 1, 0, st>>>(S.status, I.d_scalars);
        SP_CU(cudaMemcpyAsync(I.h_scalars, I.d_scalars, 4 * sizeof(double), cudaMemcpyDeviceToHost, st));
        SP_CU(cudaStreamSynchronize(st));
        const int fstat = (int)I.h_scalars[2];
        if (fstat >= 3) {  // a polling loop of the dataflow / chained kernels gave up (see SpinGuard)
            if (err) *err = "multifrontal: a polling kernel timed out waiting for a published value";
            return FK_ERR_INTERNAL;
        }
        double dn = I.h_scalars[0];
        double ssr_s = I.h_scalars[1];
        {   // Decisions of lm.rs:139,151,164,110 taken on tree-reduced sums (lm_rules.cuh): near a threshold, redo the
            // three sums in the reference's order and decide on those (and carry the exact ssr forward).
            if (lm_step_needs_exact(fstat, dn, ssr_s, ssr, n, m)) {
                SP_CU(I.sumsq_exact(I.d_delta, n, I.d_scalars + 0));
                SP_CU(I.sumsq_exact(rs, m, I.d_scalars + 1));
                SP_CU(I.sumsq_exact(r, m, I.d_scalars + 3));
                SP_CU(cudaMemcpyAsync(I.h_scalars, I.d_scalars, 4 * sizeof(double), cudaMemcpyDeviceToHost, st));
                SP_CU(cudaStreamSynchronize(st));
                dn = I.h_scalars[0];
                ssr_s = I.h_scalars[1];
                ssr = I.h_scalars[3];
                last.exact_sums++;
            }
        }
        if (fstat == 1) {  // non-positive pivot == the reference's `!solved` (lm.rs:134-137)
            lambda *= 8.0;
            push(0);
            continue;
        }
        if (fstat == 2) ssr_s = NAN;
        if (fstat == 0 && dn < 1e-12) {  // lm.rs:139-142
            exit_reason = FK_EXIT_SMALL_STEP;
            break;
        }
        if (ssr_s < ssr) {
            lambda *= 0.125;
            if (lambda < 1e-50) lambda = 1e-50;
            accepted++;
            push(1);
            std::swap(x, xs);
            std::swap(r, rs);
            std::swap(J, Jt);
            const bool stalled = (ssr - ssr_s) / ssr <= 1e-6;
            ssr = ssr_s;
            if (stalled) {
                exit_reason = FK_EXIT_STALLED;
                break;
            }
            sparse_gradient_kernel<<<I.grid_for(n), 256, 0, st>>>(S, J, r, I.d_g);
            if (outer_iters == 100) break;
            if (ssr < 1e-8) {
                exit_reason = FK_EXIT_CONVERGED_RESIDUAL;
                break;
            }
            outer_iters++;
        } else {
            lambda *= 2.0;
            push(2);
        }
    }
    SP_CU(cudaMemcpyAsync(free_values, x, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    SP_CU(cudaStreamSynchronize(st));
    if (report) {
        report->exit_reason = exit_reason;
        report->outer_iters = outer_iters;
        report->factorizations = factorizations;
        report->accepted = accepted;
        report->ssr = ssr;
        report->lambda = lambda;
        report->trace_hash = trace;
    }
    return FK_OK;
}

}  // namespace fk
