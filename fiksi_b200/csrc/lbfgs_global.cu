// fk_lbfgs_cta_kernel: L-BFGS with one CTA per sketch and the state in global memory (see lbfgs_global.cuh).
//
// Compiled with -fmad=false: every a*b+c below is two roundings.
#include <cuda_runtime.h>

#include <algorithm>
#include <mutex>

#include "lbfgs_core.cuh"
#include "lbfgs_global.cuh"

namespace fk {

namespace {

constexpr int kLbThreads = 256;
// Products of a sequential sum are formed by the whole CTA this many at a time, then added up by one thread.
constexpr uint32_t kLbChunk = 1024;

// Offsets (doubles) of the state arrays in one CTA's workspace, each on a 256-byte boundary.
struct LbLayout {
    uint64_t x, xs, g, dir, sh, yh, r, J, rho, alpha, total;
};
__host__ __device__ inline LbLayout lbfgs_layout(uint32_t n, uint32_t m, uint32_t jnnz) {
    LbLayout L{};
    uint64_t off = 0;
    auto take = [&](uint64_t count) {
        const uint64_t at = off;
        off += ((count > 0 ? count : 1) + 31) & ~uint64_t(31);
        return at;
    };
    L.x = take(n); L.xs = take(n); L.g = take(n); L.dir = take(n);
    L.sh = take(5ull * n); L.yh = take(5ull * n); L.r = take(m); L.J = take(jnnz); L.rho = take(5); L.alpha = take(5);
    L.total = off;
    return L;
}

struct CtaLbfgsOps {
    const DevProgram& P;
    const LbfgsTables& T;
    const double* vars;
    const double* params;
    uint32_t rows;   // row slots of the evaluation tables (eval_rounds x lanes; kNop rows are skipped)
    double* buf_a;   // [kLbChunk] shared
    double* buf_b;   // [kLbChunk] shared
    double* bcast;   // [2] shared
    __device__ void sync() const { __syncthreads(); }
    __device__ bool leader() const { return threadIdx.x == 0; }
    template <class F>
    __device__ void each(uint32_t cnt, F f) const {
        for (uint32_t i = threadIdx.x; i < cnt; i += blockDim.x) f(i);
    }
    // Chain 1 is added up by thread 0, chain 2 by thread 32 (another warp, so the two dependent chains run side by side).
    __device__ void dot2(const double* a1, const double* b1, uint32_t k1, const double* a2, const double* b2, uint32_t k2, double* o1,
                         double* o2) const {
        const uint32_t tid = threadIdx.x;
        double acc = 0.0;
        const uint32_t kmax = k1 > k2 ? k1 : k2;
        for (uint32_t base = 0; base < kmax; base += kLbChunk) {
            const uint32_t c1 = k1 > base ? min(kLbChunk, k1 - base) : 0u, c2 = k2 > base ? min(kLbChunk, k2 - base) : 0u;
            for (uint32_t i = tid; i < c1; i += blockDim.x) buf_a[i] = a1[base + i] * b1[base + i];
            for (uint32_t i = tid; i < c2; i += blockDim.x) buf_b[i] = a2[base + i] * b2[base + i];
            __syncthreads();
            if (tid == 0) {
#pragma unroll 8
                for (uint32_t i = 0; i < c1; i++) acc += buf_a[i];
            } else if (tid == 32) {
#pragma unroll 8
                for (uint32_t i = 0; i < c2; i++) acc += buf_b[i];
            }
            __syncthreads();
        }
        if (tid == 0) bcast[0] = acc;
        else if (tid == 32) bcast[1] = acc;
        __syncthreads();
        *o1 = bcast[0];
        *o2 = bcast[1];
        __syncthreads();  // (the next sum rewrites bcast)
    }
    __device__ double dot(const double* a, const double* b, uint32_t k) const {
        double o1, o2;
        dot2(a, b, k, nullptr, nullptr, 0u, &o1, &o2);
        return o1;
    }
    __device__ void evaluate(const double* pt, const LbfgsVecs& s) const {
        for (uint32_t row = threadIdx.x; row < rows; row += blockDim.x) eval_row_assign<-1>(P, row, pt, vars, params, s.r, s.J);
        __syncthreads();
        for (uint32_t c = threadIdx.x; c < P.n; c += blockDim.x) s.g[c] = lbfgs_grad_col(T, s.J, s.r, c);
        __syncthreads();
    }
};

__global__ void __launch_bounds__(kLbThreads, 2)
fk_lbfgs_cta_kernel(const DevProgram P, const LbfgsTables T, uint32_t n_sketches, const double* __restrict__ vars_all,
                    const double* __restrict__ params_all, double* __restrict__ free_out, fk_report* __restrict__ reports,
                    double* __restrict__ workspace, unsigned* __restrict__ next) {
    __shared__ double buf_a[kLbChunk], buf_b[kLbChunk], bcast[2];
    __shared__ unsigned s_sketch;
    const LbLayout L = lbfgs_layout(P.n, P.m, P.jnnz);
    double* base = workspace + (uint64_t)blockIdx.x * L.total;
    LbfgsVecs s;
    s.x = base + L.x; s.xs = base + L.xs; s.g = base + L.g; s.dir = base + L.dir; s.sh = base + L.sh; s.yh = base + L.yh;
    s.r = base + L.r; s.J = base + L.J; s.rho = base + L.rho; s.alpha = base + L.alpha;
    const uint32_t rows = P.eval_rounds * (P.tile ? P.tile : 1u);  // (the global sparse path lays its rows out one per lane)
    for (;;) {
        if (threadIdx.x == 0) s_sketch = atomicAdd(next, 1u);
        __syncthreads();
        const uint32_t sketch = s_sketch;
        __syncthreads();  // (s_sketch is rewritten for the next sketch)
        if (sketch >= n_sketches) return;
        const double* vars = vars_all + (size_t)sketch * P.n_vars;
        CtaLbfgsOps ops{P, T, vars, params_all + (size_t)sketch * P.n_expr, rows, buf_a, buf_b, bcast};
        lbfgs_solve(ops, P, vars, s, free_out + (size_t)sketch * P.n, reports + sketch);
    }
}

// Resident CTAs of the kernel on `device` (0: not known), once per device.
uint32_t resident_ctas(int device) {
    static std::mutex mu;
    static uint32_t cache[64] = {};
    if (device < 0 || device >= 64) return 0;
    std::lock_guard<std::mutex> lock(mu);
    if (cache[device] == 0) {
        int per_sm = 0, sms = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fk_lbfgs_cta_kernel, kLbThreads, 0) != cudaSuccess ||
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) {
            cudaGetLastError();
            return 0;
        }
        cache[device] = (uint32_t)std::max(1, per_sm * sms);
    }
    return cache[device];
}

}  // namespace

uint64_t lbfgs_cta_doubles(uint32_t n, uint32_t m, uint32_t jnnz) { return lbfgs_layout(n, m, jnnz).total; }

uint32_t lbfgs_workspace_ctas(const DevProgram& prog, uint32_t capacity) {
    int device = 0;
    if (cudaGetDevice(&device) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    const uint32_t resident = resident_ctas(device);
    if (resident == 0) return 0;
    const uint64_t budget = std::max<uint64_t>(1, (kLbWorkspaceBytes - kLbHeadDoubles * sizeof(double)) /
                                                      (sizeof(double) * lbfgs_cta_doubles(prog.n, prog.m, prog.jnnz)));
    return (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>({(uint64_t)capacity, (uint64_t)resident, budget}));
}

int launch_lbfgs_cta(const DevProgram& prog, const uint32_t* d_jcolptr, const uint32_t* d_jrow, uint32_t n, const double* vars,
                     const double* params, double* free_out, fk_report* reports, double* workspace, uint32_t ctas, void* stream) {
    if (n == 0) return 0;
    if (prog.jnnz > 0x1000000u || ctas == 0) return (int)cudaErrorInvalidConfiguration;  // (row tables: 24-bit positions)
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(workspace, 0, sizeof(unsigned), st);
    if (e != cudaSuccess) return (int)e;
    const uint32_t grid = std::min(n, ctas);
    fk_lbfgs_cta_kernel<<<grid, kLbThreads, 0, st>>>(prog, LbfgsTables{d_jcolptr, d_jrow}, n, vars, params, free_out, reports,
                                                     workspace + kLbHeadDoubles, (unsigned*)workspace);
    return (int)cudaGetLastError();
}

}  // namespace fk
