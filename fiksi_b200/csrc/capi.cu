// extern "C" entry points of libfiksi_b200.so (declared in include/fiksi_b200.h).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <atomic>
#include <cstring>
#include <functional>
#include <list>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/fiksi_b200.h"
#include "analyze.cuh"
#include "lbfgs_global.cuh"
#include "lm_kernels.cuh"
#include "lm_sketch.cuh"
#include "multifrontal.cuh"
#include "single_pass.hpp"
#include "sparse_batch.cuh"
#include "sparse_path.cuh"
#include "symbolic.hpp"
#include "system_batch.cuh"

namespace {

thread_local std::string g_error;

int fail(int code, const std::string& msg) {
    g_error = msg;
    return code;
}
int cuda_fail(cudaError_t e, const char* what) {
    g_error = std::string(what) + ": " + cudaGetErrorString(e);
    return e == cudaErrorMemoryAllocation ? FK_ERR_OOM : FK_ERR_CUDA;
}
#define CU(call)                                           \
    do {                                                   \
        cudaError_t e_ = (call);                           \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call); \
    } while (0)

// Grow-only buffer of T on one device: device memory, or pinned host memory.  reserve(need, alloc) replaces it (the contents are
// lost) by one of `alloc` elements (default `need`, at least one) when it holds fewer than `need` or nothing yet.  Freed on its
// device with its owner.
template <class T>
class GrowBuf {
public:
    explicit GrowBuf(bool pinned = false) : pinned_(pinned) {}
    GrowBuf(const GrowBuf&) = delete;
    GrowBuf& operator=(const GrowBuf&) = delete;
    ~GrowBuf() {
        if (!p_) return;
        cudaSetDevice(device_);
        release();
    }
    bool holds(size_t need) const { return p_ && cap_ >= need; }
    int reserve(size_t need, size_t alloc = 0) {
        if (holds(need)) return FK_OK;
        release();
        const size_t count = std::max<size_t>({need, alloc, 1});
        const cudaError_t e = pinned_ ? cudaMallocHost((void**)&p_, sizeof(T) * count) : cudaMalloc((void**)&p_, sizeof(T) * count);
        if (e != cudaSuccess) {
            p_ = nullptr;
            return cuda_fail(e, pinned_ ? "cudaMallocHost" : "cudaMalloc");
        }
        cudaGetDevice(&device_);
        cap_ = count;
        return FK_OK;
    }
    T* get() const { return p_; }
    operator T*() const { return p_; }

private:
    void release() {
        if (p_) pinned_ ? cudaFreeHost(p_) : cudaFree(p_);
        p_ = nullptr;
        cap_ = 0;
    }
    T* p_ = nullptr;
    size_t cap_ = 0;
    int device_ = 0;
    bool pinned_;
};

// Regions of a staging block one after the other, each at a 256-byte boundary and at least one byte long: put(bytes) returns a
// region's offset, `end` is the size of the block so far.
struct BlockLayout {
    size_t end = 0;
    size_t put(size_t bytes) {
        const size_t o = end;
        end = (end + std::max<size_t>(bytes, 1) + 255) & ~size_t(255);
        return o;
    }
};

int usable_devices() {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// Device arguments of the entry points.  Multi-device calls: n_gpus <= 0 or more than are visible means all visible devices.
int clamp_gpus(int& n_gpus) {
    const int ndev = usable_devices();
    if (ndev == 0) return fail(FK_ERR_NO_DEVICE, "no CUDA device visible; fiksi_b200 has no CPU fallback");
    if (n_gpus <= 0 || n_gpus > ndev) n_gpus = ndev;
    return FK_OK;
}
int check_device(int device) {
    int ndev = 0;
    const int rc = clamp_gpus(ndev);
    if (rc != FK_OK) return rc;
    return device >= 0 && device < ndev ? FK_OK : fail(FK_ERR_INVALID, "device index out of range");
}

// Runs fn(device, lo, hi) on contiguous shares [lo, hi) of n items, one host thread per device, and returns the first failure
// in device order.  n_gpus == 1: the calling thread on its current device (one process per GPU keeps the device it chose).
template <class Fn>
int shard_over_devices(int n_gpus, uint32_t n, const Fn& fn) {
    if (n_gpus == 1) {
        int cur = 0;
        if (cudaGetDevice(&cur) != cudaSuccess) cur = 0;
        return fn(cur, 0u, n);
    }
    std::vector<int> rcs(n_gpus, FK_OK);
    std::vector<std::string> errs(n_gpus);  // (g_error is per thread)
    std::vector<std::thread> pool;
    for (int g = 0; g < n_gpus; g++) {
        const uint32_t lo = (uint32_t)((uint64_t)n * g / n_gpus), hi = (uint32_t)((uint64_t)n * (g + 1) / n_gpus);
        pool.emplace_back([&, g, lo, hi] {
            if (hi > lo && (rcs[g] = fn(g, lo, hi)) != FK_OK) errs[g] = g_error;
        });
    }
    for (auto& th : pool) th.join();
    for (int g = 0; g < n_gpus; g++)
        if (rcs[g] != FK_OK) return fail(rcs[g], errs[g]);
    return FK_OK;
}

// The per-device state in `slots` for `device`, created empty on first use, under `mu`.
template <class T>
T* device_slot(std::mutex& mu, std::map<int, std::unique_ptr<T>>& slots, int device) {
    std::lock_guard<std::mutex> lock(mu);
    std::unique_ptr<T>& p = slots[device];
    if (!p) p.reset(new T());
    return p.get();
}

// Packs the topology tables into one device allocation and fills the DevProgram view.
struct DeviceProgram {
    int device = -1;
    void* buf = nullptr;
    fk::DevProgram view{};
    const uint32_t *jcolptr = nullptr, *jrow = nullptr;  // CSC of the Jacobian (L-BFGS)
    std::unique_ptr<fk::SkProgram> sketch;               // parameter block of the sketch-per-thread LM kernel
    std::unique_ptr<fk::SparseBatchProgram> sparse_batch;  // path 2: tables of the one-CTA-per-sketch supernodal LM kernel, built
                                                           // by the first caller that launches LM (fk_topology::program_for)
    ~DeviceProgram() {
        if (buf) {
            cudaSetDevice(device);
            cudaFree(buf);
        }
    }
};

// Host tables packed into one device allocation: add() copies a vector in at the next 16-byte boundary (room for at least one
// element) and returns its offset, upload() makes the allocation, at() points into it.
struct TablePack {
    std::vector<unsigned char> host;
    const unsigned char* base = nullptr;
    template <class V>
    size_t add(const V& vec) {
        using T = typename V::value_type;
        const size_t at = (host.size() + 15) & ~size_t(15);
        host.resize(at + std::max<size_t>(vec.size(), 1) * sizeof(T), 0);
        if (!vec.empty()) std::memcpy(host.data() + at, vec.data(), vec.size() * sizeof(T));
        return at;
    }
    // One cudaMalloc (16 zero bytes behind the last table) into *buf, which the caller frees also after an error, and one copy on
    // `stream` (0: the legacy default stream), complete on return.  The caller has selected the device.
    int upload(cudaStream_t stream, void** buf) {
        host.resize(host.size() + 16, 0);
        CU(cudaMalloc(buf, host.size()));
        base = (const unsigned char*)*buf;
        CU(cudaMemcpyAsync(*buf, host.data(), host.size(), cudaMemcpyHostToDevice, stream));
        CU(cudaStreamSynchronize(stream));
        return FK_OK;
    }
    template <class T>
    const T* at(size_t off) const { return (const T*)(base + off); }
};

int upload_program(const fk::Topology& t, int device, DeviceProgram& out) {
    CU(cudaSetDevice(device));
    TablePack pk;
    const fk::Topology::Tables& tb = t.tab;
    std::vector<uint32_t> jcolptr(t.n_free + 1), jrow(t.jac_nnz);  // CSC of the Jacobian without damping rows (L-BFGS gradient)
    for (uint32_t c = 0; c <= t.n_free; c++) jcolptr[c] = t.aug_colptr[c] - c;
    for (uint32_t c = 0; c < t.n_free; c++)
        for (uint32_t q = t.aug_colptr[c]; q + 1 < t.aug_colptr[c + 1]; q++) jrow[q - c] = t.aug_rowidx[q];
    const size_t o_jcp = pk.add(jcolptr), o_jrow = pk.add(jrow);
    size_t o_free = pk.add(t.free_vars), o_rh = pk.add(tb.row_hdr), o_rs = pk.add(tb.row_slots),
           o_af = pk.add(tb.a_flags), o_ao = pk.add(tb.a_ops), o_ad = pk.add(tb.a_dst),
           o_gf = pk.add(tb.g_flags), o_go = pk.add(tb.g_ops), o_gd = pk.add(tb.g_dst),
           o_fs = pk.add(tb.f_steps), o_fo = pk.add(tb.f_ops), o_ss = pk.add(tb.s_steps), o_so = pk.add(tb.s_ops),
           o_bs = pk.add(tb.b_steps), o_bo = pk.add(tb.b_ops);
    const size_t o_sk = (t.sk.ok && fk::sk_fits(t.sk.entries, t.sk.tab.size())) ? pk.add(t.sk.tab) : SIZE_MAX;
    out.device = device;
    const int rc = pk.upload(0, &out.buf);
    if (rc != FK_OK) return rc;
    fk::DevProgram& v = out.view;
    v.n_vars = t.n_vars; v.n_expr = t.n_expr; v.n = t.n_free; v.m = t.n_rows;
    v.jnnz = t.jac_nnz; v.lnnz = (uint32_t)t.l_rowidx.size(); v.tile = t.tile; v.uniform_kind = tb.uniform_kind;
    v.eval_rounds = tb.eval_rounds; v.a_nsteps = tb.a_nsteps; v.g_nsteps = tb.g_nsteps;
    v.f_nsteps = tb.f_nsteps; v.s_nsteps = tb.s_nsteps; v.b_nsteps = tb.b_nsteps;
    v.free_vars = pk.at<uint32_t>(o_free);
    v.row_hdr = pk.at<uint32_t>(o_rh); v.row_slots = pk.at<uint2>(o_rs);
    v.a_flags = pk.at<uint32_t>(o_af); v.a_ops = pk.at<uint32_t>(o_ao); v.a_dst = pk.at<uint32_t>(o_ad);
    v.g_flags = pk.at<uint32_t>(o_gf); v.g_ops = pk.at<uint32_t>(o_go); v.g_dst = pk.at<uint32_t>(o_gd);
    v.f_steps = pk.at<uint32_t>(o_fs); v.f_ops = pk.at<uint2>(o_fo);
    v.s_steps = pk.at<uint2>(o_ss); v.s_ops = pk.at<uint32_t>(o_so);
    v.b_steps = pk.at<uint2>(o_bs); v.b_ops = pk.at<uint32_t>(o_bo);
    out.jcolptr = pk.at<uint32_t>(o_jcp); out.jrow = pk.at<uint32_t>(o_jrow);
    v.sketch_prog = nullptr;
    if (o_sk != SIZE_MAX) {
        const fk::Topology::SketchTables& k = t.sk;
        out.sketch.reset(new fk::SkProgram());
        fk::SkProgram& p = *out.sketch;
        std::memset(&p, 0, sizeof(p));
        p.n_vars = t.n_vars; p.n_expr = t.n_expr; p.n = t.n_free; p.m = t.n_rows; p.lnnz = (uint32_t)t.l_rowidx.size(); p.entries = k.entries;
        p.xa = k.xa; p.xb = k.xb; p.w = k.w; p.f = k.f; p.fx = k.fx; p.pr = k.pr; p.nfix = k.nfix; p.npar = k.npar;
        p.off_free = k.off_free; p.off_fix = k.off_fix; p.off_par = k.off_par;
        p.off_eval = k.off_eval; p.off_factor = k.off_factor; p.off_back = k.off_back;
        p.tab_words = (uint32_t)k.tab.size();
        p.tab = pk.at<uint32_t>(o_sk);
        v.sketch_prog = out.sketch.get();
    }
    return FK_OK;
}

// The batched solve kernels (solve_kernel picks one for a topology and an optimizer): LM -- on the global sparse path the
// one-CTA-per-sketch kernel over the supernodal tree, launch_batch_lm's tile / sketch-per-thread kernels otherwise --, the L-BFGS
// tile kernel (state in shared memory) and the L-BFGS CTA kernel (state in global memory).
enum SolveKernel { kSolveLm, kSolveLbfgsTile, kSolveLbfgsCta };

// The grow-only workspaces of the solve kernels that need one: the sparse batch LM kernel and the L-BFGS CTA kernel.  A workspace
// serves one stream: two launches that may run at the same time need two.
struct SolveWorkspace {
    GrowBuf<double> lm, lbfgs;
    // Room for one launch of `kernel` over n sketches of `full`: per-CTA workspaces for min(n, resident CTAs) CTAs, within the
    // kernel's workspace limit (*ctas: that CTA count).  Nothing when it already has the room, or for a kernel without workspace.
    int reserve(const DeviceProgram& full, SolveKernel kernel, uint32_t n, uint32_t* ctas = nullptr) {
        if (kernel == kSolveLm && full.sparse_batch) {
            const uint32_t c = full.sparse_batch->workspace_ctas(n);
            if (ctas) *ctas = c;
            return lm.reserve(full.sparse_batch->workspace_doubles(c));
        }
        if (kernel == kSolveLbfgsCta) {
            const uint32_t c = fk::lbfgs_workspace_ctas(full.view, n);
            if (c == 0) return fail(FK_ERR_CUDA, "occupancy query of fk_lbfgs_cta_kernel failed");
            if (ctas) *ctas = c;
            return lbfgs.reserve(fk::lbfgs_workspace_doubles(full.view, c));
        }
        return FK_OK;
    }
};

// One launch of `kernel` over n sketches of `full` (vars[n][n_vars], params[n][n_expr] -> out[n][n_free], reps[n]) on st, its
// workspace reserved in ws first.
int solve_launch(const DeviceProgram& full, SolveKernel kernel, uint32_t n, const double* vars, const double* params, double* out,
                 fk_report* reps, SolveWorkspace& ws, cudaStream_t st) {
    if (kernel == kSolveLbfgsCta && n == 0) return FK_OK;
    uint32_t ctas = 0;
    const int rc = ws.reserve(full, kernel, n, &ctas);
    if (rc != FK_OK) return rc;
    int e;
    switch (kernel) {
        case kSolveLm:
            e = full.sparse_batch ? full.sparse_batch->launch(n, vars, params, out, reps, ws.lm, ctas, st)
                                  : fk::launch_batch_lm(full.view, n, vars, params, out, reps, st);
            return e != 0 ? cuda_fail((cudaError_t)e, "launch batched LM kernel") : FK_OK;
        case kSolveLbfgsTile:
            e = fk::launch_batch_lbfgs(full.view, full.jcolptr, full.jrow, n, vars, params, out, reps, st);
            if (e == (int)cudaErrorInvalidConfiguration) return fail(FK_ERR_TOO_LARGE, "the L-BFGS state of one sketch does not fit the tile path");
            return e != 0 ? cuda_fail((cudaError_t)e, "launch fk_batch_lbfgs_kernel") : FK_OK;
        default:
            e = fk::launch_lbfgs_cta(full.view, full.jcolptr, full.jrow, n, vars, params, out, reps, ws.lbfgs, ctas, st);
            if (e == (int)cudaErrorInvalidConfiguration) return fail(FK_ERR_TOO_LARGE, "more than 2^24 Jacobian entries");
            return e != 0 ? cuda_fail((cudaError_t)e, "launch fk_lbfgs_cta_kernel") : FK_OK;
    }
}

// One analyze launch over n sketches (kinds, slot table, vars[n][n_vars], params[n][n_expr] -> out[n][n_expr]) on `device`'s
// stream st: the kernel choose_analyze picks for n, with its workspace in the grow-only ws.  The stream is synchronised before a
// smaller workspace is freed, since an earlier launch on it may still use that one.
int analyze_launch(uint32_t n_vars, uint32_t n_expr, const uint8_t* kinds, const uint32_t* slot, uint32_t n, const double* vars,
                   const double* params, uint8_t* out, int device, GrowBuf<double>& ws, cudaStream_t st) {
    fk::AnalyzePlan plan;
    std::string err;
    int rc = fk::choose_analyze(n_vars, n_expr, n, device, &plan, &err);
    if (rc != FK_OK) return fail(rc, err);
    const size_t need = plan.workspace_bytes() / sizeof(double);  // (within fk::kAnWorkspaceBytes)
    if (need && !ws.holds(need)) {
        CU(cudaStreamSynchronize(st));
        if ((rc = ws.reserve(need)) != FK_OK) return rc;
    }
    const bool warp = plan.kernel == fk::kAnWarp;
    const int e = warp ? fk::launch_batch_analyze(n_vars, n_expr, kinds, slot, n, vars, params, out, st)
                       : fk::launch_analyze(plan, n_vars, n_expr, kinds, slot, n, vars, params, out, ws, st);
    return e != 0 ? cuda_fail((cudaError_t)e, warp ? "launch fk_batch_analyze_kernel" : "launch fk_analyze_cta_kernel") : FK_OK;
}

}  // namespace

struct fk_batch_plan;
// Per-device staging pipeline of the host-buffer batch calls: kStreams plans + streams, reused across calls.
struct DevicePipeline {
// (eight chunks in flight: a chunk's kernel lasts one LM solve however small the chunk is, so with three the copies of
// small chunks could not keep the device busy; bench truss end to end 56.2 -> 59.0 M sketches/s with 16 chunks.  Swept on
// B200 with tools/e2e_sweep.py: 4 / 6 / 8 / 16 / 32 streams x 8..32 chunks all end between 1.10 and 1.19 ms per call of
// 65,536 trusses against 0.905 ms for the kernel alone)
#ifndef FK_PIPELINE_STREAMS
#define FK_PIPELINE_STREAMS 8
#endif
    static constexpr uint32_t kStreams = FK_PIPELINE_STREAMS;
    std::mutex mu;
    int device = -1;
    uint32_t chunk = 0;
    fk_batch_plan* plans[kStreams] = {};
    cudaStream_t streams[kStreams] = {};
    // small requests (one sketch, a handful): one pinned staging block, one device block, one copy each way
    static constexpr size_t kSmallBytes = 64 * 1024;
    GrowBuf<unsigned char> small_h{true}, small_d;
    cudaStream_t small_stream = nullptr;
    SolveWorkspace small_ws;
    bool plans_lm = false;  // the plans were created for LM too
    cudaEvent_t shared_param_ev = nullptr;  // fk_batch_system_solve with one parameter row for all sketches: its upload, once per call
    // Every call on the chunk pipeline takes a token.  Its parity picks the call's copy of the shared parameter row and the events
    // recorded behind its last chunk on every stream (the _begin / _wait halves: up to two calls in flight).
    uint64_t next_token = 1;
    cudaEvent_t done_ev[2][kStreams] = {};
    double* d_shared_param[2] = {nullptr, nullptr};
    uint32_t shared_param_cap = 0;
    void release();
    ~DevicePipeline() { release(); }
};

// Device tables and grow-only device buffers of fk_batch_analyze for one (topology, device).
struct AnalyzePool {
    int device = -1;
    std::mutex mu;
    void* d_tables = nullptr;
    const uint8_t* d_kind = nullptr;
    const uint32_t* d_slot = nullptr;
    GrowBuf<double> d_vars, d_param;
    GrowBuf<uint8_t> d_out;
    GrowBuf<double> ws;  // workspace of the global-memory kernels
    cudaStream_t stream = nullptr;
    ~AnalyzePool() {
        if (device >= 0) cudaSetDevice(device);
        cudaFree(d_tables);
        if (stream) cudaStreamDestroy(stream);
    }
};

// Device tables of assemble::solve's pre-processing for one (topology, device): expression kinds, the variables that
// draw from the solve's generator (ascending) and the draws themselves (fiksi/src/rand.rs:24-39, two per variable).
struct PrepareTables {
    int device = -1;
    std::vector<uint32_t> perturb_vars;
    uint32_t seed = 0;
    void* d_tables = nullptr;
    const uint8_t* d_kind = nullptr;
    const uint32_t* d_perturb = nullptr;
    const double* d_draws = nullptr;
    const uint32_t* d_free_draw = nullptr;  // sketch kernel's raw mode: draw index per free column / per fixed variable the rows read
    const uint32_t* d_fix_draw = nullptr;
    ~PrepareTables() {
        if (device >= 0) cudaSetDevice(device);
        cudaFree(d_tables);
    }
};

struct fk_topology {
    fk::Topology t;
    std::mutex mu;
    std::map<int, std::unique_ptr<DeviceProgram>> programs;
    std::map<int, std::unique_ptr<DevicePipeline>> pipelines;
    std::map<int, std::unique_ptr<fk::SparseSolver>> sparse;  // path 2: one solver per device
    std::mutex sparse_mu;               // a SparseSolver owns one set of work vectors and CUDA graphs: one solve at a time
    std::map<int, std::unique_ptr<struct AnalyzePool>> analyze_pools;  // fk_batch_analyze: tables + grow-only buffers
    std::map<int, std::unique_ptr<struct PrepareTables>> prepare_tables;  // fk_batch_system_solve: kinds, perturbation list, draws
    std::unique_ptr<fk_topology> latency_twin;  // same topology with 32 lanes per sketch: single-system solves
    bool twin_tried = false;
    std::mutex sp_mu;                   // SinglePass plan: one sub-topology per strongly connected set
    bool sp_planned = false;
    std::vector<fk_topology*> sp_subs;
    int sb_fit = 1;                     // path 2: FK_OK when the sparse batch kernel takes the topology (1: not yet analysed)
    std::string sb_err;
    ~fk_topology();

    int sparse_for(int device, fk::SparseSolver** out, std::string* err) {
        std::lock_guard<std::mutex> lock(mu);
        auto& p = sparse[device];
        if (!p) {
            std::unique_ptr<fk::SparseSolver> s(new fk::SparseSolver());
            int rc = s->init(t, device, err);
            if (rc != FK_OK) return rc;
            p = std::move(s);
        }
        *out = p.get();
        return FK_OK;
    }

    // This topology with op tables for 32 lanes per system (single-system solves and heterogeneous batches): itself when
    // its batch-oriented lane count is already 32, else a twin that shares the symbolic analysis and re-packs the tables.
    fk_topology* lanes32() {
        if (t.path != 0 || t.tile == 32) return this;
        std::lock_guard<std::mutex> lock(mu);
        if (!twin_tried) {
            twin_tried = true;
            static const bool off = std::getenv("FK_NO_LATENCY_TWIN") != nullptr;
            if (!off) {
                std::unique_ptr<fk_topology> tw(new (std::nothrow) fk_topology());
                if (tw) {
                    tw->t = t;
                    tw->t.tile = 32;
                    if (tw->t.build_tables() == FK_OK) latency_twin = std::move(tw);
                }
            }
        }
        return latency_twin ? latency_twin.get() : this;
    }

    DevicePipeline* pipeline_for(int device) {
        std::lock_guard<std::mutex> lock(mu);
        auto& p = pipelines[device];
        if (!p) {
            p.reset(new DevicePipeline());
            p->device = device;
        }
        return p.get();
    }

    // Path 2: whether the sparse batch LM kernel takes the topology (largest front), host analysis once per topology.
    int sb_check() {
        std::lock_guard<std::mutex> lock(mu);
        if (sb_fit == 1) sb_fit = fk::sparse_batch_fits(t, nullptr, &sb_err);
        return sb_fit == FK_OK ? FK_OK : fail(sb_fit, sb_err);
    }

    // Device tables on `device`.  lm: the caller launches LM, which on the global sparse path also needs the tables of the
    // sparse batch kernel (refused above its front limit); L-BFGS needs none of them.
    int program_for(int device, const fk::DevProgram** out, const DeviceProgram** full = nullptr, bool lm = true) {
        if (lm && t.path == 2) {
            const int rc = sb_check();
            if (rc != FK_OK) return rc;
        }
        std::lock_guard<std::mutex> lock(mu);
        auto it = programs.find(device);
        if (it == programs.end()) {
            std::unique_ptr<DeviceProgram> p(new DeviceProgram());
            int rc = upload_program(t, device, *p);
            if (rc != FK_OK) return rc;
            it = programs.emplace(device, std::move(p)).first;
        }
        DeviceProgram& p = *it->second;
        if (lm && t.path == 2 && !p.sparse_batch) {
            std::string err;
            std::unique_ptr<fk::SparseBatchProgram> sb(new fk::SparseBatchProgram());
            const int rc = sb->init(t, p.view, device, &err);
            if (rc != FK_OK) return fail(rc, err);
            p.sparse_batch = std::move(sb);
        }
        *out = &p.view;
        if (full) *full = &p;
        return FK_OK;
    }
};

struct fk_batch_plan {
    fk_topology* topo = nullptr;
    int device = 0;
    uint32_t capacity = 0, n = 0;
    const fk::DevProgram* prog = nullptr;
    const DeviceProgram* full = nullptr;
    double *d_vars = nullptr, *d_params = nullptr, *d_out = nullptr, *d_er = nullptr, *d_ej = nullptr;
    fk_report* d_rep = nullptr;
    SolveWorkspace ws;
    bool lm = true;          // LM may run on the plan (false: the L-BFGS calls' internal plans, which skip its tables)
    double *d_raw_vars = nullptr, *d_raw_param = nullptr, *d_scales = nullptr;  // fk_batch_system_solve: unscaled input, scale per sketch
    uint64_t launches = 0;
    ~fk_batch_plan() {
        cudaSetDevice(device);
        cudaFree(d_vars); cudaFree(d_params); cudaFree(d_out); cudaFree(d_er); cudaFree(d_ej); cudaFree(d_rep);
        cudaFree(d_raw_vars); cudaFree(d_raw_param); cudaFree(d_scales);
    }
};

fk_topology::~fk_topology() {
    for (fk_topology* s : sp_subs) delete s;
}

void DevicePipeline::release() {
    if (device >= 0) cudaSetDevice(device);
    for (uint32_t s = 0; s < kStreams; s++) {
        if (streams[s]) cudaStreamDestroy(streams[s]);
        streams[s] = nullptr;
        delete plans[s];
        plans[s] = nullptr;
    }
    chunk = 0;
    if (small_stream) cudaStreamDestroy(small_stream);
    small_stream = nullptr;
    plans_lm = false;
    if (shared_param_ev) cudaEventDestroy(shared_param_ev);
    shared_param_ev = nullptr;
    for (int a = 0; a < 2; a++) {
        for (uint32_t k = 0; k < kStreams; k++) {
            if (done_ev[a][k]) cudaEventDestroy(done_ev[a][k]);
            done_ev[a][k] = nullptr;
        }
        if (d_shared_param[a]) cudaFree(d_shared_param[a]);
        d_shared_param[a] = nullptr;
    }
    shared_param_cap = 0;
}

extern "C" {

int fk_version(void) { return 100; }
const char* fk_last_error(void) { return g_error.c_str(); }
int fk_device_count(void) { return usable_devices(); }

int fk_topology_create(const fk_problem* problem, fk_topology** out) {
    if (!problem || !out) return fail(FK_ERR_INVALID, "null argument");
    std::unique_ptr<fk_topology> t(new (std::nothrow) fk_topology());
    if (!t) return fail(FK_ERR_OOM, "host allocation failed");
    int rc;
    try {
        rc = t->t.build(*problem);
    } catch (const std::bad_alloc&) {
        return fail(FK_ERR_OOM, "host allocation failed in symbolic analysis");
    }
    if (rc != FK_OK) return fail(rc, t->t.error);
    *out = t.release();
    return FK_OK;
}

void fk_topology_destroy(fk_topology* topo) { delete topo; }

int fk_topology_info_get(const fk_topology* topo, fk_topology_info* info) {
    if (!topo || !info) return fail(FK_ERR_INVALID, "null argument");
    topo->t.fill_info(info);
    return FK_OK;
}

int fk_topology_symbolic(const fk_topology* topo, uint32_t* aug_colptr, uint32_t* aug_rowidx, int32_t* colamd_perm,
                         int32_t* etree_parent, uint32_t* r_colptr, uint32_t* r_rowidx) {
    if (!topo) return fail(FK_ERR_INVALID, "null topology");
    const fk::Topology& t = topo->t;
    auto copy = [](auto* dst, const auto& v) {
        if (dst && !v.empty()) std::memcpy(dst, v.data(), v.size() * sizeof(v[0]));
    };
    copy(aug_colptr, t.aug_colptr); copy(aug_rowidx, t.aug_rowidx); copy(colamd_perm, t.perm);
    copy(etree_parent, t.parent); copy(r_colptr, t.r_colptr); copy(r_rowidx, t.r_rowidx);
    return FK_OK;
}

int fk_symbolic(const fk_problem* problem, uint32_t* aug_colptr, uint32_t* aug_rowidx, int32_t* colamd_perm,
                int32_t* etree_parent, uint32_t* r_colptr, uint32_t* r_rowidx) {
    fk_topology* t = nullptr;
    int rc = fk_topology_create(problem, &t);
    if (rc != FK_OK) return rc;
    rc = fk_topology_symbolic(t, aug_colptr, aug_rowidx, colamd_perm, etree_parent, r_colptr, r_rowidx);
    fk_topology_destroy(t);
    return rc;
}

int fk_topology_supernodal(const fk_topology* topo, fk_supernodal_info* info, uint32_t* sn_first, uint32_t* front,
                           int32_t* sn_parent, uint32_t* rows, uint32_t* rel, uint8_t* big, uint32_t* level, uint32_t* tasks,
                           uint32_t* launches) {
    if (!topo || !info) return fail(FK_ERR_INVALID, "null argument");
    fk::Multifrontal mf;
    std::string err;
    try {
        if (mf.build_symbolic(topo->t, &err) != cudaSuccess) return fail(FK_ERR_TOO_LARGE, err);
    } catch (const std::bad_alloc&) {
        return fail(FK_ERR_OOM, "host allocation failed in the supernodal analysis");
    }
    const fk::MfSymbolic& y = mf.sym;
    const auto seq = mf.factor_launches();
    info->n_supernodes = y.S; info->n_small_subtrees = y.nsub; info->n_big = y.nbig; info->n_levels = y.nlevels;
    info->max_front = y.max_front; info->n_tasks = (uint32_t)(y.tasks.size() / 4); info->n_launches = (uint32_t)seq.size(); info->pad0 = 0;
    info->rows_total = y.rows.size(); info->rel_total = y.rel.size(); info->panel_doubles = y.pan_total; info->update_doubles = y.upd_total;
    auto copy = [](auto* dst, const auto& v) {
        if (dst && !v.empty()) std::memcpy(dst, v.data(), v.size() * sizeof(v[0]));
    };
    if (sn_first) {
        copy(sn_first, y.c0);
        sn_first[y.S] = y.n;
    }
    copy(front, y.f); copy(sn_parent, y.sparent); copy(rows, y.rows); copy(rel, y.rel); copy(big, y.big); copy(level, y.level);
    copy(tasks, y.tasks);
    if (launches)
        for (size_t k = 0; k < seq.size(); k++) {
            launches[3 * k] = (uint32_t)seq[k].kind; launches[3 * k + 1] = seq[k].first; launches[3 * k + 2] = seq[k].count;
        }
    return FK_OK;
}

// ---- Decomposer::SinglePass on a uniform batch ---------------------------------------------------------
// The plan (one sub-topology per strongly connected set) is built once per topology and cached.  Variables
// and parameters of a shard stay resident on its device for the whole pass: per set one batched LM launch over
// all sketches and one scatter of the solved values back into the variable rows (assemble/mod.rs:201-208).
static int single_pass_plan_for(fk_topology* topo, const std::vector<fk_topology*>** out) {
    std::lock_guard<std::mutex> lock(topo->sp_mu);
    if (!topo->sp_planned) {
        const fk::Topology& t = topo->t;
        std::vector<std::vector<uint32_t>> var_exprs(t.n_vars), expr_vars(t.n_expr);
        for (uint32_t e = 0; e < t.n_expr; e++) {
            uint32_t sv[8];
            const int a = fk::expand_slots(t.kind[e], &t.idx[4 * (size_t)e], sv);
            expr_vars[e].assign(sv, sv + a);
            for (int k = 0; k < a; k++) var_exprs[sv[k]].push_back(e);
        }
        fk::SinglePassPlanner planner(var_exprs, expr_vars);
        const std::vector<fk::SinglePassStep> plan = planner.plan(t.free_vars);
        std::vector<fk_topology*> subs;
        for (const fk::SinglePassStep& step : plan) {
            fk_problem p{};
            p.n_vars = t.n_vars; p.n_expr = t.n_expr; p.kind = t.kind.data(); p.idx = t.idx.data();
            p.n_free = (uint32_t)step.free_variables.size(); p.free_vars = step.free_variables.data();
            p.n_rows = (uint32_t)step.expressions.size(); p.rows = step.expressions.data();
            fk_topology* sub = nullptr;
            int rc = fk_topology_create(&p, &sub);
            if (rc == FK_OK && sub->t.path == 2) {
                fk_topology_destroy(sub);
                rc = fail(FK_ERR_TOO_LARGE, "a strongly connected set needs the global sparse path; use fk_system_solve_opts");
            }
            if (rc != FK_OK) {
                for (fk_topology* s : subs) fk_topology_destroy(s);
                return rc;
            }
            subs.push_back(sub);
        }
        topo->sp_subs = std::move(subs);
        topo->sp_planned = true;
    }
    *out = &topo->sp_subs;
    return FK_OK;
}

static int single_pass_device_range(fk_topology* topo, const std::vector<fk_topology*>& subs, int device, uint32_t lo, uint32_t hi,
                                    double* vars, const double* param, fk_report* reports) {
    const fk::Topology& t = topo->t;
    const size_t steps = subs.size();
    uint32_t max_free = 1;
    for (const fk_topology* s : subs) max_free = std::max(max_free, s->t.n_free);
    CU(cudaSetDevice(device));
    // bound the resident set of one chunk to ~8 GiB
    const size_t per_sketch = sizeof(double) * ((size_t)t.n_vars + t.n_expr + max_free) + 2 * sizeof(fk_report) * std::max<size_t>(1, steps);
    const uint32_t chunk = (uint32_t)std::min<uint64_t>(hi - lo, std::max<uint64_t>(1, (8ull << 30) / per_sketch));
    cudaStream_t stream = nullptr;
    CU(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    const std::unique_ptr<CUstream_st, cudaError_t (*)(cudaStream_t)> own_stream(stream, cudaStreamDestroy);
    GrowBuf<double> d_vars, d_params, d_out;
    GrowBuf<fk_report> d_rep, d_rep_t;
    SolveWorkspace ws;
    int rc = d_vars.reserve((size_t)chunk * t.n_vars);
    if (rc == FK_OK) rc = d_params.reserve((size_t)chunk * t.n_expr);
    if (rc == FK_OK) rc = d_out.reserve((size_t)chunk * max_free);
    if (rc == FK_OK) rc = d_rep.reserve((size_t)chunk * steps);
    if (rc == FK_OK && reports) rc = d_rep_t.reserve((size_t)chunk * steps);
    std::vector<const DeviceProgram*> full(steps, nullptr);
    for (size_t st = 0; st < steps && rc == FK_OK; st++) {
        const fk::DevProgram* v = nullptr;
        rc = subs[st]->program_for(device, &v, &full[st]);
    }
    if (rc != FK_OK) return rc;
    for (uint32_t at = lo; at < hi; at += chunk) {
        const uint32_t cnt = std::min(chunk, hi - at);
        CU(cudaMemcpyAsync(d_vars, vars + (size_t)at * t.n_vars, sizeof(double) * (size_t)cnt * t.n_vars, cudaMemcpyHostToDevice, stream));
        if (t.n_expr) CU(cudaMemcpyAsync(d_params, param + (size_t)at * t.n_expr, sizeof(double) * (size_t)cnt * t.n_expr, cudaMemcpyHostToDevice, stream));
        for (size_t st = 0; st < steps; st++) {
            const fk::DevProgram& v = full[st]->view;
            if ((rc = solve_launch(*full[st], kSolveLm, cnt, d_vars, d_params, d_out, d_rep + st * (size_t)cnt, ws, stream)) != FK_OK) return rc;
            const int e = fk::launch_scatter_free(v.free_vars, v.n, t.n_vars, cnt, d_out, d_vars, stream);
            if (e != 0) return cuda_fail((cudaError_t)e, "launch SinglePass set");
        }
        CU(cudaMemcpyAsync(vars + (size_t)at * t.n_vars, d_vars, sizeof(double) * (size_t)cnt * t.n_vars, cudaMemcpyDeviceToHost, stream));
        if (reports && steps) {
            const int e = fk::launch_transpose_reports(d_rep, d_rep_t, cnt, (uint32_t)steps, stream);
            if (e != 0) return cuda_fail((cudaError_t)e, "launch fk_transpose_reports_kernel");
            CU(cudaMemcpyAsync(reports + (size_t)at * steps, d_rep_t, sizeof(fk_report) * (size_t)cnt * steps, cudaMemcpyDeviceToHost, stream));
        }
        CU(cudaStreamSynchronize(stream));
    }
    return FK_OK;
}

int fk_batch_solve_single_pass(const fk_topology* topo_c, uint32_t n, double* vars, const double* param, fk_report* reports,
                               uint32_t* n_steps, int n_gpus) {
    fk_topology* topo = const_cast<fk_topology*>(topo_c);
    if (!topo || (n && (!vars || (!param && topo->t.n_expr)))) return fail(FK_ERR_INVALID, "null argument");
    const std::vector<fk_topology*>* subs = nullptr;
    int rc = single_pass_plan_for(topo, &subs);
    if (rc != FK_OK) return rc;
    if (n_steps) *n_steps = (uint32_t)subs->size();
    if (n == 0) return FK_OK;
    if ((rc = clamp_gpus(n_gpus)) != FK_OK) return rc;
    return shard_over_devices(n_gpus, n, [&](int device, uint32_t lo, uint32_t hi) {
        return single_pass_device_range(topo, *subs, device, lo, hi, vars, param, reports);
    });
}

// ---- L-BFGS on a uniform batch -------------------------------------------------------------------
static int run_device_range(fk_topology* topo, int device, uint32_t lo, uint32_t hi, const double* vars, const double* param,
                            double* free_out, fk_report* reports, int optimizer = 0, uint64_t* token = nullptr);

// The L-BFGS kernel of a topology, chosen in this one place: 0 the tile kernel (state in shared memory) for every topology it
// takes, 1 the CTA kernel (state in global memory) otherwise.  Host only.
static int choose_lbfgs(const fk_topology* topo, uint32_t n_sketches) {
    (void)n_sketches;  // (the choice depends on the topology alone)
    const fk::Topology& t = topo->t;
    return t.path == 0 && fk::batch_lbfgs_tile_fits(t.n_free, t.n_rows, t.jac_nnz, t.tile) ? 0 : 1;
}

// The batched solve kernel of n sketches of a topology: optimizer 0 LM, 1 L-BFGS with the kernel of choose_lbfgs.
static SolveKernel solve_kernel(const fk_topology* topo, int optimizer, uint32_t n) {
    return optimizer == 0 ? kSolveLm : choose_lbfgs(topo, n) == 0 ? kSolveLbfgsTile : kSolveLbfgsCta;
}

int fk_batch_solve_lbfgs(const fk_topology* topo_c, int device, uint32_t n, const double* vars, const double* param, double* free_out,
                         fk_report* reports) {
    if (!topo_c) return fail(FK_ERR_INVALID, "null topology");
    if (n == 0) return FK_OK;
    if (!vars || !free_out || !reports || (!param && topo_c->t.n_expr)) return fail(FK_ERR_INVALID, "null buffer");
    if (topo_c->t.path != 0) return fail(FK_ERR_TOO_LARGE, "L-BFGS is built for the shared-memory tile paths only");
    if (choose_lbfgs(topo_c, n) != 0) return fail(FK_ERR_TOO_LARGE, "the L-BFGS state of one sketch does not fit the tile path");
    const int rc = check_device(device);
    if (rc != FK_OK) return rc;
    // same pooled plans / streams / pinned staging as the LM entry (no allocation per call)
    return run_device_range(const_cast<fk_topology*>(topo_c), device, 0, n, vars, param, free_out, reports, 1);
}

// ---- System::analyze on a batch -----------------------------------------------------------------
int fk_batch_analyze(const fk_topology* topo_c, int device, uint32_t n, const double* vars, const double* param, uint8_t* independent) {
    fk_topology* topo = const_cast<fk_topology*>(topo_c);
    if (!topo || (n && (!vars || !independent || (!param && topo->t.n_expr)))) return fail(FK_ERR_INVALID, "null argument");
    const int rc = check_device(device);
    if (rc != FK_OK) return rc;
    const fk::Topology& t = topo->t;
    if (n == 0 || t.n_expr == 0) return FK_OK;
    CU(cudaSetDevice(device));
    fk::AnalyzePlan plan;
    std::string err;
    const int prc = fk::choose_analyze(t.n_vars, t.n_expr, n, device, &plan, &err);  // the limit rule, before any allocation
    if (prc != FK_OK) return fail(prc, err);
    AnalyzePool* pool = device_slot(topo->mu, topo->analyze_pools, device);
    std::lock_guard<std::mutex> lock(pool->mu);
    if (pool->device < 0) {  // tables: once per (topology, device)
        std::vector<uint32_t> slot_var((size_t)t.n_expr * 8, 0);
        for (uint32_t e = 0; e < t.n_expr; e++) {
            uint32_t sv[8];
            const int a = fk::expand_slots(t.kind[e], &t.idx[4 * (size_t)e], sv);
            for (int k = 0; k < a; k++) slot_var[(size_t)e * 8 + k] = sv[k];
        }
        pool->device = device;
        CU(cudaStreamCreateWithFlags(&pool->stream, cudaStreamNonBlocking));
        TablePack pk;
        const size_t o_kind = pk.add(t.kind), o_slot = pk.add(slot_var);
        const int rc = pk.upload(pool->stream, &pool->d_tables);
        if (rc != FK_OK) return rc;
        pool->d_kind = pk.at<uint8_t>(o_kind);
        pool->d_slot = pk.at<uint32_t>(o_slot);
    }
    const size_t cap = std::max<uint32_t>(n, 1024), nv = std::max<uint32_t>(t.n_vars, 1);  // (grow-only: rows for at least cap sketches)
    int grc = pool->d_vars.reserve(n * nv, cap * nv);
    if (grc == FK_OK) grc = pool->d_param.reserve((size_t)n * t.n_expr, cap * t.n_expr);
    if (grc == FK_OK) grc = pool->d_out.reserve((size_t)n * t.n_expr, cap * t.n_expr);
    if (grc != FK_OK) return grc;
    CU(cudaMemcpyAsync(pool->d_vars, vars, sizeof(double) * (size_t)n * t.n_vars, cudaMemcpyHostToDevice, pool->stream));
    CU(cudaMemcpyAsync(pool->d_param, param, sizeof(double) * (size_t)n * t.n_expr, cudaMemcpyHostToDevice, pool->stream));
    grc = analyze_launch(t.n_vars, t.n_expr, pool->d_kind, pool->d_slot, n, pool->d_vars, pool->d_param, pool->d_out, device, pool->ws, pool->stream);
    if (grc != FK_OK) return grc;
    CU(cudaMemcpyAsync(independent, pool->d_out, (size_t)n * t.n_expr, cudaMemcpyDeviceToHost, pool->stream));
    CU(cudaStreamSynchronize(pool->stream));
    return FK_OK;
}

// ---- device-resident batch plan -----------------------------------------------------------------
// lm: LM may run on the plan.  The L-BFGS calls create their internal plans without, so that they skip the tables of the
// sparse batch LM kernel and its front limit.
static int plan_create(fk_topology* topo, uint32_t capacity, int device, bool lm, fk_batch_plan** out) {
    if (!topo || !out || capacity == 0) return fail(FK_ERR_INVALID, "null topology / zero capacity");
    int rc = check_device(device);
    if (rc != FK_OK) return rc;
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(FK_ERR_NO_DEVICE, "device is not sm_100 class; kernels are built for sm_100a only");
    std::unique_ptr<fk_batch_plan> p(new fk_batch_plan());
    p->topo = topo; p->device = device; p->capacity = capacity; p->lm = lm;
    rc = topo->program_for(device, &p->prog, &p->full, lm);
    if (rc != FK_OK) return rc;
    const fk::Topology& t = topo->t;
    CU(cudaMalloc(&p->d_vars, sizeof(double) * std::max<size_t>(1, (size_t)capacity * t.n_vars)));
    CU(cudaMalloc(&p->d_params, sizeof(double) * std::max<size_t>(1, (size_t)capacity * t.n_expr)));
    CU(cudaMalloc(&p->d_out, sizeof(double) * std::max<size_t>(1, (size_t)capacity * t.n_free)));
    CU(cudaMalloc(&p->d_rep, sizeof(fk_report) * (size_t)capacity));
    if (lm && (rc = p->ws.reserve(*p->full, kSolveLm, capacity)) != FK_OK) return rc;  // (out of memory surfaces here)
    *out = p.release();
    return FK_OK;
}

int fk_batch_plan_create(const fk_topology* topo, uint32_t capacity, int device, fk_batch_plan** out) {
    return plan_create(const_cast<fk_topology*>(topo), capacity, device, true, out);
}

void fk_batch_plan_destroy(fk_batch_plan* plan) { delete plan; }

int fk_batch_plan_upload(fk_batch_plan* plan, uint32_t n, const double* vars, const double* param, void* stream) {
    if (!plan || n > plan->capacity || (n && (!vars || (!param && plan->topo->t.n_expr))))
        return fail(FK_ERR_INVALID, "bad upload arguments");
    const fk::Topology& t = plan->topo->t;
    CU(cudaSetDevice(plan->device));
    plan->n = n;
    if (n && t.n_vars) CU(cudaMemcpyAsync(plan->d_vars, vars, sizeof(double) * (size_t)n * t.n_vars, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    if (n && t.n_expr) CU(cudaMemcpyAsync(plan->d_params, param, sizeof(double) * (size_t)n * t.n_expr, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return FK_OK;
}

// A solve of the plan's n sketches with `kernel` on `stream`.
static int plan_solve(fk_batch_plan* plan, SolveKernel kernel, void* stream) {
    if (!plan) return fail(FK_ERR_INVALID, "null plan");
    CU(cudaSetDevice(plan->device));
    const int rc = solve_launch(*plan->full, kernel, plan->n, plan->d_vars, plan->d_params, plan->d_out, plan->d_rep, plan->ws,
                                (cudaStream_t)stream);
    if (rc == FK_OK && plan->n) plan->launches++;
    return rc;
}

int fk_batch_plan_run(fk_batch_plan* plan, void* stream) { return plan_solve(plan, kSolveLm, stream); }

int fk_batch_plan_run_lbfgs_global(fk_batch_plan* plan, void* stream) { return plan_solve(plan, kSolveLbfgsCta, stream); }

int fk_batch_plan_run_lbfgs(fk_batch_plan* plan, void* stream) {
    if (!plan) return fail(FK_ERR_INVALID, "null plan");
    if (plan->topo->t.path != 0) return fail(FK_ERR_TOO_LARGE, "L-BFGS is built for the shared-memory tile paths only");
    return plan_solve(plan, kSolveLbfgsTile, stream);
}

int fk_batch_plan_download(fk_batch_plan* plan, double* free_out, fk_report* reports, void* stream) {
    if (!plan) return fail(FK_ERR_INVALID, "null plan");
    const fk::Topology& t = plan->topo->t;
    CU(cudaSetDevice(plan->device));
    if (free_out && plan->n && t.n_free)
        CU(cudaMemcpyAsync(free_out, plan->d_out, sizeof(double) * (size_t)plan->n * t.n_free, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    if (reports && plan->n)
        CU(cudaMemcpyAsync(reports, plan->d_rep, sizeof(fk_report) * (size_t)plan->n, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return FK_OK;
}

int fk_batch_plan_device_ptrs(fk_batch_plan* plan, void** vars, void** param, void** free_out, void** reports) {
    if (!plan) return fail(FK_ERR_INVALID, "null plan");
    if (vars) *vars = plan->d_vars;
    if (param) *param = plan->d_params;
    if (free_out) *free_out = plan->d_out;
    if (reports) *reports = plan->d_rep;
    return FK_OK;
}

uint64_t fk_batch_plan_launches(const fk_batch_plan* plan) { return plan ? plan->launches : 0; }

int fk_batch_plan_sync(fk_batch_plan* plan) {
    if (!plan) return fail(FK_ERR_INVALID, "null plan");
    CU(cudaSetDevice(plan->device));
    CU(cudaDeviceSynchronize());
    return FK_OK;
}

int fk_batch_plan_eval(fk_batch_plan* plan, int mode, void* stream) {
    if (!plan) return fail(FK_ERR_INVALID, "null plan");
    const fk::Topology& t = plan->topo->t;
    if (t.path == 2) return fail(FK_ERR_TOO_LARGE, "the evaluation kernels of a batch plan serve the shared-memory paths only; use fk_topology_eval");
    CU(cudaSetDevice(plan->device));
    if (!plan->d_er) CU(cudaMalloc(&plan->d_er, sizeof(double) * std::max<size_t>(1, (size_t)plan->capacity * t.n_rows)));
    if (!plan->d_ej && mode == 0) CU(cudaMalloc(&plan->d_ej, sizeof(double) * std::max<size_t>(1, (size_t)plan->capacity * t.jac_nnz)));
    int e = fk::launch_batch_eval(*plan->prog, plan->n, plan->d_vars, plan->d_params, plan->d_er, plan->d_ej, mode, stream);
    if (e != 0) return cuda_fail((cudaError_t)e, "launch fk_batch_eval_kernel");
    if (plan->n) plan->launches++;
    return FK_OK;
}

int fk_batch_plan_eval_download(fk_batch_plan* plan, double* out_r, double* out_j, void* stream) {
    if (!plan) return fail(FK_ERR_INVALID, "null plan");
    const fk::Topology& t = plan->topo->t;
    CU(cudaSetDevice(plan->device));
    if (out_r && plan->d_er && plan->n)
        CU(cudaMemcpyAsync(out_r, plan->d_er, sizeof(double) * (size_t)plan->n * t.n_rows, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    if (out_j && plan->d_ej && plan->n)
        CU(cudaMemcpyAsync(out_j, plan->d_ej, sizeof(double) * (size_t)plan->n * t.jac_nnz, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return FK_OK;
}

int fk_fp64_peak_tflops(int device, double* out) {
    if (!out) return fail(FK_ERR_INVALID, "null argument");
    if (usable_devices() == 0) return fail(FK_ERR_NO_DEVICE, "no CUDA device visible");
    CU(cudaSetDevice(device));
    double v = 0.0;
    int e = fk::measure_fp64_peak(&v);
    if (e != 0) return cuda_fail((cudaError_t)e, "fp64 peak microbenchmark");
    *out = v;
    return FK_OK;
}

void fk_set_lm_kernel(int choice) { fk::lm_kernel_choice().store(choice < 0 || choice > 3 ? -1 : choice); }
int fk_get_lm_kernel(void) { return fk::lm_kernel_choice().load(); }
int fk_topology_sketch_kernel_info(const fk_topology* topo, int* available, uint32_t* state_doubles, uint32_t* table_words) {
    if (!topo) return fail(FK_ERR_INVALID, "null topology");
    const fk::Topology::SketchTables& k = topo->t.sk;
    if (available) *available = (k.ok && fk::sk_fits(k.entries, k.tab.size())) ? 1 : 0;
    if (state_doubles) *state_doubles = k.entries;
    if (table_words) *table_words = (uint32_t)k.tab.size();
    return FK_OK;
}

int fk_topology_batch_kernel(const fk_topology* topo_c, uint32_t n_sketches) {
    if (!topo_c) return fail(FK_ERR_INVALID, "null topology");
    fk_topology* topo = const_cast<fk_topology*>(topo_c);
    if (topo->t.path == 2) {  // host analysis only (no device needed), once per topology
        const int rc = topo->sb_check();
        return rc == FK_OK ? 3 : rc;
    }
    const fk::Topology::SketchTables& k = topo->t.sk;
    fk::SkProgram probe{};
    probe.entries = k.entries;
    probe.tab_words = (uint32_t)k.tab.size();
    fk::DevProgram p{};
    p.sketch_prog = (k.ok && fk::sk_fits(k.entries, k.tab.size())) ? &probe : nullptr;
    if (!fk::batch_lm_uses_sketch_kernel(p, n_sketches)) return 0;
    return fk::sketch_kernel_is_pair(probe, n_sketches) ? 2 : 1;
}

int fk_topology_lbfgs_kernel(const fk_topology* topo, uint32_t n_sketches) {
    if (!topo) return fail(FK_ERR_INVALID, "null topology");
    return choose_lbfgs(topo, n_sketches);
}

int fk_topology_analyze_kernel(const fk_topology* topo_c, uint32_t n_sketches) {
    if (!topo_c) return fail(FK_ERR_INVALID, "null topology");
    int device = 0;  // (the warp kernel and the limit rule need no device; cta / group are sized on the current one)
    if (cudaGetDevice(&device) != cudaSuccess) {
        cudaGetLastError();
        device = 0;
    }
    fk::AnalyzePlan plan;
    std::string err;
    const int rc = fk::choose_analyze(topo_c->t.n_vars, topo_c->t.n_expr, n_sketches, device, &plan, &err);
    return rc == FK_OK ? plan.kernel : fail(rc, err);
}

void* fk_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
void fk_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

// ---- host-buffer batch: shard by sketch over the devices, pipeline chunks per device ----------------
// Chunk of the host-buffer pipeline: about 1/n_chunks of the request (FK_E2E_CHUNKS overrides n_chunks; copies of one chunk
// overlap the kernels of the others), at least 2,048 sketches, and with `waves` whole waves of the sketch-per-thread kernel when
// that is the kernel in use.
static uint32_t pipeline_chunk(fk_topology* topo, int device, uint32_t total, uint32_t n_chunks, bool waves) {
    static const uint32_t env_chunks = [] {
        const char* e = std::getenv("FK_E2E_CHUNKS");  // tuning knob
        const int v = e ? std::atoi(e) : 0;
        return (uint32_t)(v >= 1 && v <= 256 ? v : 0);
    }();
    if (env_chunks) n_chunks = env_chunks;
    uint32_t chunk = std::min(total, std::max<uint32_t>(2048, (total + n_chunks - 1) / n_chunks));
    const fk::DevProgram* prog = nullptr;
    if (waves && topo->program_for(device, &prog) == FK_OK && fk::batch_lm_uses_sketch_kernel(*prog, total)) {
        static int sms[64] = {0};
        if (device >= 0 && device < 64 && sms[device] == 0) {
            int v = 0;
            if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) == cudaSuccess) sms[device] = v;
        }
        const uint32_t wave = fk::sketch_kernel_wave(*prog->sketch_prog, (device >= 0 && device < 64 && sms[device]) ? sms[device] : 148);
        if (wave && chunk > wave / 2) chunk = std::min(total, ((chunk + wave - 1) / wave) * wave);
    }
    return chunk;
}

// The chunk pipeline of one (topology, device), shared by every host-buffer batch call on it.  Sketches [lo, hi) go in chunks of
// `chunk` over FK_E2E_STREAMS streams (default: all kStreams), each stream with its own pooled plan, which is reused only after its
// previous chunk has drained.  `prologue` (optional) runs once under the pipeline's lock before the first chunk, with the call's
// token slot and the number of streams in use.  `enqueue` enqueues the upload, kernels and download of one chunk on the plan's
// stream and calls mark() after the upload and after the kernels (the FK_E2E_TRACE timeline).
// token == nullptr: returns when the results are in the caller's buffers.  Otherwise it returns once every chunk is enqueued (the
// host still waits, chunk by chunk, for a free plan) and *token names the call for fk_batch_system_solve_wait.  On an error it
// first drains every stream, so that no copy into the caller's buffers is still running when it returns.
using PipelinePrologue = std::function<int(DevicePipeline& pl, int slot, uint32_t use_streams)>;
using PipelineChunk = std::function<int(fk_batch_plan* p, cudaStream_t st, uint32_t at, uint32_t cnt, const std::function<void()>& mark)>;
// lm: the chunks run LM (plans made for L-BFGS only are then made again).
static int run_pipeline(fk_topology* topo, int device, uint32_t lo, uint32_t hi, uint32_t chunk, uint64_t* token,
                        const PipelinePrologue& prologue, const PipelineChunk& enqueue, bool lm = true) {
    constexpr uint32_t kStreams = DevicePipeline::kStreams;
    static const uint32_t use_streams = [] {
        const char* e = std::getenv("FK_E2E_STREAMS");  // tuning knob: chunks in flight (at most kStreams)
        const int v = e ? std::atoi(e) : 0;
        return (uint32_t)(v >= 1 && v <= (int)kStreams ? v : (int)kStreams);
    }();
    // FK_E2E_TRACE=1 (debug): CUDA-event timeline of the chunks of every call to stderr (upload done / kernel done / download done)
    static const bool trace = std::getenv("FK_E2E_TRACE") != nullptr;
    CU(cudaSetDevice(device));
    DevicePipeline* pl = topo->pipeline_for(device);
    std::lock_guard<std::mutex> lock(pl->mu);
    int rc = FK_OK;
    if (pl->chunk < chunk || (lm && !pl->plans_lm)) {
        const uint32_t cap = std::max(chunk, pl->chunk);
        pl->release();
        for (uint32_t s = 0; s < kStreams && rc == FK_OK; s++) {
            rc = plan_create(topo, cap, device, lm, &pl->plans[s]);
            if (rc == FK_OK && cudaStreamCreateWithFlags(&pl->streams[s], cudaStreamNonBlocking) != cudaSuccess)
                rc = fail(FK_ERR_CUDA, "cudaStreamCreate failed");
        }
        if (rc != FK_OK) {
            pl->release();
            return rc;
        }
        pl->chunk = cap;
        pl->plans_lm = lm;
    }
    const uint64_t my_token = pl->next_token++;
    const int slot = (int)(my_token & 1u);
    uint32_t s = 0;
    std::vector<cudaEvent_t> tev;
    cudaEvent_t t_start = nullptr;
    const std::function<void()> mark = [&] {
        if (!trace) return;
        cudaEvent_t ev;
        cudaEventCreate(&ev);
        cudaEventRecord(ev, pl->streams[s]);
        tev.push_back(ev);
    };
    if (trace) {
        cudaEventCreate(&t_start);
        cudaEventRecord(t_start, pl->streams[0]);
    }
    if (prologue) rc = prologue(*pl, slot, use_streams);
    for (uint32_t at = lo; at < hi && rc == FK_OK; at += chunk, s = (s + 1) % use_streams) {
        const cudaError_t e = cudaStreamSynchronize(pl->streams[s]);
        if (e != cudaSuccess) {
            rc = cuda_fail(e, "cudaStreamSynchronize");
            break;
        }
        rc = enqueue(pl->plans[s], pl->streams[s], at, std::min(chunk, hi - at), mark);
        mark();
    }
    auto record_done = [&]() -> int {  // the _begin half: events behind the call's last chunk on every stream
        for (uint32_t k = 0; k < kStreams; k++) {
            if (!pl->done_ev[slot][k]) CU(cudaEventCreateWithFlags(&pl->done_ev[slot][k], cudaEventDisableTiming));
            CU(cudaEventRecord(pl->done_ev[slot][k], pl->streams[k]));
        }
        return FK_OK;
    };
    if (rc == FK_OK && token && !trace && (rc = record_done()) == FK_OK) {
        *token = my_token;
        return FK_OK;
    }
    for (uint32_t k = 0; k < kStreams; k++) {
        const cudaError_t e = cudaStreamSynchronize(pl->streams[k]);
        if (e != cudaSuccess && rc == FK_OK) rc = cuda_fail(e, "batch kernel / copy failed");
    }
    if (rc == FK_OK && token) *token = my_token;  // (tracing: the call has completed; waiting for it is a no-op)
    if (trace) {
        for (size_t c = 0; c + 2 < tev.size(); c += 3) {
            float a = 0, b = 0, d = 0;
            cudaEventElapsedTime(&a, t_start, tev[c]);
            cudaEventElapsedTime(&b, t_start, tev[c + 1]);
            cudaEventElapsedTime(&d, t_start, tev[c + 2]);
            fprintf(stderr, "[e2e trace] chunk %2zu: upload done %7.1f us, kernel done %7.1f us, download done %7.1f us\n", c / 3, a * 1e3f, b * 1e3f, d * 1e3f);
        }
        for (cudaEvent_t ev : tev) cudaEventDestroy(ev);
        cudaEventDestroy(t_start);
    }
    return rc;
}


// Small request (one sketch, a handful): the caller's (pageable) arrays go through ONE pinned staging block -- one
// copy in, the kernel, one copy out, one synchronisation -- instead of four pageable copies on the chunk pipeline.
static bool small_fits(const fk::Topology& t, uint32_t total) {
    const size_t in_v = sizeof(double) * (size_t)total * t.n_vars, in_p = sizeof(double) * (size_t)total * t.n_expr;
    const size_t out_x = sizeof(double) * (size_t)total * t.n_free, out_r = sizeof(fk_report) * (size_t)total;
    return ((in_v + in_p + 15) & ~size_t(15)) + out_x + out_r <= DevicePipeline::kSmallBytes;
}
static int small_solve(fk_topology* topo, int device, uint32_t lo, uint32_t hi, const double* vars, const double* param,
                       double* free_out, fk_report* reports, int optimizer) {
    const fk::Topology& t = topo->t;
    const uint32_t total = hi - lo;
    DevicePipeline* pl = topo->pipeline_for(device);
    std::lock_guard<std::mutex> lock(pl->mu);  // the pipeline's staging block is ours until the results are copied out
    const size_t in_v = sizeof(double) * (size_t)total * t.n_vars, in_p = sizeof(double) * (size_t)total * t.n_expr;
    const size_t out_x = sizeof(double) * (size_t)total * t.n_free, out_r = sizeof(fk_report) * (size_t)total;
    const size_t in_al = (in_v + in_p + 15) & ~size_t(15);
    const fk::DevProgram* prog = nullptr;
    const DeviceProgram* full = nullptr;
    int rc = topo->program_for(device, &prog, &full, optimizer == 0);
    if (rc != FK_OK) return rc;
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
    if ((rc = pl->small_h.reserve(DevicePipeline::kSmallBytes)) != FK_OK || (rc = pl->small_d.reserve(DevicePipeline::kSmallBytes)) != FK_OK)
        return rc;
    if (!pl->small_stream && (e = cudaStreamCreateWithFlags(&pl->small_stream, cudaStreamNonBlocking)) != cudaSuccess) {
        pl->small_stream = nullptr;
        return cuda_fail(e, "cudaStreamCreate");
    }
    std::memcpy(pl->small_h, vars + (size_t)lo * t.n_vars, in_v);
    if (in_p) std::memcpy(pl->small_h + in_v, param + (size_t)lo * t.n_expr, in_p);
    // A few kilobytes: the kernel reads its inputs from, and writes its results to, the pinned block itself (pinned host
    // memory is mapped into the device's address space under unified addressing; the kernel touches every input and output
    // once) -- two DMA set-ups less on a path that is all latency.  FK_NO_ZERO_COPY=1 keeps the two copies (A/B knob).  Not
    // for the sparse batch LM kernel or the L-BFGS kernels: they read the parameters and fixed variables again on every
    // evaluation.
    static const bool no_zero_copy = std::getenv("FK_NO_ZERO_COPY") != nullptr;
    static const bool can_map = [] {
        int dev = 0, ok = 0;
        return cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&ok, cudaDevAttrCanUseHostPointerForRegisteredMem, dev) == cudaSuccess && ok != 0;
    }();
    const bool zero_copy = !no_zero_copy && can_map && optimizer == 0 && !full->sparse_batch && in_al + out_x + out_r <= 8 * 1024;
    unsigned char* base = zero_copy ? pl->small_h : pl->small_d;
    if (!zero_copy && (e = cudaMemcpyAsync(pl->small_d, pl->small_h, in_v + in_p, cudaMemcpyHostToDevice, pl->small_stream)) != cudaSuccess) return cuda_fail(e, "cudaMemcpyAsync");
    const double *d_vars = (const double*)base, *d_param = (const double*)(base + in_v);
    double* d_out = (double*)(base + in_al);
    fk_report* d_rep = (fk_report*)(base + in_al + out_x);
    rc = solve_launch(*full, solve_kernel(topo, optimizer, total), total, d_vars, d_param, d_out, d_rep, pl->small_ws, pl->small_stream);
    if (rc != FK_OK) return rc;
    if (!zero_copy && (e = cudaMemcpyAsync(pl->small_h + in_al, pl->small_d + in_al, out_x + out_r, cudaMemcpyDeviceToHost, pl->small_stream)) != cudaSuccess) return cuda_fail(e, "cudaMemcpyAsync");
    if ((e = cudaStreamSynchronize(pl->small_stream)) != cudaSuccess) return cuda_fail(e, "batch kernel / copy failed");
    std::memcpy(free_out + (size_t)lo * t.n_free, pl->small_h + in_al, out_x);
    if (reports) std::memcpy(reports + lo, pl->small_h + in_al + out_x, out_r);
    return FK_OK;
}

// Sketches [lo, hi) of a uniform batch on one device: a small request through the staging block, anything larger through the
// chunk pipeline.  optimizer 1: L-BFGS with the kernel of choose_lbfgs.  token: see run_pipeline; the caller sets *token = 0,
// which is what a small request (complete when it returns) leaves there.
static int run_device_range(fk_topology* topo, int device, uint32_t lo, uint32_t hi, const double* vars, const double* param,
                            double* free_out, fk_report* reports, int optimizer, uint64_t* token) {
    if (hi == lo) return FK_OK;
    const fk::Topology& t = topo->t;
    if (small_fits(t, hi - lo)) return small_solve(topo, device, lo, hi, vars, param, free_out, reports, optimizer);
    // (the L-BFGS kernel is not the sketch-per-thread kernel: its chunks are not rounded to that kernel's waves)
    const uint32_t chunk = pipeline_chunk(topo, device, hi - lo, 8, optimizer == 0);
    const SolveKernel kernel = solve_kernel(topo, optimizer, hi - lo);
    return run_pipeline(topo, device, lo, hi, chunk, token, nullptr,
                        [&](fk_batch_plan* p, cudaStream_t st, uint32_t at, uint32_t cnt, const std::function<void()>& mark) {
                            int rc = fk_batch_plan_upload(p, cnt, vars + (size_t)at * t.n_vars, param ? param + (size_t)at * t.n_expr : nullptr, st);
                            if (rc != FK_OK) return rc;
                            mark();
                            rc = plan_solve(p, kernel, st);
                            if (rc != FK_OK) return rc;
                            mark();
                            return fk_batch_plan_download(p, free_out + (size_t)at * t.n_free, reports ? reports + at : nullptr, st);
                        },
                        optimizer == 0);
}

// ---- System::solve level batch: scale, perturbation and write-back on the device -----------------------------
static int prepare_tables_for(fk_topology* topo, int device, const fk_prepare_opts& o, PrepareTables** out) {
    const fk::Topology& t = topo->t;
    std::lock_guard<std::mutex> lock(topo->mu);
    auto& p = topo->prepare_tables[device];
    std::vector<uint32_t> list;
    if (o.flags & FK_PREP_PERTURB) {
        if (o.perturb_vars) list.assign(o.perturb_vars, o.perturb_vars + o.n_perturb);
        else list = t.free_vars;
        for (size_t q = 0; q < list.size(); q++)
            if (list[q] >= t.n_vars || (q && list[q] <= list[q - 1]))
                return fail(FK_ERR_INVALID, "perturbed variables must be in range, ascending and distinct");
    }
    if (p && p->perturb_vars == list && p->seed == o.seed) { *out = p.get(); return FK_OK; }
    std::unique_ptr<PrepareTables> q(new PrepareTables());
    CU(cudaSetDevice(device));
    q->device = device; q->perturb_vars = list; q->seed = o.seed;
    std::vector<double> draws(2 * list.size() + 1, 0.0);
    uint32_t st = o.seed;
    for (size_t k = 0; k < 2 * list.size(); k++) {  // rand.rs:24-39
        st = st * 1664525u + 1013904223u;
        draws[k] = (1.0 / 4294967295.0) * (double)st;
    }
    std::vector<uint32_t> where(t.n_vars, 0xFFFFFFFFu), free_draw(std::max<uint32_t>(t.n_free, 1), 0xFFFFFFFFu), fix_draw(std::max<uint32_t>(t.sk.nfix, 1), 0xFFFFFFFFu);
    for (size_t j = 0; j < list.size(); j++) where[list[j]] = (uint32_t)j;
    for (uint32_t c = 0; c < t.n_free; c++) free_draw[c] = where[t.free_vars[c]];
    if (t.sk.ok)
        for (uint32_t i = 0; i < t.sk.nfix; i++) fix_draw[i] = where[t.sk.tab[t.sk.off_fix + i]];
    TablePack pk;
    const size_t o_kind = pk.add(t.kind), o_perturb = pk.add(list), o_draws = pk.add(draws), o_free = pk.add(free_draw), o_fix = pk.add(fix_draw);
    const int rc = pk.upload(0, &q->d_tables);
    if (rc != FK_OK) return rc;
    q->d_kind = pk.at<uint8_t>(o_kind); q->d_perturb = pk.at<uint32_t>(o_perturb); q->d_draws = pk.at<double>(o_draws);
    q->d_free_draw = pk.at<uint32_t>(o_free); q->d_fix_draw = pk.at<uint32_t>(o_fix);
    p = std::move(q);
    *out = p.get();
    return FK_OK;
}

// fk_batch_system_solve, and its _begin half with a token.
static int batch_system_solve(const fk_topology* topo_c, int device, uint32_t n, const double* raw_vars, const double* raw_param,
                              const fk_prepare_opts* opts, double* free_out, double* scales_out, fk_report* reports, uint64_t* token) {
    fk_topology* topo = const_cast<fk_topology*>(topo_c);
    if (!topo || !opts) return fail(FK_ERR_INVALID, "null argument");
    if (token) *token = 0;
    if (n == 0) return FK_OK;
    const fk::Topology& t = topo->t;
    if (!raw_vars || !free_out || (!raw_param && t.n_expr)) return fail(FK_ERR_INVALID, "null buffer");
    int rc = check_device(device);
    if (rc != FK_OK) return rc;
    PrepareTables* pt = nullptr;
    if ((rc = prepare_tables_for(topo, device, *opts, &pt)) != FK_OK) return rc;
    const bool shared = (opts->flags & FK_PREP_SHARED_PARAM) != 0;
    static const bool no_fuse = std::getenv("FK_NO_FUSED_PREPARE") != nullptr;  // A/B knob
    const double* d_shared_param = nullptr;
    auto prologue = [&](DevicePipeline& pl, int slot, uint32_t use_streams) -> int {
        for (fk_batch_plan* p : pl.plans) {  // unscaled input / scale buffers of the plans, on first use
            if (!p->d_raw_vars) CU(cudaMalloc(&p->d_raw_vars, sizeof(double) * std::max<size_t>(1, (size_t)p->capacity * t.n_vars)));
            if (!p->d_raw_param) CU(cudaMalloc(&p->d_raw_param, sizeof(double) * std::max<size_t>(1, (size_t)p->capacity * t.n_expr)));
            if (!p->d_scales) CU(cudaMalloc(&p->d_scales, sizeof(double) * p->capacity));
        }
        if (!shared || !t.n_expr) return FK_OK;
        // One parameter row for all sketches: uploaded once per call, every stream waits for it (a 300-byte copy per chunk kept the
        // H2D engine ~10 us per chunk, which the first chunks of a call -- the ones the device is waiting for -- paid in full).
        if (!pl.shared_param_ev) CU(cudaEventCreateWithFlags(&pl.shared_param_ev, cudaEventDisableTiming));
        if (pl.shared_param_cap < t.n_expr) {  // (two rows: the kernels of the previous call may still read theirs)
            for (int a = 0; a < 2; a++) {
                if (pl.d_shared_param[a]) CU(cudaFree(pl.d_shared_param[a]));
                pl.d_shared_param[a] = nullptr;
                CU(cudaMalloc(&pl.d_shared_param[a], sizeof(double) * t.n_expr));
            }
            pl.shared_param_cap = t.n_expr;
        }
        d_shared_param = pl.d_shared_param[slot];
        CU(cudaMemcpyAsync(pl.d_shared_param[slot], raw_param, sizeof(double) * t.n_expr, cudaMemcpyHostToDevice, pl.streams[0]));
        CU(cudaEventRecord(pl.shared_param_ev, pl.streams[0]));
        for (uint32_t k = 1; k < use_streams; k++) CU(cudaStreamWaitEvent(pl.streams[k], pl.shared_param_ev, 0));
        return FK_OK;
    };
    // (Chunks that taper at both ends of a call -- a quarter and a half of the regular size first, halving down to 1,024 sketches at the
    // end -- bring the first kernel forward from 65 to 24 us and change nothing: 1,108 against 1,092 us per call.  The last kernel ends
    // ~1,070 us after the call started either way; the chunked kernels together take ~1,040 us where one launch over the resident
    // batch takes 905.)
    auto enqueue = [&](fk_batch_plan* p, cudaStream_t st, uint32_t at, uint32_t cnt, const std::function<void()>& mark) -> int {
        const bool fused = !no_fuse && fk::batch_lm_uses_sketch_kernel(*p->prog, cnt) && fk::sk_raw_fits(*p->prog->sketch_prog, shared);
        p->n = cnt;
        if (t.n_vars) CU(cudaMemcpyAsync(p->d_raw_vars, raw_vars + (size_t)at * t.n_vars, sizeof(double) * (size_t)cnt * t.n_vars, cudaMemcpyHostToDevice, st));
        if (t.n_expr && !shared)
            CU(cudaMemcpyAsync(p->d_raw_param, raw_param + (size_t)at * t.n_expr, sizeof(double) * (size_t)cnt * t.n_expr, cudaMemcpyHostToDevice, st));
        const double* d_param = shared ? d_shared_param : p->d_raw_param;
        mark();
        int e;
        if (fused) {  // the sketch-per-thread kernel scales, perturbs and writes back itself (SkRaw)
            fk::SkRaw raw{};
            raw.raw_vars = p->d_raw_vars; raw.raw_param = d_param; raw.shared_param = shared ? 1u : 0u;
            raw.kinds = pt->d_kind; raw.free_draw = pt->d_free_draw; raw.fix_draw = pt->d_fix_draw; raw.draws = pt->d_draws;
            raw.scales = p->d_scales;
            e = fk::launch_batch_lm_sketch(*p->prog->sketch_prog, cnt, nullptr, nullptr, p->d_out, p->d_rep, st, &raw);
            p->launches += 1;
        } else {
            p->launches += 3;
            e = fk::launch_batch_prepare(cnt, t.n_vars, t.n_expr, pt->d_kind, shared, (uint32_t)pt->perturb_vars.size(), pt->d_perturb, pt->d_draws,
                                         p->d_raw_vars, d_param, p->d_vars, p->d_params, p->d_scales, st);
            if (e == 0) {
                const int rc = solve_launch(*p->full, kSolveLm, cnt, p->d_vars, p->d_params, p->d_out, p->d_rep, p->ws, st);
                if (rc != FK_OK) return rc;
                e = fk::launch_batch_unscale(cnt, t.n_free, p->d_scales, p->d_out, st);
            }
        }
        if (e != 0) return cuda_fail((cudaError_t)e, "launch fk_batch_system_solve kernels");
        mark();
        if (t.n_free) CU(cudaMemcpyAsync(free_out + (size_t)at * t.n_free, p->d_out, sizeof(double) * (size_t)cnt * t.n_free, cudaMemcpyDeviceToHost, st));
        if (scales_out) CU(cudaMemcpyAsync(scales_out + at, p->d_scales, sizeof(double) * cnt, cudaMemcpyDeviceToHost, st));
        if (reports) CU(cudaMemcpyAsync(reports + at, p->d_rep, sizeof(fk_report) * (size_t)cnt, cudaMemcpyDeviceToHost, st));
        return FK_OK;
    };
    return run_pipeline(topo, device, 0, n, pipeline_chunk(topo, device, n, 16, true), token, prologue, enqueue);
}

int fk_batch_system_solve(const fk_topology* topo, int device, uint32_t n, const double* raw_vars, const double* raw_param,
                          const fk_prepare_opts* opts, double* free_out, double* scales_out, fk_report* reports) {
    return batch_system_solve(topo, device, n, raw_vars, raw_param, opts, free_out, scales_out, reports, nullptr);
}

int fk_batch_system_solve_begin(const fk_topology* topo, int device, uint32_t n, const double* raw_vars, const double* raw_param,
                                const fk_prepare_opts* opts, double* free_out, double* scales_out, fk_report* reports, uint64_t* token) {
    if (!token) return fail(FK_ERR_INVALID, "null token");
    return batch_system_solve(topo, device, n, raw_vars, raw_param, opts, free_out, scales_out, reports, token);
}

int fk_batch_system_solve_wait(const fk_topology* topo_c, int device, uint64_t token) {
    fk_topology* topo = const_cast<fk_topology*>(topo_c);
    if (!topo) return fail(FK_ERR_INVALID, "null topology");
    if (token == 0) return FK_OK;  // (an empty call)
    const int ndev = usable_devices();
    if (device < 0 || device >= ndev) return fail(FK_ERR_INVALID, "device index out of range");
    DevicePipeline* pl = topo->pipeline_for(device);
    cudaEvent_t ev[DevicePipeline::kStreams];
    {
        std::lock_guard<std::mutex> lock(pl->mu);
        if (token >= pl->next_token) return fail(FK_ERR_INVALID, "unknown token");
        // (a token older than the last two calls: its slot now holds a later call's events, recorded behind this call's work on
        // the same streams, so waiting for those covers it)
        for (uint32_t k = 0; k < DevicePipeline::kStreams; k++) ev[k] = pl->done_ev[token & 1u][k];
    }
    for (uint32_t k = 0; k < DevicePipeline::kStreams; k++)
        if (ev[k]) CU(cudaEventSynchronize(ev[k]));
    return FK_OK;
}

// fk_batch_solve_device, and its _begin half with a token.
static int batch_solve_device(const fk_topology* topo_c, int device, uint32_t n, const double* vars, const double* param,
                              double* free_out, fk_report* reports, uint64_t* token) {
    fk_topology* topo = const_cast<fk_topology*>(topo_c);
    if (!topo) return fail(FK_ERR_INVALID, "null topology");
    if (token) *token = 0;
    if (n == 0) return FK_OK;
    if (!vars || !free_out || (!param && topo->t.n_expr)) return fail(FK_ERR_INVALID, "null buffer");
    const int rc = check_device(device);
    if (rc != FK_OK) return rc;
    return run_device_range(topo, device, 0, n, vars, param, free_out, reports, 0, token);
}

int fk_batch_solve_device(const fk_topology* topo, int device, uint32_t n, const double* vars, const double* param,
                          double* free_out, fk_report* reports) {
    return batch_solve_device(topo, device, n, vars, param, free_out, reports, nullptr);
}

int fk_batch_solve_device_begin(const fk_topology* topo, int device, uint32_t n, const double* vars, const double* param,
                                double* free_out, fk_report* reports, uint64_t* token) {
    if (!token) return fail(FK_ERR_INVALID, "null token");
    return batch_solve_device(topo, device, n, vars, param, free_out, reports, token);
}

int fk_batch_solve_device_wait(const fk_topology* topo, int device, uint64_t token) { return fk_batch_system_solve_wait(topo, device, token); }

// n sketches of one topology over n_gpus devices: contiguous shares, one host thread per device (fk_batch_solve).
static int solve_sharded(fk_topology* topo, uint32_t n, const double* vars, const double* param, double* free_out, fk_report* reports,
                         int n_gpus, int optimizer) {
    return shard_over_devices(n_gpus, n, [&](int device, uint32_t lo, uint32_t hi) {
        return run_device_range(topo, device, lo, hi, vars, param, free_out, reports, optimizer);
    });
}

int fk_batch_solve(const fk_topology* topo_c, uint32_t n, const double* vars, const double* param, double* free_out,
                   fk_report* reports, int n_gpus) {
    fk_topology* topo = const_cast<fk_topology*>(topo_c);
    if (!topo) return fail(FK_ERR_INVALID, "null topology");
    if (n == 0) return FK_OK;
    if (!vars || !free_out || (!param && topo->t.n_expr)) return fail(FK_ERR_INVALID, "null buffer");
    const int rc = clamp_gpus(n_gpus);
    if (rc != FK_OK) return rc;
    return solve_sharded(topo, n, vars, param, free_out, reports, n_gpus, 0);
}

// ---- single system with a cached topology (any path) --------------------------------------------------
int fk_topology_lm_solve(fk_topology* topo, const double* vars, const double* param, double* free_values,
                         fk_report* report) {
    if (!topo || !free_values || (!vars && topo->t.n_vars)) return fail(FK_ERR_INVALID, "null argument");
    int cur = 0;
    if (cudaGetDevice(&cur) != cudaSuccess) cur = 0;
    int rc = check_device(cur);
    if (rc != FK_OK) return rc;
    const fk::Topology& t = topo->t;
    if (t.path == 2) {
        fk::SparseSolver* sp = nullptr;
        std::string err;
        rc = topo->sparse_for(cur, &sp, &err);
        if (rc != FK_OK) return fail(rc, err);
        // the caller's free values are the starting point (== `variables` of lm.rs:21)
        if (!param && t.n_expr) return fail(FK_ERR_INVALID, "null parameter array");
        std::lock_guard<std::mutex> lock(topo->sparse_mu);
        rc = sp->solve(vars, param, free_values, report, &err);
        return rc == FK_OK ? FK_OK : fail(rc, err);
    }
    std::vector<double> v(vars, vars + t.n_vars), out(std::max<uint32_t>(1, t.n_free));
    for (uint32_t f = 0; f < t.n_free; f++) v[t.free_vars[f]] = free_values[f];
    std::vector<double> zero;
    if (!param && t.n_expr) zero.assign(t.n_expr, 0.0);
    // One system is latency bound (one warp walks the whole LM loop): the lane count chosen for batch throughput
    // (4-16 by footprint) leaves lanes of that warp idle.  A twin of the topology with all 32 lanes, built on the
    // first single-system solve, serves these calls (same operations per entry, same results; tools/lat_probe.py:
    // 144 -> 89 us on the mixed-primitive sketch).
    fk_topology* exec = topo->lanes32();
    rc = run_device_range(exec, cur, 0, 1, v.data(), param ? param : zero.data(), out.data(), report);
    if (rc == FK_OK && t.n_free) std::memcpy(free_values, out.data(), sizeof(double) * t.n_free);
    return rc;
}

int fk_topology_eval(fk_topology* topo, const double* vars, const double* param, const double* free_values,
                     double* out_r, double* out_j, int repeats, float* ms_per_eval) {
    if (!topo || !vars || !free_values) return fail(FK_ERR_INVALID, "null argument");
    int cur = 0;
    if (cudaGetDevice(&cur) != cudaSuccess) cur = 0;
    int rc = check_device(cur);
    if (rc != FK_OK) return rc;
    if (topo->t.path != 2) return fail(FK_ERR_INVALID, "fk_topology_eval serves the global sparse path; use fk_batch_plan_eval");
    fk::SparseSolver* sp = nullptr;
    std::string err;
    rc = topo->sparse_for(cur, &sp, &err);
    if (rc == FK_OK) {
        std::lock_guard<std::mutex> lock(topo->sparse_mu);
        rc = sp->eval_once(vars, param, free_values, out_r, out_j, repeats, ms_per_eval, &err);
    }
    return rc == FK_OK ? FK_OK : fail(rc, err);
}

int fk_topology_last_timing(fk_topology* topo, float* out8) {
    if (!topo || !out8) return fail(FK_ERR_INVALID, "null argument");
    std::memset(out8, 0, 8 * sizeof(float));
    std::lock_guard<std::mutex> lock(topo->mu);
    for (auto& kv : topo->sparse) {
        const auto& l = kv.second->last;
        out8[0] = l.eval_ms; out8[1] = l.assemble_ms; out8[2] = l.factor_ms; out8[3] = l.tri_ms;
        out8[4] = (float)l.evals; out8[5] = (float)l.factors; out8[6] = l.fwd_ms; out8[7] = l.bwd_ms;
    }
    return FK_OK;
}

// ---- general entry points ------------------------------------------------------------------------------
// "Symbolic analysis once per topology" for the callers that hand over flattened problems (fk_lm_solve,
// fk_lm_solve_batch, fk_system_solve*): a process-wide LRU cache of fk_topology objects keyed by the structural
// content of the problem (sizes, kinds, indices, free set, row list).  The reference repeats the analysis on every
// LM call (fiksi/src/solve/lm.rs:98-104); an interactive solver re-solves the same sketch over and over.  Entries
// are shared_ptrs: an evicted topology lives until the solves that use it have returned.
namespace {

struct TopologyCache {
    struct Entry { uint64_t sig; std::shared_ptr<fk_topology> topo; };
    std::mutex mu;
    std::list<Entry> lru;  // front = most recently used
    std::unordered_multimap<uint64_t, std::list<Entry>::iterator> index;  // signature -> entry
    void drop(std::list<Entry>::iterator it) {
        auto range = index.equal_range(it->sig);
        for (auto q = range.first; q != range.second; ++q)
            if (q->second == it) { index.erase(q); break; }
        lru.erase(it);
    }
    size_t capacity = [] {
        const char* e = std::getenv("FK_TOPOLOGY_CACHE");
        const int v = e ? std::atoi(e) : 1024;
        return (size_t)std::max(0, v);
    }();
    uint64_t hits = 0, misses = 0;
};
TopologyCache& topology_cache() {
    static TopologyCache* c = new TopologyCache();  // never destroyed: CUDA may be gone by static-destruction time
    return *c;
}

uint64_t structural_signature(const fk_problem& p) {
    uint64_t sig = 1469598103934665603ull;
    auto mixb = [&](const void* d, size_t bytes) {
        const unsigned char* c = (const unsigned char*)d;
        for (size_t k = 0; k < bytes; k++) sig = (sig ^ c[k]) * 1099511628211ull;
    };
    const uint32_t hdr[4] = {p.n_vars, p.n_expr, p.n_free, p.n_rows};
    mixb(hdr, sizeof hdr);
    if (p.n_expr) { mixb(p.kind, p.n_expr); mixb(p.idx, 16 * (size_t)p.n_expr); }
    if (p.n_free) mixb(p.free_vars, 4 * (size_t)p.n_free);
    if (p.n_rows) mixb(p.rows, 4 * (size_t)p.n_rows);
    return sig;
}
bool same_structure(const fk_problem& a, const fk_problem& p) {
    return a.n_vars == p.n_vars && a.n_expr == p.n_expr && a.n_free == p.n_free && a.n_rows == p.n_rows &&
           (!p.n_expr || (!std::memcmp(a.kind, p.kind, p.n_expr) && !std::memcmp(a.idx, p.idx, 16 * (size_t)p.n_expr))) &&
           (!p.n_free || !std::memcmp(a.free_vars, p.free_vars, 4 * (size_t)p.n_free)) &&
           (!p.n_rows || !std::memcmp(a.rows, p.rows, 4 * (size_t)p.n_rows));
}
fk_problem structure_of(const fk::Topology& t) {  // (no values: vars / param stay null)
    fk_problem p{};
    p.n_vars = t.n_vars; p.n_expr = t.n_expr; p.kind = t.kind.data(); p.idx = t.idx.data();
    p.n_free = t.n_free; p.free_vars = t.free_vars.data(); p.n_rows = t.n_rows; p.rows = t.rows.data();
    return p;
}
bool problem_arrays_ok(const fk_problem& p) {
    return !((p.n_vars && !p.vars) || (p.n_expr && (!p.kind || !p.idx)) || (p.n_free && !p.free_vars) || (p.n_rows && !p.rows));
}

std::shared_ptr<fk_topology> cache_lookup(uint64_t sig, const fk_problem& p) {
    TopologyCache& c = topology_cache();
    std::lock_guard<std::mutex> lock(c.mu);
    auto range = c.index.equal_range(sig);
    for (auto q = range.first; q != range.second; ++q)
        if (same_structure(structure_of(q->second->topo->t), p)) {
            c.lru.splice(c.lru.begin(), c.lru, q->second);  // (list iterators stay valid)
            c.hits++;
            return c.lru.front().topo;
        }
    c.misses++;
    return nullptr;
}
void cache_insert(uint64_t sig, const std::shared_ptr<fk_topology>& topo) {
    TopologyCache& c = topology_cache();
    std::lock_guard<std::mutex> lock(c.mu);
    if (c.capacity == 0) return;
    c.lru.push_front({sig, topo});
    c.index.emplace(sig, c.lru.begin());
    while (c.lru.size() > c.capacity) c.drop(std::prev(c.lru.end()));
    // large single systems keep hundreds of megabytes of factor storage on the device: at most four of them stay
    if (topo->t.path == 2) {
        size_t large = 0;
        for (auto it = c.lru.begin(); it != c.lru.end();) {
            auto cur = it++;
            if (cur->topo->t.path == 2 && ++large > 4) c.drop(cur);
        }
    }
}

}  // namespace

void fk_topology_cache_configure(uint32_t capacity) {
    TopologyCache& c = topology_cache();
    std::lock_guard<std::mutex> lock(c.mu);
    c.capacity = capacity;
    while (c.lru.size() > c.capacity) c.drop(std::prev(c.lru.end()));
}
void fk_topology_cache_clear(void) {
    TopologyCache& c = topology_cache();
    std::lock_guard<std::mutex> lock(c.mu);
    c.index.clear();
    c.lru.clear();
}
void fk_topology_cache_stats(uint64_t* hits, uint64_t* misses, uint32_t* entries) {
    TopologyCache& c = topology_cache();
    std::lock_guard<std::mutex> lock(c.mu);
    if (hits) *hits = c.hits;
    if (misses) *misses = c.misses;
    if (entries) *entries = (uint32_t)c.lru.size();
}

// Staging of the heterogeneous-batch kernel, one per device: pinned host block + device block (grow-only), one stream.
struct HeteroPool {
    std::mutex mu;
    int device = -1;
    GrowBuf<unsigned char> h{true}, d;
    cudaStream_t stream = nullptr;
};
static HeteroPool* hetero_pool_for(int device) {
    static std::mutex m;
    static std::map<int, HeteroPool*> pools;  // never destroyed (CUDA may be gone at static-destruction time)
    std::lock_guard<std::mutex> lock(m);
    HeteroPool*& p = pools[device];
    if (!p) {
        p = new HeteroPool();
        p->device = device;
    }
    return p;
}

// Whether a structure of `instances` systems goes to fk_hetero_lm_kernel (one warp per system) rather than a uniform batch
// launch: path 0, fewer than 64 systems (from there the sketch-per-thread kernel is the faster one) and an LM state within
// 48 KiB.  The launch also needs the topology's 32-lane tables (hetero_topology).
static bool hetero_fits(const fk::Topology& t, size_t instances) {
    return t.path == 0 && instances < 64 && fk::lm_smem_doubles(t.n_free, t.n_rows, t.jac_nnz, (uint32_t)t.l_rowidx.size()) * 8 <= 48 * 1024;
}

// The topology with 32-lane tables (fk_topology::lanes32) through which a structure of `instances` systems goes to
// fk_hetero_lm_kernel, or null when it keeps a uniform batch launch: hetero_fits fails, or there are no 32-lane tables
// (FK_NO_LATENCY_TWIN).
static fk_topology* hetero_topology(fk_topology* topo, size_t instances) {
    if (!hetero_fits(topo->t, instances)) return nullptr;
    fk_topology* t32 = topo->lanes32();
    return t32->t.tile == 32 ? t32 : nullptr;
}

// The programs of fk_hetero_lm_kernel on `device` (32-lane tables, no sketch-kernel block) and the largest LM state among them.
static int hetero_programs(int device, const std::vector<fk_topology*>& topos32, std::vector<fk::DevProgram>& progs, uint32_t* max_state) {
    progs.assign(topos32.size(), fk::DevProgram{});
    *max_state = 1;
    for (size_t g = 0; g < topos32.size(); g++) {
        const fk::DevProgram* v = nullptr;
        const int rc = topos32[g]->program_for(device, &v);
        if (rc != FK_OK) return rc;
        progs[g] = *v;
        progs[g].sketch_prog = nullptr;
        *max_state = std::max(*max_state, fk::lm_smem_doubles(v->n, v->m, v->jnnz, v->lnnz));
    }
    return FK_OK;
}

// One launch of fk_hetero_lm_kernel over device-resident programs, jobs and input rows.
static int hetero_launch(const fk::DevProgram* d_progs, const fk::HeteroJob* d_jobs, size_t nj, uint32_t max_state, const double* d_in,
                         double* d_out, fk_report* d_rep, cudaStream_t st) {
    const int e = fk::launch_hetero_lm(d_progs, d_jobs, (uint32_t)nj, max_state, d_in, d_out, d_rep, st);
    return e != 0 ? cuda_fail((cudaError_t)e, "launch fk_hetero_lm_kernel") : FK_OK;
}

// Solves jobs (group index, member) of small path-0 groups with ONE launch of fk_hetero_lm_kernel on `device`: the programs,
// jobs and input rows staged in a pinned block, one copy up, the launch, one copy down.
struct HeteroItem { uint32_t group, problem; };
static int hetero_solve(int device, const std::vector<fk_topology*>& topos32, const std::vector<HeteroItem>& items,
                        const fk_problem* const* problems, double* const* free_values, fk_report* reports) {
    HeteroPool* pool = hetero_pool_for(device);
    std::lock_guard<std::mutex> lock(pool->mu);
    CU(cudaSetDevice(device));
    const size_t ng = topos32.size(), nj = items.size();
    std::vector<fk::DevProgram> progs;
    uint32_t max_state = 1;
    if (const int rc = hetero_programs(device, topos32, progs, &max_state); rc != FK_OK) return rc;
    // layout of the staging block: [programs][jobs][inputs: vars row + param row per job] | [outputs][reports]
    std::vector<fk::HeteroJob> jobs(nj);
    size_t in_doubles = 0, out_doubles = 0;
    for (size_t k = 0; k < nj; k++) {
        const fk::Topology& t = topos32[items[k].group]->t;
        jobs[k].prog = items[k].group; jobs[k].pad = 0;
        jobs[k].vars_off = in_doubles; in_doubles += t.n_vars;
        jobs[k].param_off = in_doubles; in_doubles += t.n_expr;
        jobs[k].out_off = out_doubles; out_doubles += t.n_free;
    }
    BlockLayout blk;
    const size_t o_progs = blk.put(ng * sizeof(fk::DevProgram)), o_jobs = blk.put(nj * sizeof(fk::HeteroJob));
    const size_t o_in = blk.put(in_doubles * sizeof(double)), o_out = blk.put(out_doubles * sizeof(double)), o_rep = blk.put(nj * sizeof(fk_report));
    const size_t total = blk.end, alloc = std::max<size_t>(total + total / 2, 1 << 20);
    int grc = pool->h.reserve(total, alloc);
    if (grc == FK_OK) grc = pool->d.reserve(total, alloc);
    if (grc != FK_OK) return grc;
    if (!pool->stream) CU(cudaStreamCreateWithFlags(&pool->stream, cudaStreamNonBlocking));
    std::memcpy(pool->h + o_progs, progs.data(), ng * sizeof(fk::DevProgram));
    std::memcpy(pool->h + o_jobs, jobs.data(), nj * sizeof(fk::HeteroJob));
    double* in = reinterpret_cast<double*>(pool->h + o_in);
    for (size_t k = 0; k < nj; k++) {
        const fk::Topology& t = topos32[items[k].group]->t;
        const fk_problem* p = problems[items[k].problem];
        double* v = in + jobs[k].vars_off;
        if (t.n_vars) std::memcpy(v, p->vars, sizeof(double) * t.n_vars);
        for (uint32_t f = 0; f < t.n_free; f++) v[t.free_vars[f]] = free_values[items[k].problem][f];
        double* q = in + jobs[k].param_off;
        if (t.n_expr) {
            if (p->param) std::memcpy(q, p->param, sizeof(double) * t.n_expr);
            else std::fill(q, q + t.n_expr, 0.0);
        }
    }
    CU(cudaMemcpyAsync(pool->d, pool->h, o_out, cudaMemcpyHostToDevice, pool->stream));
    const int rc = hetero_launch(reinterpret_cast<const fk::DevProgram*>(pool->d + o_progs), reinterpret_cast<const fk::HeteroJob*>(pool->d + o_jobs),
                                 nj, max_state, reinterpret_cast<const double*>(pool->d + o_in), reinterpret_cast<double*>(pool->d + o_out),
                                 reinterpret_cast<fk_report*>(pool->d + o_rep), pool->stream);
    if (rc != FK_OK) return rc;
    CU(cudaMemcpyAsync(pool->h + o_out, pool->d + o_out, total - o_out, cudaMemcpyDeviceToHost, pool->stream));
    CU(cudaStreamSynchronize(pool->stream));
    const double* out = reinterpret_cast<const double*>(pool->h + o_out);
    const fk_report* reps = reinterpret_cast<const fk_report*>(pool->h + o_rep);
    for (size_t k = 0; k < nj; k++) {
        const fk::Topology& t = topos32[items[k].group]->t;
        if (t.n_free) std::memcpy(free_values[items[k].problem], out + jobs[k].out_off, sizeof(double) * t.n_free);
        if (reports) reports[items[k].problem] = reps[k];
    }
    return FK_OK;
}

// The problems of a batch call, grouped by structure: one topology per group, from the cache or analysed on host threads.
struct BatchGroup {
    uint64_t sig = 0;
    std::shared_ptr<fk_topology> topo;
    std::vector<uint32_t> members;
    int rc = FK_OK;
    std::string err;
    // staging of the group's uniform batch
    std::vector<double> vars, param, out;
    std::vector<fk_report> reps;
    int device = 0;
    bool done = false;  // solved by the heterogeneous launch
};
static int group_by_topology(uint32_t n, const fk_problem* const* problems, double* const* free_values, std::vector<BatchGroup>& groups) {
    // ---- group the problems by topology -----------------------------------------------------------------
    std::multimap<uint64_t, size_t> by_sig;
    for (uint32_t i = 0; i < n; i++) {
        const fk_problem* p = problems[i];
        if (!p || !free_values[i]) return fail(FK_ERR_INVALID, "null problem in batch");
        if (!problem_arrays_ok(*p)) return fail(FK_ERR_INVALID, "null array in fk_problem");
        const uint64_t sig = structural_signature(*p);
        size_t gi = SIZE_MAX;
        auto range = by_sig.equal_range(sig);
        for (auto it = range.first; it != range.second && gi == SIZE_MAX; ++it)
            if (same_structure(*problems[groups[it->second].members[0]], *p)) gi = it->second;
        if (gi == SIZE_MAX) {
            groups.emplace_back();
            groups.back().sig = sig;
            gi = groups.size() - 1;
            by_sig.emplace(sig, gi);
        }
        groups[gi].members.push_back(i);
    }
    // ---- topologies: cache first, the misses are analysed on host threads ------------------------------------
    std::vector<size_t> missing;
    for (size_t g = 0; g < groups.size(); g++) {
        groups[g].topo = cache_lookup(groups[g].sig, *problems[groups[g].members[0]]);
        if (!groups[g].topo) missing.push_back(g);
    }
    if (!missing.empty()) {
        auto build_one = [&](size_t g) {
            fk_topology* t = nullptr;
            groups[g].rc = fk_topology_create(problems[groups[g].members[0]], &t);
            if (groups[g].rc != FK_OK) groups[g].err = g_error;
            else groups[g].topo.reset(t, fk_topology_destroy);
        };
        const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
        const size_t workers = std::min<size_t>(missing.size(), hw);
        if (workers <= 1) {
            for (size_t g : missing) build_one(g);
        } else {
            std::atomic<size_t> next{0};
            std::vector<std::thread> pool;
            for (size_t w = 0; w < workers; w++)
                pool.emplace_back([&] {
                    for (size_t k = next++; k < missing.size(); k = next++) build_one(missing[k]);
                });
            for (auto& th : pool) th.join();
        }
        for (size_t g : missing) {
            if (groups[g].rc != FK_OK) return fail(groups[g].rc, groups[g].err);
            cache_insert(groups[g].sig, groups[g].topo);
        }
    }
    return FK_OK;
}

// The group's members as one uniform batch (their free values written into their variable rows; no parameters: zeros).
static void stage_group(BatchGroup& gr, const fk_problem* const* problems, double* const* free_values) {
    const fk::Topology& t = gr.topo->t;
    const size_t cnt = gr.members.size();
    gr.vars.resize(cnt * t.n_vars); gr.param.resize(cnt * std::max<uint32_t>(t.n_expr, 1)); gr.out.resize(cnt * std::max<uint32_t>(t.n_free, 1));
    gr.reps.resize(cnt);
    for (size_t k = 0; k < cnt; k++) {
        const fk_problem* p = problems[gr.members[k]];
        if (t.n_vars) std::memcpy(&gr.vars[k * t.n_vars], p->vars, sizeof(double) * t.n_vars);
        for (uint32_t f = 0; f < t.n_free; f++) gr.vars[k * t.n_vars + t.free_vars[f]] = free_values[gr.members[k]][f];
        if (t.n_expr) {
            if (p->param) std::memcpy(&gr.param[k * t.n_expr], p->param, sizeof(double) * t.n_expr);
            else std::fill(gr.param.begin() + k * t.n_expr, gr.param.begin() + (k + 1) * t.n_expr, 0.0);
        }
    }
}
static void unstage_group(const BatchGroup& gr, double* const* free_values, fk_report* reports) {
    const fk::Topology& t = gr.topo->t;
    for (size_t k = 0; k < gr.members.size(); k++) {
        std::memcpy(free_values[gr.members[k]], &gr.out[k * t.n_free], sizeof(double) * t.n_free);
        if (reports) reports[gr.members[k]] = gr.reps[k];
    }
}

int fk_lm_solve_batch(uint32_t n, const fk_problem* const* problems, double* const* free_values, fk_report* reports,
                      int n_gpus) {
    if (n == 0) return FK_OK;
    if (!problems || !free_values) return fail(FK_ERR_INVALID, "null argument");
    if (const int rc = clamp_gpus(n_gpus); rc != FK_OK) return rc;
    std::vector<BatchGroup> groups;
    if (const int rc = group_by_topology(n, problems, free_values, groups); rc != FK_OK) return rc;
    int cur = 0;
    if (cudaGetDevice(&cur) != cudaSuccess) cur = 0;
    // ---- solve.  With several devices and at least as many groups, whole groups go to devices round robin; otherwise
    // every large group is sharded by sketch over the devices (fk_batch_solve).
    const bool groups_to_devices = n_gpus > 1 && groups.size() >= (size_t)n_gpus;
    size_t rr = 0;
    int first_rc = FK_OK;
    std::string first_err;
    auto note = [&](int rc) { if (rc != FK_OK && first_rc == FK_OK) { first_rc = rc; first_err = g_error; } };
    // Several small groups: ONE launch of the heterogeneous kernel for all of them (one warp per system) instead of one
    // launch, two copies and a synchronisation per topology.  Groups of 64 systems and more keep the uniform batch kernels
    // (from there the sketch-per-thread kernel is the faster one).  (FK_NO_HETERO=1: A/B knob.)
    {
        static const bool no_hetero = std::getenv("FK_NO_HETERO") != nullptr;
        std::vector<size_t> small;
        for (size_t g = 0; g < groups.size(); g++) {
            if (hetero_fits(groups[g].topo->t, groups[g].members.size())) small.push_back(g);
        }
        if (!no_hetero && small.size() >= 2) {
            std::vector<fk_topology*> topos32;
            std::vector<HeteroItem> items;
            for (size_t q = 0; q < small.size(); q++) {
                BatchGroup& gr = groups[small[q]];
                fk_topology* t32 = hetero_topology(gr.topo.get(), gr.members.size());
                if (!t32) continue;
                for (uint32_t i : gr.members) items.push_back({(uint32_t)topos32.size(), i});
                topos32.push_back(t32);
                gr.done = true;
            }
            if (!items.empty() && n_gpus > 1 && items.size() >= 64u * (size_t)n_gpus) {
                // several devices: contiguous shares of the systems, one host thread and one launch per device
                note(shard_over_devices(n_gpus, (uint32_t)items.size(), [&](int device, uint32_t lo, uint32_t hi) {
                    const std::vector<HeteroItem> part(items.begin() + lo, items.begin() + hi);
                    return hetero_solve(device, topos32, part, problems, free_values, reports);
                }));
            } else if (!items.empty()) {
                note(hetero_solve(cur, topos32, items, problems, free_values, reports));
            }
        }
    }
    for (BatchGroup& gr : groups) {
        if (gr.done || gr.topo->t.path == 2) continue;  // (large systems below)
        stage_group(gr, problems, free_values);
        gr.device = groups_to_devices ? (int)(rr++ % (size_t)n_gpus) : cur;
    }
    for (BatchGroup& gr : groups) {
        if (gr.done) continue;
        const fk::Topology& t = gr.topo->t;
        const size_t cnt = gr.members.size();
        if (t.path == 2) {  // large systems: one after the other through the global sparse path
            for (uint32_t i : gr.members) {
                note(fk_topology_lm_solve(gr.topo.get(), problems[i]->vars, problems[i]->param, free_values[i], reports ? &reports[i] : nullptr));
            }
            continue;
        }
        const int rc = groups_to_devices || n_gpus == 1 || small_fits(t, (uint32_t)cnt)
            ? run_device_range(gr.topo.get(), gr.device, 0, (uint32_t)cnt, gr.vars.data(), gr.param.data(), gr.out.data(), gr.reps.data())
            : solve_sharded(gr.topo.get(), (uint32_t)cnt, gr.vars.data(), gr.param.data(), gr.out.data(), gr.reps.data(), n_gpus, 0);
        if (rc != FK_OK) { note(rc); continue; }
        unstage_group(gr, free_values, reports);
    }
    if (cudaSetDevice(cur) != cudaSuccess) cudaGetLastError();
    return first_rc == FK_OK ? FK_OK : fail(first_rc, first_err);
}

int fk_lbfgs_solve_batch(uint32_t n, const fk_problem* const* problems, double* const* free_values, fk_report* reports, int n_gpus) {
    if (n == 0) return FK_OK;
    if (!problems || !free_values) return fail(FK_ERR_INVALID, "null argument");
    if (const int rc = clamp_gpus(n_gpus); rc != FK_OK) return rc;
    std::vector<BatchGroup> groups;
    if (const int rc = group_by_topology(n, problems, free_values, groups); rc != FK_OK) return rc;
    int cur = 0;
    if (cudaGetDevice(&cur) != cudaSuccess) cur = 0;
    // With several devices and at least as many groups, whole groups go to devices round robin; otherwise every large group
    // is sharded by sketch over the devices.
    const bool groups_to_devices = n_gpus > 1 && groups.size() >= (size_t)n_gpus;
    size_t rr = 0;
    int first_rc = FK_OK;
    std::string first_err;
    for (BatchGroup& gr : groups) {
        stage_group(gr, problems, free_values);
        gr.device = groups_to_devices ? (int)(rr++ % (size_t)n_gpus) : cur;
        const uint32_t cnt = (uint32_t)gr.members.size();
        const int rc = groups_to_devices || n_gpus == 1 || small_fits(gr.topo->t, cnt)
            ? run_device_range(gr.topo.get(), gr.device, 0, cnt, gr.vars.data(), gr.param.data(), gr.out.data(), gr.reps.data(), 1)
            : solve_sharded(gr.topo.get(), cnt, gr.vars.data(), gr.param.data(), gr.out.data(), gr.reps.data(), n_gpus, 1);
        if (rc == FK_OK) unstage_group(gr, free_values, reports);
        else if (first_rc == FK_OK) { first_rc = rc; first_err = g_error; }
        std::vector<double>().swap(gr.vars);  // (large systems: one group's staging at a time)
        std::vector<double>().swap(gr.out);
    }
    if (cudaSetDevice(cur) != cudaSuccess) cudaGetLastError();
    return first_rc == FK_OK ? FK_OK : fail(first_rc, first_err);
}

int fk_lbfgs_solve(const fk_problem* problem, double* free_values, fk_report* report) {
    const fk_problem* ps[1] = {problem};
    double* fv[1] = {free_values};
    return fk_lbfgs_solve_batch(1, ps, fv, report, 1);
}

int fk_lm_solve(const fk_problem* problem, double* free_values, fk_report* report) {
    const fk_problem* ps[1] = {problem};
    double* fv[1] = {free_values};
    return fk_lm_solve_batch(1, ps, fv, report, 1);
}

}  // extern "C"

// ---- fk_system_batch_solve: System::solve over n variants of one drawing -------------------------------------------
namespace fk {

int system_batch_fail(int code, const std::string& msg) { return fail(code, msg); }

// The problems grouped by structure, one topology per group (group_by_topology without free values).
static int group_by_structure(const std::vector<const fk_problem*>& problems, std::vector<BatchGroup>& groups) {
    if (problems.empty()) return FK_OK;
    static double dummy = 0.0;  // (group_by_topology checks the free-value pointers; nothing is written through them)
    std::vector<double*> fv(problems.size(), &dummy);
    return group_by_topology((uint32_t)problems.size(), problems.data(), fv.data(), groups);
}

// Variants per chunk of n: FK_SYSTEM_BATCH_CHUNK=n (test knob), else the chunk's buffers (`bytes` per variant) within about 1 GiB
// of device memory, at least one; then at most INT32_MAX sketches per launch (`sketches` per variant) and rows of `row` values
// per variant within 32-bit offsets.
static uint32_t system_batch_chunk_env() {  // FK_SYSTEM_BATCH_CHUNK, read once (0: not set)
    static const uint32_t env = [] {
        const char* e = std::getenv("FK_SYSTEM_BATCH_CHUNK");
        const long v = e ? std::atol(e) : 0;
        return (uint32_t)(v >= 1 && v <= (long)UINT32_MAX ? v : 0);
    }();
    return env;
}
static uint32_t system_batch_chunk(uint32_t n, uint64_t bytes, uint64_t sketches, uint64_t row) {
    const uint32_t env = system_batch_chunk_env();
    uint64_t chunk = env ? env : std::max<uint64_t>(1, (1ull << 30) / bytes);
    chunk = std::min<uint64_t>(chunk, std::max<uint64_t>(1, (uint64_t)INT32_MAX / std::max<uint64_t>(1, sketches)));
    chunk = std::min<uint64_t>(chunk, std::max<uint64_t>(1, (uint64_t)UINT32_MAX / std::max<uint64_t>(1, row)));
    return (uint32_t)std::min<uint64_t>(chunk, n);
}

// The state of a system batch call on one device, all on one stream: the layout's tables, the template rows and the grow-only chunk
// buffers.  d_vt / d_pt: the variants' scaled variables and parameters where the call keeps them resident (not
// fk_system_batch_solve).  The caller holds mu.
struct SystemDevice {
    std::mutex mu;
    int device = -1;
    cudaStream_t stream = nullptr;
    bool ready = false;  // tables uploaded
    void* d_tables = nullptr;
    double *d_tmpl_vars = nullptr, *d_tmpl_param = nullptr;
    GrowBuf<double> d_raw_param, d_vt, d_pt;
    // Once per device: the stream, the tables of `pk` and the template rows (an earlier failed attempt's are freed first).
    int upload_tables(int dev, TablePack& pk, uint32_t n_vars, uint32_t n_expr) {
        device = dev;
        if (!stream) CU(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        cudaFree(d_tables); cudaFree(d_tmpl_vars); cudaFree(d_tmpl_param);
        d_tables = nullptr;
        d_tmpl_vars = d_tmpl_param = nullptr;
        const int rc = pk.upload(stream, &d_tables);
        if (rc != FK_OK) return rc;
        CU(cudaMalloc(&d_tmpl_vars, sizeof(double) * std::max<uint32_t>(n_vars, 1)));
        CU(cudaMalloc(&d_tmpl_param, sizeof(double) * std::max<uint32_t>(n_expr, 1)));
        return FK_OK;
    }
    ~SystemDevice() {
        if (device < 0) return;
        cudaSetDevice(device);
        cudaFree(d_tables); cudaFree(d_tmpl_vars); cudaFree(d_tmpl_param);
        if (stream) cudaStreamDestroy(stream);
    }
};

// The template rows up, then body(at, cnt) for the chunks [at, at + cnt) of variants [lo, hi) on d's stream, then a synchronise
// whether or not one failed: no copy into the caller's buffers may still be running when the call returns.  `what` names a
// failure the synchronise reports.
template <class Chunk>
static int run_chunks(SystemDevice* d, uint32_t n_vars, uint32_t n_expr, const double* tmpl_vars, const double* tmpl_param, uint32_t lo,
                      uint32_t hi, uint32_t chunk, const char* what, const Chunk& body) {
    auto run = [&]() -> int {
        if (n_vars) CU(cudaMemcpyAsync(d->d_tmpl_vars, tmpl_vars, sizeof(double) * n_vars, cudaMemcpyHostToDevice, d->stream));
        if (n_expr) CU(cudaMemcpyAsync(d->d_tmpl_param, tmpl_param, sizeof(double) * n_expr, cudaMemcpyHostToDevice, d->stream));
        for (uint32_t at = lo; at < hi; at += chunk) {
            const int rc = body(at, std::min(chunk, hi - at));
            if (rc != FK_OK) return rc;
        }
        return FK_OK;
    };
    int rc = run();
    const cudaError_t e = cudaStreamSynchronize(d->stream);
    if (rc == FK_OK && e != cudaSuccess) rc = cuda_fail(e, what);
    return rc;
}

// The solve batches' device state: the prepare kernel's tables and descriptors (d_desc), the structures' batch plans, and the
// chunk's raw, scale and output rows.  Plus, for fk_system_batch_solve, the scatter kernel's tables.
struct SystemBatchDevice : SystemDevice {
    uint32_t chunk = 0;  // variants the plans and chunk buffers hold
    bool lm = false;  // the plans were made for LM (which on the global sparse path needs the sparse batch tables)
    std::vector<std::unique_ptr<fk_batch_plan>> plans;
    const uint8_t* d_kind = nullptr;
    const uint32_t *d_expr_con = nullptr, *d_var_struct = nullptr, *d_var_off = nullptr, *d_comp_struct = nullptr, *d_comp_member = nullptr;
    const double* d_draws = nullptr;
    std::vector<SbStructure> desc;  // (host copy; the buffer pointers change with the plans)
    GrowBuf<SbStructure> d_desc;
    GrowBuf<double> d_raw_vars, d_scales, d_vars_out;
    GrowBuf<fk_report> d_rep_out;

    // The plans and chunk buffers of `cap` variants, the plans made again (and dropped after a failure): per structure s a plan of
    // cap * st[s].mult sketches, the raw, scale and output rows with n_rep reports per variant, and with `resident` vt and pt.
    template <class Structure>
    int grow_chunk(const SystemBatchLayout& L, const std::vector<Structure>& st, uint32_t cap, bool lm_plans, uint32_t n_rep, bool resident) {
        plans.clear();
        chunk = 0;
        int rc = FK_OK;
        for (size_t s = 0; s < st.size() && rc == FK_OK; s++) {
            fk_batch_plan* p = nullptr;
            if ((rc = plan_create(st[s].topo.get(), cap * st[s].mult, device, lm_plans, &p)) == FK_OK) plans.emplace_back(p);
        }
        if (rc == FK_OK) rc = d_raw_vars.reserve((size_t)cap * L.n_vars);
        if (rc == FK_OK) rc = d_raw_param.reserve((size_t)cap * L.n_constraints);
        if (rc == FK_OK) rc = d_scales.reserve(cap);
        if (rc == FK_OK) rc = d_vars_out.reserve((size_t)cap * L.n_vars);
        if (rc == FK_OK) rc = d_rep_out.reserve((size_t)cap * n_rep);
        if (rc == FK_OK && resident) rc = d_vt.reserve((size_t)cap * L.n_vars);
        if (rc == FK_OK && resident) rc = d_pt.reserve((size_t)cap * L.kind.size());
        if (rc == FK_OK) rc = d_desc.reserve(desc.size());
        if (rc != FK_OK) {
            plans.clear();
            return rc;
        }
        chunk = cap;
        lm = lm_plans;
        return FK_OK;
    }
};

// Bytes per variant of the structures' plan rows (st[s].mult sketches each); *max_mult: the most sketches per variant of one plan.
template <class Structure>
static uint64_t plan_bytes(const std::vector<Structure>& st, uint64_t* max_mult) {
    uint64_t bytes = 0;
    *max_mult = 1;
    for (const Structure& S : st) {
        const fk::Topology& t = S.topo->t;
        bytes += S.mult * (sizeof(double) * ((uint64_t)t.n_vars + t.n_expr + t.n_free) + sizeof(fk_report));
        *max_mult = std::max<uint64_t>(*max_mult, S.mult);
    }
    return bytes;
}

// Variants [lo, hi) of a solve batch on one device, chunk after chunk on its stream: the raw rows up, the prepare kernel over the
// n_desc descriptors of d_desc, step(cnt, raw, raw_stride) (the solves and the write-back into d_vars_out / d_rep_out), then
// vars_out and n_rep reports per variant down.
template <class Step>
static int solve_chunks(SystemBatchDevice* d, const SystemBatchLayout& L, const SystemBatchCall& c, uint32_t lo, uint32_t hi, uint32_t chunk,
                        uint32_t n_rep, uint32_t n_desc, const char* what, const Step& step) {
    const uint32_t n_expr = (uint32_t)L.kind.size();
    const cudaStream_t st = d->stream;
    return run_chunks(d, L.n_vars, n_expr, c.tmpl_vars, c.tmpl_param, lo, hi, chunk, what, [&](uint32_t at, uint32_t cnt) -> int {
        const double* raw = d->d_tmpl_vars;
        uint32_t raw_stride = 0;
        if (c.vars) {
            if (L.n_vars)
                CU(cudaMemcpyAsync(d->d_raw_vars, c.vars + (size_t)at * L.n_vars, sizeof(double) * (size_t)cnt * L.n_vars, cudaMemcpyHostToDevice, st));
            raw = d->d_raw_vars;
            raw_stride = L.n_vars;
        }
        if (c.params && L.n_constraints)
            CU(cudaMemcpyAsync(d->d_raw_param, c.params + (size_t)at * L.n_constraints, sizeof(double) * (size_t)cnt * L.n_constraints,
                               cudaMemcpyHostToDevice, st));
        const int e = launch_system_batch_prepare(cnt, L.n_vars, n_expr, L.n_constraints, d->d_kind, d->d_expr_con, d->d_draws, c.perturb, raw,
                                                  raw_stride, c.params ? d->d_raw_param.get() : nullptr, d->d_tmpl_param, n_desc, d->d_desc, d->d_scales, st);
        if (e != 0) return cuda_fail((cudaError_t)e, "launch fk_system_batch_prepare_kernel");
        const int rc = step(cnt, raw, raw_stride);
        if (rc != FK_OK) return rc;
        if (L.n_vars)
            CU(cudaMemcpyAsync(c.vars_out + (size_t)at * L.n_vars, d->d_vars_out, sizeof(double) * (size_t)cnt * L.n_vars, cudaMemcpyDeviceToHost, st));
        if (n_rep)
            CU(cudaMemcpy2DAsync(c.reports + (size_t)at * c.reports_per_variant, sizeof(fk_report) * c.reports_per_variant, d->d_rep_out,
                                 sizeof(fk_report) * n_rep, sizeof(fk_report) * n_rep, cnt, cudaMemcpyDeviceToHost, st));
        return FK_OK;
    });
}

struct SystemBatch {
    SystemBatchLayout L;
    struct Structure {
        std::shared_ptr<fk_topology> topo;
        std::vector<uint32_t> members;                    // component indices
        uint32_t mult = 0;                                // members.size(): the plan's sketches per variant
        std::vector<uint32_t> slot_var, slot_draw, expr;  // [mult][nv], [mult][nv], [mult][ne]
    };
    std::vector<Structure> st;
    std::vector<uint32_t> comp_struct, comp_member;  // per component
    std::vector<uint32_t> var_struct, var_off;       // per system variable: structure solving it (kSbNone: none), offset in the variant's block
    std::mutex mu;
    std::map<int, std::unique_ptr<SystemBatchDevice>> devices;
};

int system_batch_create(SystemBatchLayout&& layout, const std::vector<const fk_problem*>& problems, std::shared_ptr<SystemBatch>* out) {
    std::shared_ptr<SystemBatch> b = std::make_shared<SystemBatch>();
    b->L = std::move(layout);
    const SystemBatchLayout& L = b->L;
    const uint32_t nc = (uint32_t)problems.size();
    std::vector<BatchGroup> groups;
    const int rc = group_by_structure(problems, groups);
    if (rc != FK_OK) return rc;
    b->comp_struct.assign(nc, kSbNone);
    b->comp_member.assign(nc, 0);
    b->var_struct.assign(L.n_vars, kSbNone);
    b->var_off.assign(L.n_vars, 0);
    for (BatchGroup& g : groups) {
        SystemBatch::Structure S;
        S.topo = g.topo;
        S.members = g.members;
        S.mult = (uint32_t)g.members.size();
        const uint32_t si = (uint32_t)b->st.size(), nf = g.topo->t.n_free;
        for (uint32_t m = 0; m < S.members.size(); m++) {
            const SystemBatchLayout::Component& c = L.comps[S.members[m]];
            S.slot_var.insert(S.slot_var.end(), c.slot_var.begin(), c.slot_var.end());
            S.slot_draw.insert(S.slot_draw.end(), c.slot_draw.begin(), c.slot_draw.end());
            S.expr.insert(S.expr.end(), c.expr.begin(), c.expr.end());
            b->comp_struct[S.members[m]] = si;
            b->comp_member[S.members[m]] = m;
            for (uint32_t f = 0; f < c.free_var.size(); f++) {
                b->var_struct[c.free_var[f]] = si;
                b->var_off[c.free_var[f]] = m * nf + f;
            }
        }
        b->st.push_back(std::move(S));
    }
    *out = std::move(b);
    return FK_OK;
}

void system_batch_layout(const SystemBatch& b, uint32_t* n_components, uint32_t* n_structures, std::vector<uint32_t>* multiplicity) {
    if (n_components) *n_components = (uint32_t)b.L.comps.size();
    if (n_structures) *n_structures = (uint32_t)b.st.size();
    if (multiplicity) {
        multiplicity->clear();
        for (const SystemBatch::Structure& S : b.st) multiplicity->push_back(S.mult);
    }
}

// Tables once per device; plans and chunk buffers grow with the chunk (and are made again when LM follows L-BFGS).  *chunk: the
// variants per chunk for n variants.  The caller holds d->mu.
static int system_batch_device(SystemBatch& b, SystemBatchDevice* d, int device, uint32_t n, bool lm, uint32_t* chunk) {
    CU(cudaSetDevice(device));
    const SystemBatchLayout& L = b.L;
    const uint32_t ns = (uint32_t)b.st.size(), nc = (uint32_t)L.comps.size();
    if (!d->ready) {
        TablePack pk;
        const size_t o_kind = pk.add(L.kind), o_con = pk.add(L.expr_constraint), o_draws = pk.add(L.draws), o_vs = pk.add(b.var_struct),
                     o_vo = pk.add(b.var_off), o_cs = pk.add(b.comp_struct), o_cm = pk.add(b.comp_member);
        std::vector<size_t> o_sv(ns), o_sd(ns), o_ex(ns);
        for (uint32_t s = 0; s < ns; s++) {
            o_sv[s] = pk.add(b.st[s].slot_var);
            o_sd[s] = pk.add(b.st[s].slot_draw);
            o_ex[s] = pk.add(b.st[s].expr);
        }
        const int rc = d->upload_tables(device, pk, L.n_vars, (uint32_t)L.kind.size());
        if (rc != FK_OK) return rc;
        d->d_kind = pk.at<uint8_t>(o_kind);
        d->d_expr_con = pk.at<uint32_t>(o_con);
        d->d_draws = pk.at<double>(o_draws);
        d->d_var_struct = pk.at<uint32_t>(o_vs); d->d_var_off = pk.at<uint32_t>(o_vo);
        d->d_comp_struct = pk.at<uint32_t>(o_cs); d->d_comp_member = pk.at<uint32_t>(o_cm);
        d->desc.assign(ns, SbStructure{});
        for (uint32_t s = 0; s < ns; s++) {
            const fk::Topology& tp = b.st[s].topo->t;
            SbStructure& S = d->desc[s];
            S.slot_var = pk.at<uint32_t>(o_sv[s]); S.slot_draw = pk.at<uint32_t>(o_sd[s]); S.expr = pk.at<uint32_t>(o_ex[s]);
            S.nv = tp.n_vars; S.ne = tp.n_expr; S.nf = tp.n_free; S.mult = b.st[s].mult;
        }
        d->ready = true;
    }
    // per variant: the raw rows, its scale, vars_out and a report per component, and the plans' rows
    uint64_t mult = 1;
    const uint64_t bytes = sizeof(double) * (2ull * L.n_vars + L.n_constraints + 1) + sizeof(fk_report) * (uint64_t)nc + plan_bytes(b.st, &mult);
    *chunk = system_batch_chunk(n, bytes, mult, std::max({L.n_vars, L.n_constraints, nc}));
    if (d->chunk >= *chunk && (d->lm || !lm) && d->plans.size() == ns) return FK_OK;
    const int rc = d->grow_chunk(L, b.st, std::max(*chunk, d->chunk), lm, nc, false);
    if (rc != FK_OK) return rc;
    for (uint32_t s = 0; s < ns; s++) {
        const fk_batch_plan* p = d->plans[s].get();
        SbStructure& S = d->desc[s];
        S.vars = p->d_vars; S.params = p->d_params; S.out = p->d_out; S.reps = p->d_rep;
    }
    if (ns) CU(cudaMemcpyAsync(d->d_desc, d->desc.data(), sizeof(SbStructure) * ns, cudaMemcpyHostToDevice, d->stream));
    CU(cudaStreamSynchronize(d->stream));  // (desc may change before a later call's copy)
    return FK_OK;
}

// Variants [lo, hi) on one device: per chunk the prepare kernel (gather into every structure's rows), one launch per structure
// and the scatter kernel.
static int system_batch_range(SystemBatch& b, const SystemBatchCall& c, int device, uint32_t lo, uint32_t hi) {
    const SystemBatchLayout& L = b.L;
    const uint32_t ns = (uint32_t)b.st.size(), nc = (uint32_t)L.comps.size();
    const uint32_t n_rep = c.reports ? std::min(c.reports_per_variant, nc) : 0;
    SystemBatchDevice* d = device_slot(b.mu, b.devices, device);
    std::lock_guard<std::mutex> lock(d->mu);
    uint32_t chunk = 0;
    const int rc = system_batch_device(b, d, device, hi - lo, c.optimizer == 0, &chunk);
    if (rc != FK_OK) return rc;
    return solve_chunks(d, L, c, lo, hi, chunk, n_rep, ns, "fk_system_batch_solve kernels / copies",
                        [&](uint32_t cnt, const double* raw, uint32_t raw_stride) -> int {
                            for (uint32_t s = 0; s < ns; s++) {
                                fk_batch_plan* p = d->plans[s].get();
                                p->n = cnt * b.st[s].mult;
                                const int r = plan_solve(p, solve_kernel(p->topo, c.optimizer, p->n), d->stream);
                                if (r != FK_OK) return r;
                            }
                            const int e = launch_system_batch_scatter(cnt, L.n_vars, raw, raw_stride, d->d_scales, d->d_var_struct, d->d_var_off, n_rep,
                                                                      d->d_comp_struct, d->d_comp_member, d->d_desc, d->d_vars_out, d->d_rep_out, d->stream);
                            return e != 0 ? cuda_fail((cudaError_t)e, "launch fk_system_batch_scatter_kernel") : FK_OK;
                        });
}

int system_batch_solve(SystemBatch& b, const SystemBatchCall& c) {
    if (c.optimizer == 0)  // LM on the global sparse path: the front limit of fk_batch_solve
        for (const SystemBatch::Structure& S : b.st)
            if (S.topo->t.path == 2 && S.topo->sb_check() != FK_OK)
                return fail(FK_ERR_TOO_LARGE, "component " + std::to_string(S.members[0]) + ": " + S.topo->sb_err +
                                                  "; Optimizer::LBfgs takes systems of every size");
    if (c.n == 0) return FK_OK;
    int n_gpus = c.n_gpus;
    const int rc = clamp_gpus(n_gpus);
    if (rc != FK_OK) return rc;
    return shard_over_devices(n_gpus, c.n, [&](int device, uint32_t lo, uint32_t hi) { return system_batch_range(b, c, device, lo, hi); });
}

// ---- fk_system_batch_solve_single_pass: Decomposer::SinglePass over n variants of one drawing ---------------------------
// (fk_system_batch_solve_recursive_assembly runs on the same plan: its steps in place of the sets, with their moves.)
// The solve batches' device state plus the per-wave descriptors of the gather / scatter kernel.  The resident rows vt and pt are
// what the waves read and write; d_desc holds the one identity structure through which the prepare kernel writes them.  Plans are
// one per structure (capacity chunk * the structure's most sets in one wave).
struct SystemSpDevice : SystemBatchDevice {
    const uint8_t* d_solved = nullptr;
    const uint32_t *d_pvar = nullptr, *d_pdraw = nullptr;  // the perturbations of waves >= 1, wave after wave
    std::vector<uint32_t> pert_off;                        // [n_waves + 1]
    std::vector<SpGroup> groups;                           // (host copy) every wave's groups, wave after wave
    std::vector<uint32_t> group_off;                       // [n_waves + 1]
    GrowBuf<SpGroup> d_groups;
};

struct SystemSpBatch {
    SystemBatchLayout L;  // comps: the sets
    struct Structure {
        std::shared_ptr<fk_topology> topo;
        std::vector<uint32_t> members;  // set indices
        uint32_t mult = 0;              // most sets of the structure in one wave: the plan's sketches per variant
    };
    std::vector<Structure> st;
    std::vector<uint32_t> set_struct;
    struct Group {  // the sets of one structure in one wave, in plan order: the tables of its SpGroup
        uint32_t structure = 0;
        std::vector<uint32_t> sets, slot_var, expr, free_var, move_off{0}, moves;
    };
    std::vector<std::vector<Group>> waves;
    std::vector<std::vector<uint32_t>> wave_perturb;  // variables whose perturbation runs at the start of wave w >= 1
    std::vector<uint8_t> solved;                      // per system variable: some set solves it (or a step moves it)
    std::mutex mu;
    std::map<int, std::unique_ptr<SystemSpDevice>> devices;
};

int system_sp_batch_create(SystemBatchLayout&& layout, const std::vector<const fk_problem*>& problems, std::shared_ptr<SystemSpBatch>* out) {
    std::shared_ptr<SystemSpBatch> b = std::make_shared<SystemSpBatch>();
    b->L = std::move(layout);
    const SystemBatchLayout& L = b->L;
    const uint32_t n_sets = (uint32_t)problems.size();
    std::vector<BatchGroup> groups;
    const int rc = group_by_structure(problems, groups);
    if (rc != FK_OK) return rc;
    b->set_struct.assign(n_sets, kSbNone);
    for (BatchGroup& g : groups) {
        for (uint32_t k : g.members) b->set_struct[k] = (uint32_t)b->st.size();
        b->st.push_back({g.topo, g.members, 0});
    }
    b->waves.assign(L.n_waves, {});
    b->solved.assign(L.n_vars, 0);
    for (uint32_t k = 0; k < n_sets; k++) {
        std::vector<SystemSpBatch::Group>& wave = b->waves[L.comp_wave[k]];
        const uint32_t si = b->set_struct[k];
        auto it = std::find_if(wave.begin(), wave.end(), [&](const SystemSpBatch::Group& g) { return g.structure == si; });
        if (it == wave.end()) {
            wave.emplace_back();
            wave.back().structure = si;
            it = wave.end() - 1;
        }
        const SystemBatchLayout::Component& c = L.comps[k];
        it->sets.push_back(k);
        it->slot_var.insert(it->slot_var.end(), c.slot_var.begin(), c.slot_var.end());
        it->expr.insert(it->expr.end(), c.expr.begin(), c.expr.end());
        it->free_var.insert(it->free_var.end(), c.free_var.begin(), c.free_var.end());
        it->moves.insert(it->moves.end(), c.moves.begin(), c.moves.end());
        it->move_off.push_back((uint32_t)(it->moves.size() / 2));
        b->st[si].mult = std::max(b->st[si].mult, (uint32_t)it->sets.size());
        for (uint32_t g : c.free_var)
            if (g != kSbNone) b->solved[g] = 1;
        for (size_t m = 0; m < c.moves.size(); m += 2) b->solved[c.moves[m]] = b->solved[c.moves[m] + 1] = 1;
    }
    // (a perturbation scheduled behind the last wave precedes no set: nothing reads it, and vars_out keeps unsolved variables raw)
    b->wave_perturb.assign(L.n_waves, {});
    for (uint32_t i = 0; i < L.n_vars; i++)
        if (L.var_wave[i] != kSbNone && L.var_wave[i] > 0 && L.var_wave[i] < L.n_waves) b->wave_perturb[L.var_wave[i]].push_back(i);
    *out = std::move(b);
    return FK_OK;
}

void system_sp_batch_layout(const SystemSpBatch& b, uint32_t* n_sets, uint32_t* n_waves, uint32_t* n_structures,
                            std::vector<uint32_t>* set_wave, std::vector<uint32_t>* set_structure) {
    if (n_sets) *n_sets = (uint32_t)b.L.comps.size();
    if (n_waves) *n_waves = b.L.n_waves;
    if (n_structures) *n_structures = (uint32_t)b.st.size();
    if (set_wave) *set_wave = b.L.comp_wave;
    if (set_structure) *set_structure = b.set_struct;
}

// Tables once per device; plans, buffers and descriptors grow with the chunk.  *chunk: the variants per chunk for n variants.
// The caller holds d->mu.
static int system_sp_device(SystemSpBatch& b, SystemSpDevice* d, int device, uint32_t n, uint32_t* chunk) {
    CU(cudaSetDevice(device));
    const SystemBatchLayout& L = b.L;
    const uint32_t n_expr = (uint32_t)L.kind.size(), ns = (uint32_t)b.st.size(), nw = L.n_waves, n_sets = (uint32_t)L.comps.size();
    if (!d->ready) {
        // the identity structure of the prepare kernel: every variable (with its draw where the perturbation runs before any
        // set) and every expression
        std::vector<uint32_t> ident_var(L.n_vars), ident_draw(L.n_vars, kSbNone), ident_expr(n_expr);
        for (uint32_t i = 0; i < L.n_vars; i++) {
            ident_var[i] = i;
            if (L.var_wave[i] == 0) ident_draw[i] = L.var_draw[i];
        }
        for (uint32_t e = 0; e < n_expr; e++) ident_expr[e] = e;
        std::vector<uint32_t> pvar, pdraw;
        d->pert_off.assign(1, 0);
        for (uint32_t w = 0; w < nw; w++) {
            for (uint32_t i : b.wave_perturb[w]) {
                pvar.push_back(i);
                pdraw.push_back(L.var_draw[i]);
            }
            d->pert_off.push_back((uint32_t)pvar.size());
        }
        TablePack pk;
        const size_t o_kind = pk.add(L.kind), o_con = pk.add(L.expr_constraint), o_draws = pk.add(L.draws), o_iv = pk.add(ident_var),
                     o_id = pk.add(ident_draw), o_ie = pk.add(ident_expr), o_solved = pk.add(b.solved), o_pv = pk.add(pvar), o_pd = pk.add(pdraw);
        struct GroupAt { size_t sv, ex, fv, st, mo, mv; };
        std::vector<GroupAt> at;
        for (const auto& wave : b.waves)
            for (const SystemSpBatch::Group& g : wave)
                at.push_back({pk.add(g.slot_var), pk.add(g.expr), pk.add(g.free_var), pk.add(g.sets), pk.add(g.move_off), pk.add(g.moves)});
        const int rc = d->upload_tables(device, pk, L.n_vars, n_expr);
        if (rc != FK_OK) return rc;
        d->d_kind = pk.at<uint8_t>(o_kind);
        d->d_expr_con = pk.at<uint32_t>(o_con);
        d->d_draws = pk.at<double>(o_draws);
        d->d_solved = pk.at<uint8_t>(o_solved);
        d->d_pvar = pk.at<uint32_t>(o_pv); d->d_pdraw = pk.at<uint32_t>(o_pd);
        d->desc.assign(1, SbStructure{});
        SbStructure& I = d->desc[0];
        I.slot_var = pk.at<uint32_t>(o_iv); I.slot_draw = pk.at<uint32_t>(o_id); I.expr = pk.at<uint32_t>(o_ie);
        I.nv = L.n_vars; I.ne = n_expr; I.nf = 0; I.mult = 1;
        d->groups.clear();
        d->group_off.assign(1, 0);
        size_t q = 0;
        for (const auto& wave : b.waves) {
            for (const SystemSpBatch::Group& g : wave) {
                const fk::Topology& tp = b.st[g.structure].topo->t;
                SpGroup G{};
                G.s.slot_var = pk.at<uint32_t>(at[q].sv); G.s.expr = pk.at<uint32_t>(at[q].ex);
                G.free_var = pk.at<uint32_t>(at[q].fv); G.step = pk.at<uint32_t>(at[q].st);
                G.move_off = pk.at<uint32_t>(at[q].mo); G.moves = pk.at<uint32_t>(at[q].mv);
                G.s.nv = tp.n_vars; G.s.ne = tp.n_expr; G.s.nf = tp.n_free; G.s.mult = (uint32_t)g.sets.size();
                d->groups.push_back(G);
                q++;
            }
            d->group_off.push_back((uint32_t)d->groups.size());
        }
        d->ready = true;
    }
    // per variant: the raw rows, its scale, vars_out, the resident rows, a report per set, and the plans' rows
    uint64_t mult = 1;
    const uint64_t bytes = sizeof(double) * (3ull * L.n_vars + L.n_constraints + n_expr + 1) + sizeof(fk_report) * (uint64_t)n_sets +
                           plan_bytes(b.st, &mult);
    *chunk = system_batch_chunk(n, bytes, mult, std::max({L.n_vars, L.n_constraints, n_expr, n_sets}));
    if (d->chunk >= *chunk && d->plans.size() == ns) return FK_OK;
    int rc = d->grow_chunk(L, b.st, std::max(*chunk, d->chunk), true, n_sets, true);
    if (rc == FK_OK) rc = d->d_groups.reserve(d->groups.size());
    if (rc != FK_OK) {
        d->plans.clear();
        d->chunk = 0;
        return rc;
    }
    d->desc[0].vars = d->d_vt;
    d->desc[0].params = d->d_pt;
    for (size_t q = 0, w = 0; w < b.waves.size(); w++)
        for (const SystemSpBatch::Group& g : b.waves[w]) {
            const fk_batch_plan* p = d->plans[g.structure].get();
            SpGroup& G = d->groups[q++];
            G.s.vars = p->d_vars; G.s.params = p->d_params; G.s.out = p->d_out; G.s.reps = p->d_rep;
        }
    CU(cudaMemcpyAsync(d->d_desc, d->desc.data(), sizeof(SbStructure), cudaMemcpyHostToDevice, d->stream));
    if (!d->groups.empty())
        CU(cudaMemcpyAsync(d->d_groups, d->groups.data(), sizeof(SpGroup) * d->groups.size(), cudaMemcpyHostToDevice, d->stream));
    CU(cudaStreamSynchronize(d->stream));  // (the descriptors may change before a later call's copy)
    return FK_OK;
}

// Variants [lo, hi) on one device: per chunk the prepare kernel (scale, the perturbations that precede every set, the resident rows
// vt / pt); per wave one gather / scatter launch and one LM launch per structure present; a last gather / scatter launch with the
// write-back.
static int system_sp_range(SystemSpBatch& b, const SystemBatchCall& c, int device, uint32_t lo, uint32_t hi) {
    const SystemBatchLayout& L = b.L;
    const uint32_t n_expr = (uint32_t)L.kind.size(), nw = L.n_waves, n_sets = (uint32_t)L.comps.size();
    const uint32_t n_rep = c.reports ? std::min(c.reports_per_variant, n_sets) : 0;
    SystemSpDevice* d = device_slot(b.mu, b.devices, device);
    std::lock_guard<std::mutex> lock(d->mu);
    uint32_t chunk = 0;
    const int rc = system_sp_device(b, d, device, hi - lo, &chunk);
    if (rc != FK_OK) return rc;
    return solve_chunks(d, L, c, lo, hi, chunk, n_rep, 1, "fk_system_batch_solve_single_pass / _recursive_assembly kernels / copies",
                        [&](uint32_t cnt, const double* raw, uint32_t raw_stride) -> int {
                            for (uint32_t w = 0; w <= nw; w++) {
                                const uint32_t s_lo = w ? d->group_off[w - 1] : 0, s_hi = w ? d->group_off[w] : 0;
                                const uint32_t g_lo = w < nw ? d->group_off[w] : 0, g_hi = w < nw ? d->group_off[w + 1] : 0;
                                const uint32_t p_lo = c.perturb && w < nw ? d->pert_off[w] : 0, p_hi = c.perturb && w < nw ? d->pert_off[w + 1] : 0;
                                const int e = launch_system_sp_gather_scatter(
                                    cnt, L.n_vars, n_expr, d->d_vt, d->d_pt, s_hi - s_lo, d->d_groups + s_lo, n_rep, d->d_rep_out, p_hi - p_lo,
                                    d->d_pvar + p_lo, d->d_pdraw + p_lo, d->d_draws, g_hi - g_lo, d->d_groups + g_lo, d->d_solved, raw, raw_stride,
                                    d->d_scales, w == nw ? d->d_vars_out.get() : nullptr, d->stream);
                                if (e != 0) return cuda_fail((cudaError_t)e, "launch fk_system_sp_gather_scatter_kernel");
                                if (w == nw) break;
                                for (const SystemSpBatch::Group& g : b.waves[w]) {  // LM under SinglePass / RecursiveAssembly whatever the optimizer (assemble/mod.rs:191, :224)
                                    fk_batch_plan* p = d->plans[g.structure].get();
                                    p->n = cnt * (uint32_t)g.sets.size();
                                    const int r = fk_batch_plan_run(p, d->stream);
                                    if (r != FK_OK) return r;
                                }
                            }
                            return FK_OK;
                        });
}

int system_sp_batch_solve(SystemSpBatch& b, const SystemBatchCall& c) {
    for (const SystemSpBatch::Structure& S : b.st)  // sets / steps on the global sparse path: the front limit of fk_batch_solve
        if (S.topo->t.path == 2 && S.topo->sb_check() != FK_OK) {
            const uint32_t k = S.members[0];
            const std::string what = b.L.step_constraint.empty()
                                         ? "set " + std::to_string(k) + " (first expression " + std::to_string(b.L.comps[k].expr[0])
                                         : "step " + std::to_string(k) + " (first constraint " + std::to_string(b.L.step_constraint[k]);
            return fail(FK_ERR_TOO_LARGE, what + "): " + S.topo->sb_err + "; fk_system_solve_opts solves it one variant at a time");
        }
    if (c.n == 0) return FK_OK;
    int n_gpus = c.n_gpus;
    const int rc = clamp_gpus(n_gpus);
    if (rc != FK_OK) return rc;
    return shard_over_devices(n_gpus, c.n, [&](int device, uint32_t lo, uint32_t hi) { return system_sp_range(b, c, device, lo, hi); });
}

// ---- fk_system_batch_analyze / fk_system_batch_residuals: System::analyze and calculate_residual over n variants -----------
// Per device: the layout's tables, the template rows, the chunk buffers (variables vt and expanded parameters pt are what the
// analyze kernels and fk_system_residuals_kernel read), the outputs of each operation (grown on its first call) and the analyze
// workspace.
struct SystemAnDevice : SystemDevice {
    const uint8_t* d_kind = nullptr;
    const uint32_t *d_slot = nullptr, *d_expr_con = nullptr, *d_con_off = nullptr;
    GrowBuf<double> d_res;
    GrowBuf<uint8_t> d_indep, d_dep;
    GrowBuf<double> d_ws;
};

struct SystemAnBatch {
    SystemAnLayout L;
    uint32_t n_expr = 0, n_constraints = 0;
    uint64_t sig = 0;  // hash of the structure (n_vars, kinds, slot table, constraint ranges): fk_systems_analyze merges by it
    std::mutex mu;
    std::map<int, std::unique_ptr<SystemAnDevice>> devices;
};

int system_an_batch_create(SystemAnLayout&& layout, std::shared_ptr<SystemAnBatch>* out) {
    std::shared_ptr<SystemAnBatch> b = std::make_shared<SystemAnBatch>();
    b->L = std::move(layout);
    b->n_expr = (uint32_t)b->L.kind.size();
    b->n_constraints = b->L.con_off.empty() ? 0 : (uint32_t)b->L.con_off.size() - 1;
    uint64_t h = 1469598103934665603ull;  // FNV-1a
    auto mix = [&h](const void* p, size_t bytes) {
        for (size_t i = 0; i < bytes; i++) h = (h ^ ((const unsigned char*)p)[i]) * 1099511628211ull;
    };
    mix(&b->L.n_vars, sizeof(uint32_t));
    mix(b->L.kind.data(), b->L.kind.size());
    mix(b->L.slot_var.data(), sizeof(uint32_t) * b->L.slot_var.size());
    mix(b->L.con_off.data(), sizeof(uint32_t) * b->L.con_off.size());
    b->sig = h;
    *out = std::move(b);
    return FK_OK;
}

// Tables once per device; the input buffers and the outputs of the call's operation (analyze: per-expression flags and
// per-constraint counts; residuals: per-constraint values) grow with the chunk.  *chunk: the variants per chunk for n variants.
// The caller holds d->mu.
static int system_an_device(const SystemAnBatch& b, SystemAnDevice* d, int device, uint32_t n, bool analyze, uint32_t* chunk) {
    CU(cudaSetDevice(device));
    const SystemAnLayout& L = b.L;
    const uint32_t ne = b.n_expr, ncon = b.n_constraints;
    if (!d->ready) {
        TablePack pk;
        const size_t o_kind = pk.add(L.kind), o_slot = pk.add(L.slot_var), o_con = pk.add(L.expr_constraint), o_off = pk.add(L.con_off);
        const int rc = d->upload_tables(device, pk, L.n_vars, ne);
        if (rc != FK_OK) return rc;
        d->d_kind = pk.at<uint8_t>(o_kind);
        d->d_slot = pk.at<uint32_t>(o_slot);
        d->d_expr_con = pk.at<uint32_t>(o_con);
        d->d_con_off = pk.at<uint32_t>(o_off);
        d->ready = true;
    }
    // per variant: the raw parameters, vt and pt, and the operation's outputs
    const uint64_t bytes = sizeof(double) * ((uint64_t)L.n_vars + ncon + ne) + (analyze ? (uint64_t)ne + ncon : sizeof(double) * ncon);
    *chunk = system_batch_chunk(n, bytes, 1, std::max({L.n_vars, ncon, ne}));
    const size_t cap = *chunk;
    int rc = d->d_raw_param.reserve(cap * ncon);
    if (rc == FK_OK) rc = d->d_vt.reserve(cap * L.n_vars);
    if (rc == FK_OK) rc = d->d_pt.reserve(cap * ne);
    if (rc == FK_OK && analyze) rc = d->d_indep.reserve(cap * ne);
    if (rc == FK_OK && analyze) rc = d->d_dep.reserve(cap * ncon);
    if (rc == FK_OK && !analyze) rc = d->d_res.reserve(cap * ncon);
    return rc;
}

// Variants [lo, hi) on one device, per chunk: upload (or broadcast the template), expand the parameters, then analyze + reduce or
// the residuals, download.
static int system_an_range(SystemAnBatch& b, const SystemAnCall& c, int device, uint32_t lo, uint32_t hi) {
    const SystemAnLayout& L = b.L;
    const uint32_t ne = b.n_expr, ncon = b.n_constraints;
    const bool analyze = c.dependent != nullptr;
    SystemAnDevice* d = device_slot(b.mu, b.devices, device);
    std::lock_guard<std::mutex> lock(d->mu);
    uint32_t chunk = 0;
    const int rc = system_an_device(b, d, device, hi - lo, analyze, &chunk);
    if (rc != FK_OK) return rc;
    const cudaStream_t st = d->stream;
    return run_chunks(d, L.n_vars, ne, c.tmpl_vars, c.tmpl_param, lo, hi, chunk, "fk_system_batch_analyze / _residuals kernels / copies",
                      [&](uint32_t at, uint32_t cnt) -> int {
        if (c.vars)
            CU(cudaMemcpyAsync(d->d_vt, c.vars + (size_t)at * L.n_vars, sizeof(double) * (size_t)cnt * L.n_vars, cudaMemcpyHostToDevice, st));
        if (c.params)
            CU(cudaMemcpyAsync(d->d_raw_param, c.params + (size_t)at * ncon, sizeof(double) * (size_t)cnt * ncon, cudaMemcpyHostToDevice, st));
        int e = launch_system_an_expand(cnt, L.n_vars, ne, ncon, c.vars ? nullptr : d->d_tmpl_vars, d->d_vt, d->d_expr_con,
                                        c.params ? d->d_raw_param.get() : nullptr, d->d_tmpl_param, d->d_pt, st);
        if (e != 0) return cuda_fail((cudaError_t)e, "launch fk_system_an_expand_kernel");
        if (!analyze) {
            e = launch_system_residuals(cnt, L.n_vars, ne, ncon, d->d_kind, d->d_slot, d->d_con_off, d->d_vt, d->d_pt, d->d_res, st);
            if (e != 0) return cuda_fail((cudaError_t)e, "launch fk_system_residuals_kernel");
            CU(cudaMemcpyAsync(c.residuals + (size_t)at * ncon, d->d_res, sizeof(double) * (size_t)cnt * ncon, cudaMemcpyDeviceToHost, st));
            return FK_OK;
        }
        const int rc = analyze_launch(L.n_vars, ne, d->d_kind, d->d_slot, cnt, d->d_vt, d->d_pt, d->d_indep, device, d->d_ws, st);
        if (rc != FK_OK) return rc;
        e = launch_system_an_reduce(cnt, ne, ncon, d->d_indep, d->d_con_off, d->d_dep, st);
        if (e != 0) return cuda_fail((cudaError_t)e, "launch fk_system_an_reduce_kernel");
        CU(cudaMemcpyAsync(c.dependent + (size_t)at * ncon, d->d_dep, (size_t)cnt * ncon, cudaMemcpyDeviceToHost, st));
        return FK_OK;
    });
}

int system_an_batch_run(SystemAnBatch& b, const SystemAnCall& c) {
    if (c.n == 0 || b.n_constraints == 0) return FK_OK;
    int n_gpus = c.n_gpus;
    int rc = clamp_gpus(n_gpus);
    if (rc != FK_OK) return rc;
    if (c.dependent) {  // the size limit of the analyze kernels (it depends on neither the batch size nor the device: the current one)
        int device = 0;
        if (cudaGetDevice(&device) != cudaSuccess) device = 0;
        AnalyzePlan plan;
        std::string err;
        rc = choose_analyze(b.L.n_vars, b.n_expr, c.n, device, &plan, &err);
        if (rc != FK_OK) return fail(rc, err);
    }
    return shard_over_devices(n_gpus, c.n, [&](int device, uint32_t lo, uint32_t hi) { return system_an_range(b, c, device, lo, hi); });
}

// ---- fk_systems_solve: System::solve over n different drawings ------------------------------------------------------------
// The call's plan: the structures of every drawing's SystemBatch merged across drawings (same structural signature and an
// exact comparison -- not the topology pointer, which differs with the topology cache off or after an eviction), each with
// its launch kind, and the instances (solved components) in drawing order, component order inside a drawing.  Built per call.
struct SystemsPlan {
    struct Structure {
        std::shared_ptr<fk_topology> topo;
        uint32_t kind = 1;                           // 0 heterogeneous launch, 1 uniform batch, 2 sparse batch kernel (LM, path 2)
        uint32_t instances = 0;
        uint32_t hetero = kSbNone;                   // kind 0: its program in the heterogeneous launch
        uint32_t first_drawing = 0, first_comp = 0;  // where it first appears (named by refusals)
    };
    std::vector<Structure> st;
    std::vector<uint32_t> inst_struct;           // per instance
    std::vector<size_t> inst_off;                // [n + 1] first instance of each drawing
    std::vector<size_t> var_off;                 // [n + 1] first variable of each drawing in the call's flat rows
    std::vector<fk_topology*> topos32;           // the 32-lane topologies of the kind-0 structures
    const std::vector<double>* draws = nullptr;  // the longest of the drawings' draws: each drawing's are a prefix (LCG seeded 42)
};

static void systems_plan_create(const std::vector<SystemsDrawing>& d, int optimizer, SystemsPlan& P) {
    static const std::vector<double> no_draws;
    P.draws = &no_draws;
    P.inst_off.assign(1, 0);
    P.var_off.assign(1, 0);
    std::multimap<uint64_t, uint32_t> by_sig;
    std::unordered_map<const fk_topology*, uint32_t> by_topo;  // (one topology is one structure: skips the signature)
    for (uint32_t i = 0; i < d.size(); i++) {
        const SystemBatch& b = *d[i].plan;
        std::vector<uint32_t> merged(b.st.size());
        for (uint32_t s = 0; s < b.st.size(); s++) {
            const auto known = by_topo.find(b.st[s].topo.get());
            if (known != by_topo.end()) {
                merged[s] = known->second;
                P.st[known->second].instances += b.st[s].mult;
                continue;
            }
            const fk_problem p = structure_of(b.st[s].topo->t);
            const uint64_t sig = structural_signature(p);
            uint32_t m = kSbNone;
            for (auto r = by_sig.equal_range(sig); r.first != r.second && m == kSbNone; ++r.first)
                if (same_structure(structure_of(P.st[r.first->second].topo->t), p)) m = r.first->second;
            by_topo.emplace(b.st[s].topo.get(), m == kSbNone ? (uint32_t)P.st.size() : m);
            if (m == kSbNone) {
                m = (uint32_t)P.st.size();
                by_sig.emplace(sig, m);
                SystemsPlan::Structure S;
                S.topo = b.st[s].topo;
                S.first_drawing = i;
                S.first_comp = b.st[s].members[0];
                P.st.push_back(std::move(S));
            }
            merged[s] = m;
            P.st[m].instances += b.st[s].mult;
        }
        for (uint32_t k = 0; k < b.L.comps.size(); k++) P.inst_struct.push_back(merged[b.comp_struct[k]]);
        P.inst_off.push_back(P.inst_struct.size());
        P.var_off.push_back(P.var_off.back() + b.L.n_vars);
        if (b.L.draws.size() > P.draws->size()) P.draws = &b.L.draws;
    }
    // fk_lm_solve_batch's rule; L-BFGS has no heterogeneous kernel, so every structure gets its own launch
    for (SystemsPlan::Structure& S : P.st) {
        const fk::Topology& t = S.topo->t;
        S.kind = optimizer == 0 && t.path == 2 ? 2 : 1;
        fk_topology* t32 = optimizer == 0 ? hetero_topology(S.topo.get(), S.instances) : nullptr;
        if (!t32) continue;
        S.kind = 0;
        S.hetero = (uint32_t)P.topos32.size();
        P.topos32.push_back(t32);
    }
}

void systems_layout(const std::vector<SystemsDrawing>& d, int optimizer, uint32_t* n_components, std::vector<uint32_t>* instances,
                    std::vector<uint32_t>* launch_kind) {
    SystemsPlan P;
    systems_plan_create(d, optimizer, P);
    *n_components = (uint32_t)P.inst_struct.size();
    instances->clear();
    launch_kind->clear();
    for (const SystemsPlan::Structure& S : P.st) {
        instances->push_back(S.instances);
        launch_kind->push_back(S.kind);
    }
}

// Per device, reused across calls (never destroyed: CUDA may be gone at static-destruction time): one stream, a grow-only
// pinned staging block and device arena, and the grow-only workspaces of the solve kernels and of the global-memory analyze
// kernels (launches on the one stream run one after the other, so one workspace serves them all).  fk_systems_solve,
// fk_systems_analyze and fk_systems_residuals share it.
struct SystemsDevice {
    std::mutex mu;
    cudaStream_t stream = nullptr;
    GrowBuf<unsigned char> h{true}, d;
    SolveWorkspace ws;
    GrowBuf<double> an_ws;
};
static SystemsDevice* systems_device_for(int device) {
    static std::mutex m;
    static std::map<int, SystemsDevice*> devs;
    std::lock_guard<std::mutex> lock(m);
    SystemsDevice*& p = devs[device];
    if (!p) p = new SystemsDevice();
    return p;
}

// Drawings [lo, hi) of a many-drawing call on one device, chunk after chunk on its SystemsDevice's stream.  The cut: drawings in
// order, at least one per chunk, closed at about 1 GiB of bytes(a, b) -- the device bytes drawing b adds to a chunk that starts at
// drawing a --, at FK_SYSTEM_BATCH_CHUNK drawings and, given inst_off (the instances before each drawing), at INT32_MAX instances,
// so that every launch stays within INT32_MAX sketches.  layout(c) places the rows of chunk c (c.a, c.b set): the pinned staging
// block takes its first c.o_work bytes and the device arena its c.end bytes, both reserved for the largest chunk.  Then
// prepare(D, chunks) once and body(D, c) for every chunk; after a failure the stream is synchronised, so that nothing of the failed
// chunk still runs when the staging is reused.
template <class Chunk, class Bytes, class Layout, class Prepare, class Body>
static int run_drawing_chunks(int device, uint32_t lo, uint32_t hi, const size_t* inst_off, const Bytes& bytes, const Layout& layout,
                              const Prepare& prepare, const Body& body) {
    CU(cudaSetDevice(device));
    SystemsDevice* D = systems_device_for(device);
    std::lock_guard<std::mutex> lock(D->mu);
    if (!D->stream) CU(cudaStreamCreateWithFlags(&D->stream, cudaStreamNonBlocking));
    std::vector<Chunk> chunks;
    size_t h_need = 0, d_need = 0;
    const uint32_t cap = system_batch_chunk_env();
    for (uint32_t a = lo; a < hi;) {
        uint32_t b = a;
        uint64_t total = 0;
        while (b < hi) {
            const uint64_t db = bytes(a, b);
            if (b > a && (total + db > (1ull << 30) || (cap && b - a >= cap) || (inst_off && inst_off[b + 1] - inst_off[a] > (uint64_t)INT32_MAX)))
                break;
            total += db;
            b++;
        }
        chunks.emplace_back();
        Chunk& c = chunks.back();
        c.a = a;
        c.b = b;
        layout(c);
        h_need = std::max(h_need, c.o_work);
        d_need = std::max(d_need, c.end);
        a = b;
    }
    int rc = D->h.reserve(h_need, h_need + h_need / 4);
    if (rc == FK_OK) rc = D->d.reserve(d_need, d_need + d_need / 4);
    if (rc == FK_OK) rc = prepare(*D, chunks);
    for (size_t k = 0; k < chunks.size() && rc == FK_OK; k++)
        if ((rc = body(*D, chunks[k])) != FK_OK) cudaStreamSynchronize(D->stream);
    return rc;
}

// One chunk of drawings [a, b) on one device and where its rows live in the arena: [0, o_output) the input the host stages in
// pinned memory (same offsets) and sends with one copy, [o_output, o_work) the rows that come back with one copy, [o_work, end)
// device only.
struct SystemsChunk {
    uint32_t a = 0, b = 0;
    size_t i0 = 0, i1 = 0;       // its instances
    std::vector<uint32_t> count;  // per structure: instances in the chunk
    struct Rows { size_t vars = 0, params = 0, out = 0, reps = 0; };
    std::vector<Rows> rows;       // per uniform / sparse structure present: its batch rows
    size_t nj = 0, tab_words = 0, nvars = 0, nexpr = 0, hin = 0, hout = 0;
    size_t o_draws = 0, o_progs = 0, o_jobs = 0, o_inst = 0, o_ioff = 0, o_voff = 0, o_eoff = 0, o_tabs = 0, o_rawv = 0, o_rawp = 0,
           o_kinds = 0, o_output = 0, o_outv = 0, o_outr = 0, o_work = 0, o_scales = 0, o_hin = 0, o_hout = 0, o_hrep = 0, end = 0;
};

static void systems_chunk_layout(const std::vector<SystemsDrawing>& d, const SystemsPlan& P, SystemsChunk& c) {
    const size_t ns = P.st.size(), n = c.b - c.a;
    c.i0 = P.inst_off[c.a];
    c.i1 = P.inst_off[c.b];
    c.count.assign(ns, 0);
    for (uint32_t i = c.a; i < c.b; i++) {
        const SystemBatchLayout& L = d[i].plan->L;
        c.nvars += L.n_vars;
        c.nexpr += L.kind.size();
        for (size_t g = P.inst_off[i]; g < P.inst_off[i + 1]; g++) {
            const SystemsPlan::Structure& S = P.st[P.inst_struct[g]];
            const fk::Topology& t = S.topo->t;
            c.count[P.inst_struct[g]]++;
            c.tab_words += 2 * (size_t)t.n_vars + t.n_expr + t.n_free;
            if (S.kind == 0) {
                c.nj++;
                c.hin += (size_t)t.n_vars + t.n_expr;
                c.hout += t.n_free;
            }
        }
    }
    BlockLayout blk;
    const size_t ni = c.i1 - c.i0;
    c.o_draws = blk.put(sizeof(double) * P.draws->size());
    c.o_progs = blk.put(sizeof(fk::DevProgram) * P.topos32.size());
    c.o_jobs = blk.put(sizeof(fk::HeteroJob) * c.nj);
    c.o_inst = blk.put(sizeof(SysInst) * ni);
    c.o_ioff = blk.put(sizeof(uint32_t) * (n + 1));
    c.o_voff = blk.put(sizeof(uint64_t) * (n + 1));
    c.o_eoff = blk.put(sizeof(uint64_t) * (n + 1));
    c.o_tabs = blk.put(sizeof(uint32_t) * c.tab_words);
    c.o_rawv = blk.put(sizeof(double) * c.nvars);
    c.o_rawp = blk.put(sizeof(double) * c.nexpr);
    c.o_kinds = blk.put(c.nexpr);
    c.o_output = blk.end;
    c.o_outv = blk.put(sizeof(double) * c.nvars);
    c.o_outr = blk.put(sizeof(fk_report) * ni);
    c.o_work = blk.end;
    c.o_scales = blk.put(sizeof(double) * n);
    c.o_hin = blk.put(sizeof(double) * c.hin);
    c.o_hout = blk.put(sizeof(double) * c.hout);
    c.o_hrep = blk.put(sizeof(fk_report) * c.nj);
    c.rows.assign(ns, SystemsChunk::Rows{});
    for (size_t s = 0; s < ns; s++) {
        if (P.st[s].kind == 0 || c.count[s] == 0) continue;
        const fk::Topology& t = P.st[s].topo->t;
        SystemsChunk::Rows& r = c.rows[s];
        r.vars = blk.put(sizeof(double) * c.count[s] * t.n_vars);
        r.params = blk.put(sizeof(double) * c.count[s] * t.n_expr);
        r.out = blk.put(sizeof(double) * c.count[s] * t.n_free);
        r.reps = blk.put(sizeof(fk_report) * c.count[s]);
    }
    c.end = blk.end;
}

// Device bytes one drawing adds to a chunk (the budget of system_batch_chunk: about 1 GiB per chunk).
static uint64_t systems_drawing_bytes(const std::vector<SystemsDrawing>& d, const SystemsPlan& P, uint32_t i) {
    const SystemBatchLayout& L = d[i].plan->L;
    uint64_t bytes = sizeof(double) * (2ull * L.n_vars + L.kind.size() + 1) + L.kind.size() + 20;
    for (size_t g = P.inst_off[i]; g < P.inst_off[i + 1]; g++) {
        const fk::Topology& t = P.st[P.inst_struct[g]].topo->t;
        bytes += sizeof(SysInst) + sizeof(fk::HeteroJob) + 2 * sizeof(fk_report) + sizeof(uint32_t) * (2ull * t.n_vars + t.n_expr + t.n_free) +
                 sizeof(double) * ((uint64_t)t.n_vars + t.n_expr + t.n_free);
    }
    return bytes;
}

// Drawings [lo, hi) on one device, chunk after chunk on its stream: stage and upload, fk_systems_prepare_kernel, one
// heterogeneous launch, one launch per uniform or sparse structure, fk_systems_scatter_kernel, download; then the chunk's
// variables and reports into the call's rows (vars_out, reports).
static int systems_range(const std::vector<SystemsDrawing>& d, const SystemsPlan& P, int optimizer, int perturb, int device, uint32_t lo,
                         uint32_t hi, double* vars_out, fk_report* reports) {
    const size_t ns = P.st.size();
    std::vector<const DeviceProgram*> full(ns, nullptr);
    std::vector<fk::DevProgram> progs;
    uint32_t max_state = 1;
    // the programs of the structures present, the workspaces of their largest launch, the programs of the heterogeneous launch
    auto prepare = [&](SystemsDevice& D, const std::vector<SystemsChunk>& chunks) -> int {
        std::vector<uint32_t> max_count(ns, 0);
        for (const SystemsChunk& c : chunks)
            for (size_t s = 0; s < ns; s++) max_count[s] = std::max(max_count[s], c.count[s]);
        for (size_t s = 0; s < ns; s++) {
            if (P.st[s].kind == 0 || max_count[s] == 0) continue;
            const fk::DevProgram* v = nullptr;
            int rc = P.st[s].topo->program_for(device, &v, &full[s], optimizer == 0);
            if (rc == FK_OK) rc = D.ws.reserve(*full[s], solve_kernel(P.st[s].topo.get(), optimizer, max_count[s]), max_count[s]);
            if (rc != FK_OK) return rc;
        }
        return P.topos32.empty() ? FK_OK : hetero_programs(device, P.topos32, progs, &max_state);
    };
    auto run = [&](SystemsDevice& D, const SystemsChunk& c) -> int {
        const cudaStream_t st = D.stream;
        unsigned char* H = D.h;
        unsigned char* G = D.d;
        const uint32_t n = c.b - c.a;
        if (!P.draws->empty()) std::memcpy(H + c.o_draws, P.draws->data(), sizeof(double) * P.draws->size());
        if (!progs.empty()) std::memcpy(H + c.o_progs, progs.data(), sizeof(fk::DevProgram) * progs.size());
        fk::HeteroJob* jobs = (fk::HeteroJob*)(H + c.o_jobs);
        SysInst* inst = (SysInst*)(H + c.o_inst);
        uint32_t* ioff = (uint32_t*)(H + c.o_ioff);
        uint64_t* voff = (uint64_t*)(H + c.o_voff);
        uint64_t* eoff = (uint64_t*)(H + c.o_eoff);
        uint32_t* tabs = (uint32_t*)(H + c.o_tabs);
        double* rawv = (double*)(H + c.o_rawv);
        double* rawp = (double*)(H + c.o_rawp);
        uint8_t* kinds = (uint8_t*)(H + c.o_kinds);
        double* hin = (double*)(G + c.o_hin);
        double* hout = (double*)(G + c.o_hout);
        fk_report* hrep = (fk_report*)(G + c.o_hrep);
        std::vector<uint32_t> rank(ns, 0);
        size_t j = 0, tw = 0, jin = 0, jout = 0, vo = 0, eo = 0;
        for (uint32_t i = c.a; i < c.b; i++) {
            const SystemBatchLayout& L = d[i].plan->L;
            const uint32_t di = i - c.a, ne = (uint32_t)L.kind.size();
            ioff[di] = (uint32_t)(P.inst_off[i] - c.i0);
            voff[di] = vo;
            eoff[di] = eo;
            if (L.n_vars) std::memcpy(rawv + vo, d[i].vars, sizeof(double) * L.n_vars);
            if (ne) {
                std::memcpy(rawp + eo, d[i].param, sizeof(double) * ne);
                std::memcpy(kinds + eo, L.kind.data(), ne);
            }
            for (size_t k = 0; k < L.comps.size(); k++) {
                const size_t g = P.inst_off[i] + k;
                const uint32_t s = P.inst_struct[g];
                const SystemsPlan::Structure& S = P.st[s];
                const SystemBatchLayout::Component& comp = L.comps[k];
                const uint32_t nv = (uint32_t)comp.slot_var.size(), nx = (uint32_t)comp.expr.size(), nf = (uint32_t)comp.free_var.size();
                SysInst& I = inst[g - c.i0];
                I.tab = tw;
                I.drawing = di;
                I.nv = nv;
                I.ne = nx;
                I.nf = nf;
                for (const std::vector<uint32_t>* v : {&comp.slot_var, &comp.slot_draw, &comp.expr, &comp.free_var}) {
                    if (!v->empty()) std::memcpy(tabs + tw, v->data(), sizeof(uint32_t) * v->size());
                    tw += v->size();
                }
                if (S.kind == 0) {
                    fk::HeteroJob& J = jobs[j];
                    J.prog = S.hetero;
                    J.pad = 0;
                    J.vars_off = jin;
                    J.param_off = jin + nv;
                    J.out_off = jout;
                    I.vars = hin + jin;
                    I.params = hin + jin + nv;
                    I.out = hout + jout;
                    I.rep = hrep + j;
                    jin += (size_t)nv + nx;
                    jout += nf;
                    j++;
                } else {
                    const SystemsChunk::Rows& r = c.rows[s];
                    const size_t q = rank[s]++;
                    I.vars = (double*)(G + r.vars) + q * nv;
                    I.params = (double*)(G + r.params) + q * nx;
                    I.out = (const double*)(G + r.out) + q * nf;
                    I.rep = (const fk_report*)(G + r.reps) + q;
                }
            }
            vo += L.n_vars;
            eo += ne;
        }
        ioff[n] = (uint32_t)(c.i1 - c.i0);
        voff[n] = vo;
        eoff[n] = eo;
        CU(cudaMemcpyAsync(G, H, c.o_output, cudaMemcpyHostToDevice, st));
        const uint64_t* d_voff = (const uint64_t*)(G + c.o_voff);
        const uint32_t* d_ioff = (const uint32_t*)(G + c.o_ioff);
        const SysInst* d_inst = (const SysInst*)(G + c.o_inst);
        const uint32_t* d_tabs = (const uint32_t*)(G + c.o_tabs);
        const double* d_rawv = (const double*)(G + c.o_rawv);
        double* d_scales = (double*)(G + c.o_scales);
        int e = launch_systems_prepare(n, d_voff, (const uint64_t*)(G + c.o_eoff), d_ioff, (const uint8_t*)(G + c.o_kinds), d_rawv,
                                       (const double*)(G + c.o_rawp), (const double*)(G + c.o_draws), perturb, d_inst, d_tabs, d_scales, st);
        if (e != 0) return cuda_fail((cudaError_t)e, "launch fk_systems_prepare_kernel");
        if (c.nj) {
            const int rc = hetero_launch((const fk::DevProgram*)(G + c.o_progs), (const fk::HeteroJob*)(G + c.o_jobs), c.nj, max_state, hin, hout,
                                         hrep, st);
            if (rc != FK_OK) return rc;
        }
        for (size_t s = 0; s < ns; s++) {
            const uint32_t cnt = c.count[s];
            if (P.st[s].kind == 0 || cnt == 0) continue;
            const SystemsChunk::Rows& r = c.rows[s];
            const int rc = solve_launch(*full[s], solve_kernel(P.st[s].topo.get(), optimizer, cnt), cnt, (const double*)(G + r.vars),
                                        (const double*)(G + r.params), (double*)(G + r.out), (fk_report*)(G + r.reps), D.ws, st);
            if (rc != FK_OK) return rc;
        }
        e = launch_systems_scatter(n, d_voff, d_ioff, d_rawv, d_scales, d_inst, d_tabs, (double*)(G + c.o_outv), (fk_report*)(G + c.o_outr), st);
        if (e != 0) return cuda_fail((cudaError_t)e, "launch fk_systems_scatter_kernel");
        CU(cudaMemcpyAsync(H + c.o_output, G + c.o_output, c.o_work - c.o_output, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        if (c.nvars) std::memcpy(vars_out + P.var_off[c.a], H + c.o_outv, sizeof(double) * c.nvars);
        if (c.i1 > c.i0) std::memcpy(reports + c.i0, H + c.o_outr, sizeof(fk_report) * (c.i1 - c.i0));
        return FK_OK;
    };
    return run_drawing_chunks<SystemsChunk>(
        device, lo, hi, P.inst_off.data(), [&](uint32_t, uint32_t b) { return systems_drawing_bytes(d, P, b); },
        [&](SystemsChunk& c) { systems_chunk_layout(d, P, c); }, prepare, run);
}

int systems_solve(const std::vector<SystemsDrawing>& d, int optimizer, int perturb, int n_gpus, double* vars_out, fk_report* reports) {
    SystemsPlan P;
    systems_plan_create(d, optimizer, P);
    for (const SystemsPlan::Structure& S : P.st)  // LM on the global sparse path: the front limit of fk_batch_solve
        if (S.kind == 2 && S.topo->sb_check() != FK_OK)
            return fail(FK_ERR_TOO_LARGE, "drawing " + std::to_string(S.first_drawing) + ", component " + std::to_string(S.first_comp) + ": " +
                                              S.topo->sb_err + "; Optimizer::LBfgs takes systems of every size");
    if (d.empty()) return FK_OK;
    const int rc = clamp_gpus(n_gpus);
    if (rc != FK_OK) return rc;
    return shard_over_devices(n_gpus, (uint32_t)d.size(), [&](int device, uint32_t lo, uint32_t hi) {
        return systems_range(d, P, optimizer, perturb, device, lo, hi, vars_out, reports);
    });
}

// ---- fk_systems_analyze / fk_systems_residuals: System::analyze and calculate_residual over n different drawings -------------
// The call's plan: the drawings' SystemAnBatch plans merged into structures (one plan object is one structure; other plans join
// one when the signature and an exact comparison of n_vars, kinds, slot table and constraint ranges agree), each with its analyze
// launch kind, and every drawing's first constraint in the call's output.  Built per call.
struct SystemsAnPlan {
    struct Structure {
        const SystemAnBatch* b = nullptr;  // its first drawing's plan: the tables
        uint32_t kind = 0;                 // 0 heterogeneous warp launch, 1 one launch of the kernel choose_analyze picks
        uint32_t instances = 0, first_drawing = 0;
        size_t tab_words = 0;              // slot_var[8 n_expr], the kinds in whole words, con_off[n_constraints + 1]
    };
    std::vector<Structure> st;
    std::vector<uint32_t> drawing_struct;  // per drawing
    std::vector<size_t> con_off;           // [n + 1]
};

constexpr uint32_t kSystemsAnUniform = 64;  // instances from which a warp-sized structure gets a launch of its own

// analyze == false (the residuals): every structure kind 0, the rows in drawing order.
static void systems_an_plan_create(const std::vector<SystemsAnDrawing>& d, bool analyze, SystemsAnPlan& P) {
    const int forced = analyze ? forced_analyze_kernel() : -1;
    std::multimap<uint64_t, uint32_t> by_sig;
    std::unordered_map<const SystemAnBatch*, uint32_t> by_plan;
    P.con_off.assign(1, 0);
    for (uint32_t i = 0; i < d.size(); i++) {
        const SystemAnBatch* b = d[i].plan;
        uint32_t m = kSbNone;
        const auto known = by_plan.find(b);
        if (known != by_plan.end()) {
            m = known->second;
        } else {
            for (auto r = by_sig.equal_range(b->sig); r.first != r.second && m == kSbNone; ++r.first) {
                const SystemAnLayout& L = P.st[r.first->second].b->L;
                if (L.n_vars == b->L.n_vars && L.kind == b->L.kind && L.slot_var == b->L.slot_var && L.con_off == b->L.con_off) m = r.first->second;
            }
            if (m == kSbNone) {
                m = (uint32_t)P.st.size();
                by_sig.emplace(b->sig, m);
                SystemsAnPlan::Structure S;
                S.b = b;
                S.first_drawing = i;
                const bool warp = (forced < 0 || forced == kAnWarp) && batch_analyze_warp_fits(b->L.n_vars, b->n_expr);
                S.kind = analyze && !warp ? 1 : 0;  // (kind 0 may still become 1 below, by its instance count)
                S.tab_words = 8 * (size_t)b->n_expr + (b->n_expr + 3) / 4 + b->n_constraints + 1;
                P.st.push_back(S);
            }
            by_plan.emplace(b, m);
        }
        P.st[m].instances++;
        P.drawing_struct.push_back(m);
        P.con_off.push_back(P.con_off.back() + d[i].plan->n_constraints);
    }
    // A structure with many instances runs faster in its own fk_batch_analyze_kernel launch (choose_analyze's warp kernel): its
    // exact footprint rather than the class's power of two sets the warps per SM.  The cut is fk_lm_solve_batch's for its
    // heterogeneous launch.
    for (SystemsAnPlan::Structure& S : P.st)
        if (analyze && S.instances >= kSystemsAnUniform) S.kind = 1;
}

void systems_an_layout(const std::vector<SystemsAnDrawing>& d, std::vector<uint32_t>* instances, std::vector<uint32_t>* launch_kind) {
    SystemsAnPlan P;
    systems_an_plan_create(d, true, P);
    instances->clear();
    launch_kind->clear();
    for (const SystemsAnPlan::Structure& S : P.st) {
        instances->push_back(S.instances);
        launch_kind->push_back(S.kind);
    }
}

// One chunk of drawings [a, b) on one device.  Arena: [0, o_output) the input staged in pinned memory (same offsets) and sent with
// one copy -- per drawing its SysAnJob, the constraint offsets, the kind-0 jobs, the tables of the structures present, the
// variable and parameter rows --, [o_output, o_work) the counts or residuals that come back with one copy, [o_work, end) the
// flags.  Rows (and flags, at the parameter offsets): the kind-0 drawings in drawing order, then one block per kind-1 structure
// present, its drawings in drawing order, so that its uniform launch reads them in place.
struct SystemsAnChunk {
    uint32_t a = 0, b = 0;
    std::vector<uint32_t> count;                 // per structure: drawings in the chunk
    std::vector<size_t> tab, vblk, eblk;         // per structure present: table offset (words); kind 1: its block's row offsets
    size_t nj = 0, tab_words = 0, nvars = 0, nexpr = 0, ncon = 0;
    size_t o_desc = 0, o_base = 0, o_jobs = 0, o_tabs = 0, o_vars = 0, o_params = 0, o_output = 0, o_work = 0, end = 0;
};

static void systems_an_chunk_layout(const std::vector<SystemsAnDrawing>& d, const SystemsAnPlan& P, bool analyze, SystemsAnChunk& c) {
    const size_t ns = P.st.size(), n = c.b - c.a;
    c.count.assign(ns, 0);
    c.tab.assign(ns, 0);
    c.vblk.assign(ns, 0);
    c.eblk.assign(ns, 0);
    for (uint32_t i = c.a; i < c.b; i++) {
        const uint32_t s = P.drawing_struct[i];
        const SystemAnBatch& B = *d[i].plan;
        if (c.count[s]++ == 0) {
            c.tab[s] = c.tab_words;
            c.tab_words += P.st[s].tab_words;
        }
        if (P.st[s].kind == 0) {
            c.nvars += B.L.n_vars;
            c.nexpr += B.n_expr;
            if (B.n_expr) c.nj++;
        }
    }
    for (size_t s = 0; s < ns; s++) {
        if (P.st[s].kind == 0 || c.count[s] == 0) continue;
        c.vblk[s] = c.nvars;
        c.eblk[s] = c.nexpr;
        c.nvars += (size_t)c.count[s] * P.st[s].b->L.n_vars;
        c.nexpr += (size_t)c.count[s] * P.st[s].b->n_expr;
    }
    c.ncon = P.con_off[c.b] - P.con_off[c.a];
    BlockLayout blk;
    c.o_desc = blk.put(sizeof(SysAnJob) * n);
    c.o_base = blk.put(sizeof(uint64_t) * (n + 1));
    c.o_jobs = blk.put(sizeof(SysAnJob) * c.nj);
    c.o_tabs = blk.put(sizeof(uint32_t) * c.tab_words);
    c.o_vars = blk.put(sizeof(double) * c.nvars);
    c.o_params = blk.put(sizeof(double) * c.nexpr);
    c.o_output = blk.put(analyze ? c.ncon : sizeof(double) * c.ncon);
    c.o_work = blk.end;
    if (analyze) blk.put(c.nexpr);
    c.end = blk.end;
}

// The warp footprint class of a drawing: its batch_analyze_warp_bytes rounded up to a power of two, at most 200 KiB.  One
// heterogeneous launch per class, so that one large drawing does not set the shared memory (and the warps per CTA) of every
// small one.
static size_t an_footprint_class(uint32_t n_vars, uint32_t n_expr) {
    const size_t bytes = batch_analyze_warp_bytes(n_vars, n_expr);
    size_t c = 16;
    while (c < bytes) c <<= 1;
    return std::min<size_t>(c, 200 * 1024);
}

// Drawings [lo, hi) on one device, chunk after chunk on its stream: stage and upload; analyze: one heterogeneous launch per
// footprint class, one launch per kind-1 structure, fk_systems_an_reduce_kernel; residuals: fk_systems_residuals_kernel;
// download, then the chunk's counts or residuals into the call's output.
static int systems_an_range(const std::vector<SystemsAnDrawing>& d, const SystemsAnPlan& P, int device, uint32_t lo, uint32_t hi,
                            uint8_t* dependent, double* residuals) {
    const bool analyze = dependent != nullptr;
    const size_t ns = P.st.size();
    std::vector<uint32_t> seen(ns, kSbNone);  // the chunk that last counted a structure's tables
    auto bytes = [&](uint32_t a, uint32_t b) -> uint64_t {
        const uint32_t s = P.drawing_struct[b];
        const SystemAnBatch& B = *d[b].plan;
        uint64_t db = sizeof(double) * ((uint64_t)B.L.n_vars + B.n_expr) + B.n_expr + 2 * sizeof(SysAnJob) + sizeof(uint64_t) +
                      (analyze ? 1 : sizeof(double)) * (uint64_t)B.n_constraints;
        if (seen[s] != a) db += sizeof(uint32_t) * P.st[s].tab_words;
        seen[s] = a;  // (a drawing the cut leaves out starts the next chunk, which counts the tables again)
        return db;
    };
    auto run = [&](SystemsDevice& D, const SystemsAnChunk& c) -> int {
        const cudaStream_t st = D.stream;
        unsigned char* H = D.h;
        unsigned char* G = D.d;
        const uint32_t n = c.b - c.a;
        SysAnJob* desc = (SysAnJob*)(H + c.o_desc);
        uint64_t* base = (uint64_t*)(H + c.o_base);
        SysAnJob* jobs = (SysAnJob*)(H + c.o_jobs);
        uint32_t* tabs = (uint32_t*)(H + c.o_tabs);
        double* rv = (double*)(H + c.o_vars);
        double* rp = (double*)(H + c.o_params);
        for (size_t s = 0; s < ns; s++) {
            if (c.count[s] == 0) continue;
            const SystemAnBatch& B = *P.st[s].b;
            uint32_t* t = tabs + c.tab[s];
            std::memcpy(t, B.L.slot_var.data(), sizeof(uint32_t) * B.L.slot_var.size());
            std::memset(t + 8 * (size_t)B.n_expr, 0, sizeof(uint32_t) * ((B.n_expr + 3) / 4));
            if (B.n_expr) std::memcpy(t + 8 * (size_t)B.n_expr, B.L.kind.data(), B.n_expr);
            std::memcpy(t + 8 * (size_t)B.n_expr + (B.n_expr + 3) / 4, B.L.con_off.data(), sizeof(uint32_t) * B.L.con_off.size());
        }
        std::vector<uint32_t> rank(ns, 0);
        std::vector<std::pair<size_t, uint32_t>> cls;  // (footprint class, drawing in the chunk) of every job
        cls.reserve(c.nj);
        uint64_t v0 = 0, e0 = 0;
        for (uint32_t i = c.a; i < c.b; i++) {
            const uint32_t s = P.drawing_struct[i], di = i - c.a;
            const SystemAnBatch& B = *d[i].plan;
            SysAnJob& J = desc[di];
            J.tab = (uint32_t)c.tab[s];
            J.n_vars = B.L.n_vars;
            J.n_expr = B.n_expr;
            J.pad = 0;
            if (P.st[s].kind == 0) {
                J.vars = v0;
                J.exprs = e0;
                v0 += B.L.n_vars;
                e0 += B.n_expr;
                if (B.n_expr) cls.emplace_back(an_footprint_class(B.L.n_vars, B.n_expr), di);
            } else {
                const uint64_t q = rank[s]++;
                J.vars = c.vblk[s] + q * B.L.n_vars;
                J.exprs = c.eblk[s] + q * B.n_expr;
            }
            if (B.L.n_vars) std::memcpy(rv + J.vars, d[i].vars, sizeof(double) * B.L.n_vars);
            if (B.n_expr) std::memcpy(rp + J.exprs, d[i].param, sizeof(double) * B.n_expr);
            base[di] = P.con_off[i] - P.con_off[c.a];
        }
        base[n] = c.ncon;
        std::stable_sort(cls.begin(), cls.end(), [](const auto& x, const auto& y) { return x.first < y.first; });
        for (size_t k = 0; k < cls.size(); k++) jobs[k] = desc[cls[k].second];
        CU(cudaMemcpyAsync(G, H, c.o_output, cudaMemcpyHostToDevice, st));
        const SysAnJob* d_desc = (const SysAnJob*)(G + c.o_desc);
        const uint64_t* d_base = (const uint64_t*)(G + c.o_base);
        const uint32_t* d_tabs = (const uint32_t*)(G + c.o_tabs);
        const double* d_vars = (const double*)(G + c.o_vars);
        const double* d_params = (const double*)(G + c.o_params);
        int e;
        if (!analyze) {
            e = launch_systems_residuals(n, c.ncon, d_base, d_desc, d_tabs, d_vars, d_params, (double*)(G + c.o_output), st);
            if (e != 0) return cuda_fail((cudaError_t)e, "launch fk_systems_residuals_kernel");
        } else {
            uint8_t* d_flags = G + c.o_work;
            for (size_t k = 0; k < cls.size();) {  // one launch per footprint class
                size_t k1 = k;
                while (k1 < cls.size() && cls[k1].first == cls[k].first) k1++;
                e = launch_systems_analyze((const SysAnJob*)(G + c.o_jobs) + k, (uint32_t)(k1 - k), cls[k].first, d_tabs, d_vars, d_params, d_flags, st);
                if (e != 0) return cuda_fail((cudaError_t)e, "launch fk_systems_analyze_kernel");
                k = k1;
            }
            for (size_t s = 0; s < ns; s++) {
                if (P.st[s].kind == 0 || c.count[s] == 0) continue;
                const SystemAnBatch& B = *P.st[s].b;
                const uint32_t* slot = d_tabs + c.tab[s];
                const int rc = analyze_launch(B.L.n_vars, B.n_expr, sys_an_kinds(slot, B.n_expr), slot, c.count[s], d_vars + c.vblk[s],
                                              d_params + c.eblk[s], d_flags + c.eblk[s], device, D.an_ws, st);
                if (rc != FK_OK) return rc;
            }
            e = launch_systems_an_reduce(n, c.ncon, d_base, d_desc, d_tabs, d_flags, G + c.o_output, st);
            if (e != 0) return cuda_fail((cudaError_t)e, "launch fk_systems_an_reduce_kernel");
        }
        const size_t out_bytes = (analyze ? 1 : sizeof(double)) * c.ncon;
        if (out_bytes) CU(cudaMemcpyAsync(H + c.o_output, G + c.o_output, out_bytes, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        if (out_bytes) {
            if (analyze) std::memcpy(dependent + P.con_off[c.a], H + c.o_output, out_bytes);
            else std::memcpy(residuals + P.con_off[c.a], H + c.o_output, out_bytes);
        }
        return FK_OK;
    };
    return run_drawing_chunks<SystemsAnChunk>(
        device, lo, hi, nullptr, bytes, [&](SystemsAnChunk& c) { systems_an_chunk_layout(d, P, analyze, c); },
        [](SystemsDevice&, const std::vector<SystemsAnChunk>&) { return FK_OK; }, run);
}

int systems_an_run(const std::vector<SystemsAnDrawing>& d, uint8_t* dependent, double* residuals, int n_gpus) {
    SystemsAnPlan P;
    systems_an_plan_create(d, dependent != nullptr, P);
    for (const SystemsAnPlan::Structure& S : P.st) {  // the size limit of the analyze kernels (the kernel itself is chosen per chunk)
        if (S.kind == 0) continue;
        int device = 0;
        if (cudaGetDevice(&device) != cudaSuccess) device = 0;
        AnalyzePlan plan;
        std::string err;
        const int rc = choose_analyze(S.b->L.n_vars, S.b->n_expr, S.instances, device, &plan, &err);
        if (rc != FK_OK) return fail(rc, "drawing " + std::to_string(S.first_drawing) + ": " + err);
    }
    if (P.con_off.back() == 0) return FK_OK;
    const int rc = clamp_gpus(n_gpus);
    if (rc != FK_OK) return rc;
    return shard_over_devices(n_gpus, (uint32_t)d.size(), [&](int device, uint32_t lo, uint32_t hi) {
        return systems_an_range(d, P, device, lo, hi, dependent, residuals);
    });
}

}  // namespace fk
