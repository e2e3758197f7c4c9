// Batched Levenberg–Marquardt kernels (K1, K2, K3, K4 of SURVEY §2): one tile of TILE lanes (a
// sub-warp, a warp, or a whole CTA) owns one sketch / connected component and runs the complete
// LM loop of fiksi/src/solve/lm.rs:21-193 on it out of shared memory.
#pragma once
#include <atomic>
#include <cstddef>
#include <cstdint>

#include "../../include/fiksi_b200.h"

namespace fk {

// Device view of a Topology's lane-padded op tables (Topology::Tables; all pointers device
// memory, shared by every sketch of the topology, read through the read-only path).
struct DevProgram {
    uint32_t n_vars, n_expr, n, m, jnnz, lnnz, tile;
    int32_t uniform_kind;
    uint32_t eval_rounds, a_nsteps, g_nsteps, f_nsteps, s_nsteps, b_nsteps;
    const uint32_t* free_vars;  // [n]
    const uint32_t* row_hdr;    // [eval_rounds*tile]
    const uint2* row_slots;     // [rows][8] {source, jpos}
    const uint32_t* a_flags;    // [a_nsteps+1]
    const uint32_t* a_ops;      // [(a_nsteps+1)*tile]
    const uint32_t* a_dst;
    const uint32_t* g_flags;
    const uint32_t* g_ops;
    const uint32_t* g_dst;
    const uint32_t* f_steps;    // [f_nsteps+1]
    const uint2* f_ops;
    const uint2* s_steps;       // [s_nsteps+1]
    const uint32_t* s_ops;
    const uint2* b_steps;       // [b_nsteps+1]
    const uint32_t* b_ops;
    // HOST pointer: parameter block of the sketch-per-thread kernel (lm_sketch.cuh), null when the topology
    // stays on the tile kernel.  launch_batch_lm picks between the two.
    const struct SkProgram* sketch_prog;
};

// Shared-memory doubles one sketch needs: x, xs, g (3n) + w / trial residuals (max(n, m)) + J
// (jnnz) + L / trial Jacobian (max(lnnz, jnnz)).
__host__ __device__ inline uint32_t lm_smem_doubles(uint32_t n, uint32_t m, uint32_t jnnz, uint32_t lnnz) {
    return 3u * n + (n > m ? n : m) + jnnz + (jnnz > lnnz ? jnnz : lnnz);
}

// Shared-memory doubles of one sketch in the L-BFGS kernel: x, xs, g, direction (4n) + s / y history
// (10n) + residuals (m) + Jacobian values (jnnz) + rho, alpha (10).
__host__ __device__ inline uint32_t lbfgs_smem_doubles(uint32_t n, uint32_t m, uint32_t jnnz) { return 14u * n + m + jnnz + 10u; }

// One system of a heterogeneous batch (fk_hetero_lm_kernel): its program and the offsets (in doubles) of its variable row,
// parameter row and output row in the call's device buffers.
struct HeteroJob {
    uint32_t prog, pad;
    uint64_t vars_off, param_off, out_off;
};
// d_progs: DevProgram views built for 32 lanes; max_state_doubles: largest lm_smem_doubles() over them.
int launch_hetero_lm(const DevProgram* d_progs, const HeteroJob* d_jobs, uint32_t n_jobs, uint32_t max_state_doubles, const double* d_in,
                     double* d_out, fk_report* d_reports, void* stream);

// Launchers (defined in lm_kernels.cu).  `stream` is a cudaStream_t.
int launch_batch_lm(const DevProgram& prog, uint32_t n_sketches, const double* vars, const double* params,
                    double* free_out, fk_report* reports, void* stream);
// Which kernel launch_batch_lm takes for a batch of this size: 1 sketch-per-thread, 0 tile kernel.
int batch_lm_uses_sketch_kernel(const DevProgram& prog, uint32_t n_sketches);
// -1 automatic (by batch size), 0 tile kernel, 1 sketch-per-thread kernel where the topology has one.
std::atomic<int>& lm_kernel_choice();
int launch_batch_eval(const DevProgram& prog, uint32_t n_sketches, const double* vars,
                      const double* params, double* out_r, double* out_j, int mode, void* stream);
// System::analyze on a batch, one warp per sketch: kinds[n_expr], slot_var[n_expr][8] device tables; out[n][n_expr].
// Returns cudaErrorInvalidConfiguration when one n_expr x n_vars matrix does not fit shared memory
// (batch_analyze_warp_fits: at most 200 KiB per warp with the column order and the flags).
size_t batch_analyze_warp_bytes(uint32_t n_vars, uint32_t n_expr);
bool batch_analyze_warp_fits(uint32_t n_vars, uint32_t n_expr);
int launch_batch_analyze(uint32_t n_vars, uint32_t n_expr, const uint8_t* kinds, const uint32_t* slot_var, uint32_t n_sketches,
                         const double* vars, const double* params, uint8_t* out, void* stream);
// fk_systems_analyze: one drawing of a call over many different drawings.  Its tables start at tabs + tab: slot_var[n_expr][8],
// the kinds (n_expr bytes, padded to whole words), con_off[n_constraints + 1] (the constraints' expression ranges).  vars: offset of
// its variable row; exprs: offset of its parameter row and of its flags (one per expression in both).
struct SysAnJob {
    uint64_t vars, exprs;
    uint32_t tab, n_vars, n_expr, pad;
};
__host__ __device__ inline const uint8_t* sys_an_kinds(const uint32_t* slot_var, uint32_t n_expr) {
    return reinterpret_cast<const uint8_t*>(slot_var + 8 * (size_t)n_expr);
}
__host__ __device__ inline const uint32_t* sys_an_con_off(const uint32_t* slot_var, uint32_t n_expr) {
    return slot_var + 8 * (size_t)n_expr + (n_expr + 3) / 4;
}
// The analyze warp kernel over n_jobs different drawings, jobs[j] one warp each: flags[J.exprs + r] = 1 iff row r increased the
// rank, as launch_batch_analyze's flags.  warp_bytes: every job's shared memory (at least its batch_analyze_warp_bytes, a
// multiple of 16, at most 200 KiB); warps per CTA as launch_batch_analyze takes them for that footprint.
int launch_systems_analyze(const SysAnJob* jobs, uint32_t n_jobs, size_t warp_bytes, const uint32_t* tabs, const double* vars,
                           const double* params, uint8_t* flags, void* stream);
// L-BFGS on a uniform batch (tile paths with 4 / 8 / 16 / 32 lanes only); d_jcolptr[n+1], d_jrow[jnnz]: CSC
// of the Jacobian.  Returns cudaErrorInvalidConfiguration when the topology does not take a tile path.
// batch_lbfgs_tile_fits: whether it takes a topology with these sizes and lanes (host only).
bool batch_lbfgs_tile_fits(uint32_t n, uint32_t m, uint32_t jnnz, uint32_t tile);
int launch_batch_lbfgs(const DevProgram& prog, const uint32_t* d_jcolptr, const uint32_t* d_jrow, uint32_t n_sketches, const double* vars,
                       const double* params, double* free_out, fk_report* reports, void* stream);
// SinglePass (fiksi/src/assemble/mod.rs:201-208): writes the solved free values of one set back into the
// resident variable rows so that later sets read them as fixed values.  vars[k][free_vars[f]] = free_out[k][f].
int launch_scatter_free(const uint32_t* d_free_vars, uint32_t n_free, uint32_t n_vars, uint32_t n_sketches, const double* free_out,
                        double* vars, void* stream);
// reports_out[k][st] = reports_in[st][k] (per-set report planes -> the caller's per-sketch rows).
int launch_transpose_reports(const fk_report* in, fk_report* out, uint32_t n_sketches, uint32_t steps, void* stream);
// assemble::solve's scale + seeded perturbation (fiksi/src/assemble/mod.rs:32-44,58-79,113-124) for n sketches:
// raw_vars[n][n_vars], raw_param [n][n_expr] (or one row when shared_param) -> vars, params (scaled), scales[n].
int launch_batch_prepare(uint32_t n_sketches, uint32_t n_vars, uint32_t n_expr, const uint8_t* kinds, int shared_param, uint32_t n_perturb,
                         const uint32_t* perturb_vars, const double* draws, const double* raw_vars, const double* raw_param, double* vars,
                         double* params, double* scales, void* stream);
// free_values[k][f] *= scales[k] (assemble/mod.rs:161-166).
int launch_batch_unscale(uint32_t n_sketches, uint32_t n_free, const double* scales, double* free_values, void* stream);
const char* lm_kernel_name();
// DFMA throughput microbenchmark on the current device (TFLOP/s, 2 flops per DFMA).
int measure_fp64_peak(double* tflops);

}  // namespace fk
