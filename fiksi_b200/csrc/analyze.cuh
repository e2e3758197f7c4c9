// System::analyze beyond shared memory (SURVEY 8f-2): the dense Jacobian of every expression over every variable and the
// reference's incremental Gauss-Jordan elimination (fiksi/src/analyze/numerical/mod.rs:33-147) with the matrix in global
// memory.  Three kernels serve fk_batch_analyze; choose_analyze picks one from the shape, the batch size and the device:
//   warp   one warp per sketch, the whole matrix in shared memory (fk_batch_analyze_kernel, lm_kernels.cu), wherever it fits;
//   cta    one CTA per sketch, a persistent grid over the batch (the batch fills the device);
//   group  G CTAs per sketch under a cooperative launch: the first CTA runs the per-row elimination chain, all G share the
//          Jordan update of the earlier rows, grid.sync() between the two phases of a row (single systems, small batches).
//
// Limit rule (enforced before any allocation): n_vars <= kAnMaxVars, so that the row being reduced fits shared memory, and
// one sketch's workspace -- min(n_expr, n_vars) rows of n_vars doubles (stride padded to 32), the column order and the
// flags -- within kAnWorkspaceBytes.  The 64x50 lattice (6,400 variables, 328 MB) is taken; BASELINE config 3 (200,000
// variables, 320 GB) is refused.
#pragma once
#include <cstdint>
#include <string>

namespace fk {

constexpr uint32_t kAnThreads = 256;
// Largest n_vars: the row being reduced is n_vars doubles of shared memory (208 KiB of the 227 KB a CTA may have).
constexpr uint32_t kAnMaxVars = 26624;
// Device memory of the workspaces of one (topology, device): a large sketch gets fewer concurrent CTAs, not tens of GiB.
// 4 GiB holds every resident CTA's matrix up to 24x20 lattices and 128 of 32x32's 33.5 MB matrices.
constexpr uint64_t kAnWorkspaceBytes = 4ull << 30;
constexpr uint64_t kAnHeadDoubles = 32;  // the sketch counter of the persistent grid

enum AnalyzeKernel { kAnWarp = 0, kAnCta = 1, kAnGroup = 2 };

// One fk_batch_analyze launch as choose_analyze plans it.
struct AnalyzePlan {
    int kernel = kAnWarp;
    uint32_t nsteps = 0, ld = 0;   // rows of the workspace matrix (min(n_expr, n_vars)) and its row stride
    uint64_t slot_doubles = 0;     // one sketch's workspace
    uint32_t slots = 0, group = 1; // workspaces (sketches in flight) and CTAs per sketch; grid = slots * group
    uint64_t workspace_bytes() const { return kernel == kAnWarp ? 0 : sizeof(double) * (kAnHeadDoubles + slots * slot_doubles); }
};

// The kernel of a batch of n_sketches sketches with n_vars variables and n_expr expressions on `device`: the warp kernel
// where its matrix fits shared memory; otherwise one CTA per sketch when the batch fills the device (fewer than two CTAs
// per sketch would be left for groups), groups of CTAs below that.  FK_ANALYZE_KERNEL=warp|cta|group forces one (tests,
// A/B); a forced warp kernel on a matrix it cannot hold is refused.  Returns FK_OK, FK_ERR_TOO_LARGE (with the sizes in
// *err) or a CUDA failure as FK_ERR_CUDA.
int choose_analyze(uint32_t n_vars, uint32_t n_expr, uint32_t n_sketches, int device, AnalyzePlan* plan, std::string* err);

// Launches plan.kernel (cta / group) on `ws` (plan.workspace_bytes(), used by this launch alone until it completes).
int launch_analyze(const AnalyzePlan& plan, uint32_t n_vars, uint32_t n_expr, const uint8_t* kinds, const uint32_t* slot_var,
                   uint32_t n_sketches, const double* vars, const double* params, uint8_t* out, double* ws, void* stream);

}  // namespace fk
