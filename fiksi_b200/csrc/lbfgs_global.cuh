// L-BFGS (fiksi/src/solve/lbfgs.rs) for systems of any size: ONE CTA PER SKETCH runs lbfgs_solve (lbfgs_core.cuh) with
// the sketch's state in a per-CTA workspace in global memory, in the tile kernel's layout (x, xs, g, dir, sh[5][n],
// yh[5][n], r[m], J[jnnz], rho[5], alpha[5]).  Every floating-point operation happens in the tile kernel's order, so the
// results are bit-identical to it and to the oracle: rows and columns are spread over the CTA's threads, and each
// control scalar is a sequential sum in index order whose products the whole CTA forms first.
// A persistent grid: each CTA takes sketch after sketch, so the workspace scales with the resident CTAs, not the batch.
#pragma once
#include <cstdint>

#include "../../include/fiksi_b200.h"
#include "lm_kernels.cuh"

namespace fk {

// Device memory of one workspace (one per batch plan).  A large system gets fewer CTAs in flight, not more memory.
constexpr uint64_t kLbWorkspaceBytes = 1ull << 30;
constexpr uint64_t kLbHeadDoubles = 32;  // the sketch counter of the persistent grid

// Doubles of one CTA's state for a topology with n free variables, m rows and jnnz Jacobian entries.
uint64_t lbfgs_cta_doubles(uint32_t n, uint32_t m, uint32_t jnnz);
// CTAs a workspace for launches of up to `capacity` sketches has room for on the current device: at most one per resident
// CTA and at most what kLbWorkspaceBytes holds (at least one).  0 when the device cannot be queried.
uint32_t lbfgs_workspace_ctas(const DevProgram& prog, uint32_t capacity);
inline uint64_t lbfgs_workspace_doubles(const DevProgram& prog, uint32_t ctas) {
    return kLbHeadDoubles + (uint64_t)ctas * lbfgs_cta_doubles(prog.n, prog.m, prog.jnnz);
}
// Solves n sketches (vars[n][n_vars], params[n][n_expr] -> free_out[n][n_free], reports[n]) with min(n, ctas) CTAs on
// `workspace` (lbfgs_workspace_doubles(prog, ctas) doubles, used by this launch alone until it completes).  Returns
// cudaErrorInvalidConfiguration when a Jacobian position does not fit the 24 bits of the row tables.
int launch_lbfgs_cta(const DevProgram& prog, const uint32_t* d_jcolptr, const uint32_t* d_jrow, uint32_t n, const double* vars,
                     const double* params, double* free_out, fk_report* reports, double* workspace, uint32_t ctas, void* stream);

}  // namespace fk
