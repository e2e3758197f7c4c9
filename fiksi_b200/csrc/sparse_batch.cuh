// Batched LM for topologies on the global sparse path (info.path == 2): ONE CTA PER SKETCH runs the whole LM loop of
// fiksi/src/solve/lm.rs:21-193 on the device -- evaluation, g = -Jᵀr, the supernodal multifrontal LDLᵀ of JᵀJ + lambda I,
// both triangular solves and every accept / reject decision -- with the same decisions, trace codes and report counters
// as the single-system path (sparse_path.cu).  The sketch's vectors, Jacobians, factor panels and pending update matrices
// live in a per-CTA workspace in global memory (L2 resident for the sizes this kernel serves); the front being factorised
// lives in shared memory as a packed lower triangle, which bounds the largest front the kernel takes (kSbMaxFront).
// A persistent grid: each CTA takes sketch after sketch, so the workspace scales with the resident CTAs, not the batch.
#pragma once
#include <algorithm>
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/fiksi_b200.h"

namespace fk {

struct Topology;
struct DevProgram;

// Largest front order the kernel holds in shared memory: a packed lower triangle of f(f+1)/2 doubles, at most
// 236 * 237 / 2 * 8 = 223,728 bytes of the 227 KB a CTA may have.
constexpr uint32_t kSbMaxFront = 236;

// Device memory of one workspace (one per batch plan; the host-buffer pipeline keeps eight plans per (topology, device)).
// Lattices up to 64x50 stay below it with every resident CTA (64x50: 148 x 3.9 MiB); systems with many variables and small
// fronts (long trusses) get fewer CTAs instead of tens of gigabytes.
constexpr uint64_t kSbWorkspaceBytes = 1ull << 30;

// Device tables of one (topology, device); host side of the kernel's parameter block.
struct SbDev {
    uint32_t n, m, n_vars, n_expr, S;
    // evaluation tables of the topology (DevProgram, tile == 1 layout) and the free variables
    const uint32_t* row_hdr;
    const uint2* row_slots;
    const uint32_t* free_vars;
    const uint32_t* g_ptr;    // [n+1] per permuted column: (Jacobian position, row) pairs of g = -Jᵀr
    const uint32_t* g_pairs;
    const int32_t* perm;      // perm[k] = original column at permuted position k
    const uint32_t* l_colptr; // [n+1] L column starts: entry (i, j) of L is h list l_colptr[j] + (i - j) of its front
    const uint32_t* h_ptr;    // [lnnz+1] contributions to every L entry of H = JᵀJ
    const uint32_t* h_pairs;  // 2 Jacobian positions per contribution
    const uint32_t* post;     // [S] supernodes in postorder (children ascending)
    const uint4* sn;          // [S] {first column, pivot columns, front order, row list offset}
    const uint4* sn2;         // [S] {rel offset, unused, panel offset, update-stack offset}
    const uint32_t* child_ptr;  // [S+1]
    const uint32_t* child;
    const uint32_t* rows;
    const uint32_t* rel;
    // per-CTA workspace layout (doubles from the CTA's base)
    uint32_t o_x, o_xs, o_g, o_w, o_d, o_r, o_rs, o_J, o_Jt, o_pan, o_stk;
    uint64_t ws_doubles;
};

// Host analysis of a topology for the kernel (no CUDA calls): the largest front, and the message of FK_ERR_TOO_LARGE when it
// exceeds kSbMaxFront.  Returns FK_OK or FK_ERR_TOO_LARGE / FK_ERR_INTERNAL.
int sparse_batch_fits(const Topology& t, uint32_t* max_front, std::string* err);

class SparseBatchProgram {
public:
    SparseBatchProgram() = default;
    ~SparseBatchProgram();
    SparseBatchProgram(const SparseBatchProgram&) = delete;
    SparseBatchProgram& operator=(const SparseBatchProgram&) = delete;
    // Supernodal analysis, postorder, update-stack offsets and uploads.  `prog` holds the evaluation tables on `device`.
    int init(const Topology& t, const DevProgram& prog, int device, std::string* err);
    // CTAs a workspace for launches of up to `capacity` sketches has room for: at most one per resident CTA (the persistent
    // grid), and at most what kSbWorkspaceBytes holds (at least one).  Fewer CTAs only means fewer sketches in flight.
    uint32_t workspace_ctas(uint32_t capacity) const {
        const uint64_t budget = std::max<uint64_t>(1, kSbWorkspaceBytes / (sizeof(double) * dev_.ws_doubles));
        return (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>({capacity, resident_, budget}));
    }
    uint64_t workspace_doubles(uint32_t ctas) const { return kHeadDoubles + (uint64_t)ctas * dev_.ws_doubles; }
    // Solves n sketches (vars[n][n_vars], params[n][n_expr] -> free_out[n][n_free], reports[n]) with min(n, ctas) CTAs on
    // `workspace` (workspace_doubles(ctas) doubles, used by this launch alone until it completes).
    int launch(uint32_t n, const double* vars, const double* params, double* free_out, fk_report* reports, double* workspace, uint32_t ctas,
               void* stream) const;
    static constexpr uint64_t kHeadDoubles = 32;  // the sketch counter of the persistent grid

private:
    SbDev dev_{};
    std::vector<void*> owned_;
    int device_ = -1;
    uint32_t resident_ = 0, smem_ = 0;
};

}  // namespace fk
