// Host-side symbolic pipeline of the product: everything that depends only on the topology of a
// flattened problem (kinds, indices, free set, row list) and is therefore computed once and
// reused by every Levenberg–Marquardt iteration of every sketch with that topology.
//
// Replaces, per LM call in the reference:
//   Subsystem slot lookups            fiksi/src/subsystem.rs:126-166, variable_map.rs:57-72
//   SparseColMat::from_triplet_mat    solvi/src/sparse_col_mat.rs:690-737   (CSC pattern, per step!)
//   colamd_rs::colamd                 colamd_rs/src/colamd.rs:354-494
//   permute_columns / elimination_tree / CholeskyStructure
//                                     solvi/src/sparse_col_mat.rs:456-502,
//                                     solvi/src/decomposition/sparse/cholesky.rs:31-84,359-595
// and adds what the normal-equation formulation needs (reference has no counterpart): the
// contribution lists of H = JᵀJ, the LDLᵀ update schedule and the triangular-solve schedules.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/fiksi_b200.h"

namespace fk {

// Number of variable slots per expression kind (fiksi/src/constraints/expressions.rs:48-182).
inline int kind_arity(uint8_t kind) {
    static const int a[FK_NUM_KINDS] = {2, 4, 6, 6, 6, 5, 8, 8, 8, 8, 7, 6, 6};
    return kind < FK_NUM_KINDS ? a[kind] : -1;
}
// Expands the stored base indices into variable slots.  Returns arity or -1.
int expand_slots(uint8_t kind, const uint32_t idx[4], uint32_t out[8]);

// Sketch-kernel table records that eliminate two columns (Topology::SketchTables): the flag in the record's first word,
// and the largest C (entries below column k's diagonal) such a record takes.
constexpr uint32_t kSkPairFlag = 0x10000u;
constexpr uint32_t kSkPairMaxC = 8;

struct Topology {
    // ---- copy of the structural inputs -----------------------------------------------------
    uint32_t n_vars = 0, n_expr = 0, n_free = 0, n_rows = 0;
    std::vector<uint8_t> kind;       // [n_expr]
    std::vector<uint32_t> idx;       // [n_expr][4]
    std::vector<uint32_t> free_vars; // [n_free]
    std::vector<uint32_t> rows;      // [n_rows]
    uint64_t signature = 0;          // hash of the above (grouping key of fk_lm_solve_batch)

    // ---- per-row slot tables (a1, a4, a5 of SURVEY §8a) ------------------------------------
    std::vector<uint8_t> row_kind;   // [n_rows]
    std::vector<uint32_t> row_expr;  // [n_rows] expression id (parameter index)
    std::vector<uint32_t> slot_var;  // [n_rows][8] global variable index
    std::vector<int32_t> slot_col;   // [n_rows][8] free column, -1 if fixed, -2 if unused slot
    std::vector<int32_t> slot_pos;   // [n_rows][8] position in the Jacobian value array, -1 if none
    std::vector<uint8_t> slot_dup;   // [n_rows][8] 1: an earlier slot of this row has the same column
    uint64_t eval_bytes = 0;         // algorithmic bytes of one residual+Jacobian evaluation (§8d)

    // ---- patterns ---------------------------------------------------------------------------
    // Augmented (n_rows + n_free) x n_free CSC pattern: per column ascending expression rows, then
    // the damping row n_rows + c (fiksi/src/solve/lm.rs:92-98).  Bit-exact parity object #1.
    std::vector<uint32_t> aug_colptr, aug_rowidx;
    uint32_t jac_nnz = 0;            // aug_nnz - n_free; Jacobian values are stored in CSC order
    std::vector<int32_t> perm;       // COLAMD: perm[k] = original column at position k.  Parity #2.
    std::vector<int32_t> iperm;      // iperm[c] = position of original column c
    std::vector<int32_t> parent;     // column elimination tree of A*P (-1 root)
    std::vector<uint32_t> r_colptr, r_rowidx;  // R = Lᵀ pattern, per column ascending rows, diagonal last
    std::vector<uint32_t> l_colptr, l_rowidx;  // L pattern (CSC), per column diagonal first, then ascending
    uint32_t etree_height = 0;
    uint64_t chol_flops = 0;

    // ---- schedules for the shared-memory LM kernel (empty when the problem takes the global path)
    std::vector<uint32_t> h_ptr;     // [l_nnz+1] contributions of every L position
    std::vector<uint32_t> h_pairs;   // 2 Jacobian positions per contribution
    std::vector<uint32_t> g_ptr;     // [n_free+1] per permuted column: (Jacobian position, row) pairs
    std::vector<uint32_t> g_pairs;
    std::vector<uint32_t> u_ptr;     // [n_free+1] per column: update triples (dst, a, b) of the LDLᵀ step
    std::vector<uint32_t> u_trip;
    std::vector<uint32_t> r_lpos;    // [r_nnz] position in L storage of every R entry (back substitution)
    uint32_t max_col_updates = 0;

    uint32_t path = 0, tile = 32, smem_bytes = 0;

    // ---- lane-padded, packed op tables of the shared-memory kernel (built for `tile` lanes) ----------
    // Every phase of the kernel is a sequence of "rounds"; in a round each lane executes at most one
    // packed op (0xFFFFFFFF.. = no-op), so the device loops have uniform trip counts and no
    // data-dependent branches.  All positions are 16-bit offsets into per-sketch shared arrays.
    struct Tables {
        int32_t uniform_kind = -1;          // all rows share this kind (specialised evaluator), else -1
        uint32_t eval_rounds = 0;           // ceil(m / tile)
        std::vector<uint32_t> row_hdr;      // [eval_rounds*tile] kind | expr << 8, NOP for padding
        std::vector<uint32_t> row_slots;    // [rows][8][2]: {source, jpos}: source = col | 0x80000000|var
        // Every sequential phase is a flat list of steps; step s executes ops[s*tile + lane].  Step
        // flags: bit 16 = first step of a column / accumulation, bit 17 = last (barrier / store).
        // Each list carries one padding step at the end so the kernel can prefetch step s+1.
        uint32_t a_nsteps = 0, g_nsteps = 0, f_nsteps = 0, s_nsteps = 0, b_nsteps = 0;
        std::vector<uint32_t> a_flags, a_ops, a_dst;  // H = JtJ: ops ja | jb << 16, dst = L position
        std::vector<uint32_t> g_flags, g_ops, g_dst;  // g = Jt r: ops jpos | row << 16, dst = column
        std::vector<uint32_t> f_steps;      // LDLt: diag position | flags
        std::vector<uint32_t> f_ops;        // [steps*tile][2]: {dst | a << 16, b}
        std::vector<uint32_t> s_steps;      // forward substitution [steps][2]: {diag position | flags, k}
        std::vector<uint32_t> s_ops;        // row | lpos << 16
        std::vector<uint32_t> b_steps;      // backward substitution [steps][2]: {diag position | flags, k | perm[k] << 16}
        std::vector<uint32_t> b_ops;        // row | lpos << 16
    } tab;
    int build_tables();

    // ---- tables of the sketch-per-thread LM kernel (lm_sketch.cu) -----------------------------------------
    // One THREAD owns one sketch; the state of the 32 sketches of a warp is interleaved in shared memory
    // (`entry * 32 + lane` doubles), so every access of a warp is 32 consecutive doubles (no bank conflicts)
    // and the tables below are warp-uniform: a CTA keeps one copy in shared memory and every warp reads them
    // with 16-byte broadcast loads.  Table words are 32 bit; positions are BYTE offsets (entry << 8) relative to the
    // region they address.  Regions of a sketch's state, in entries (doubles):
    //   xa, xb [n]   accepted / trial free values (the two roles swap per lane on accept)
    //   w  [n]       g = -J^T r in permuted order, then right-hand side and solution of the solve
    //   f  [lnnz]    H = J^T J in L storage, factorised in place
    //   fx [nfix]    values of the fixed variables some row reads;  pr [npar] parameters some row reads
    struct SketchTables {
        bool ok = false;          // false: the topology stays on the tile kernel (reason in `why`)
        std::string why;
        uint32_t entries = 0;
        uint32_t xa = 0, xb = 0, w = 0, f = 0, fx = 0, pr = 0, nfix = 0, npar = 0;
        // sections of `tab` (offsets in words):
        //   free   [n]      variable index of free column c
        //   fix    [nfix]   variable index;  par [npar] expression index
        //   (records of the three sections below start on 16-byte boundaries; header = first 4 words)
        //   eval   per row: header (kind | 0x100 if a slot is fixed | words of this row << 16), parameter
        //          position in pr, A sources (position in x; 0x80000000 | position in fx for a fixed variable),
        //          A gradient targets in w (0xFFFFFFFF none), A(A+1)/2 targets in f ((a, b), b <= a; 0xFFFFFFFF none)
        //   factor per column k: C (entries below the diagonal), diagonal position, position of k in w, 0,
        //          C positions in f, C positions in w (rows), C(C+1)/2 update targets in f ((a, b), b <= a)
        //   back   per column k descending: C, diagonal position, position of k in w, position of perm[k] in x,
        //          C positions in f, C positions in w (rows)
        //   Column pairs (build_sketch_tables): when L(:,k) = {k+1} u L(:,k+1) and C <= kSkPairMaxC, ONE record
        //   eliminates columns k and k+1 and carries kSkPairFlag in its first word.  The factor pair record is column
        //   k's record: column k+1's diagonal, entries and w position are column k's target (0, 0), targets (a, 0) for
        //   a >= 1 and first w row.  The back pair record (for k+1, then k) is column k's back record followed by the
        //   C - 1 positions in f of column k+1's entries, column k+1's diagonal position and the position of perm[k+1].
        uint32_t off_free = 0, off_fix = 0, off_par = 0, off_eval = 0, off_factor = 0, off_back = 0;
        std::vector<uint32_t> tab;
    } sk;
    void build_sketch_tables();

    std::string error;

    // Runs the whole pipeline.  Returns FK_OK or an error status (message in `error`).
    // `lanes` != 0 overrides the lanes per sketch of the tile path (the latency-oriented twin of a topology uses 32).
    int build(const fk_problem& p, uint32_t lanes = 0);
    void fill_info(fk_topology_info* info) const;
};

}  // namespace fk
