/*
 * fiksi_b200 — C ABI of the B200-native Fiksi numeric solve path.
 *
 * This header is the drop-in boundary.  In the reference the seam is a crate-private Rust generic,
 *     pub(crate) fn levenberg_marquardt<P: Problem>(problem: &mut P, variables: &mut [f64])
 *         (fiksi/src/solve/lm.rs:21, trait Problem at fiksi/src/solve/mod.rs:29-49),
 * called from fiksi/src/assemble/mod.rs:150 with a `Subsystem` built at assemble/mod.rs:132-146.
 * A per-row callback cannot cross to a GPU, so the boundary moves up to the data `Subsystem::new`
 * receives: the flattened problem below.  Everything is plain pointers and sizes; all pointers are
 * HOST memory owned by the caller unless a function says "device".  No function aborts: each
 * returns FK_OK (0) or a negative fk_status and leaves a message for fk_last_error().
 *
 * There is no CPU fallback: every solve entry point fails with FK_ERR_NO_DEVICE / FK_ERR_CUDA when
 * no sm_100a device is usable.
 */
#ifndef FIKSI_B200_H
#define FIKSI_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FK_API __attribute__((visibility("default")))

typedef enum fk_status {
    FK_OK = 0,
    FK_ERR_INVALID = -1,    /* null pointer, index out of range, unknown kind */
    FK_ERR_NO_DEVICE = -2,  /* no CUDA device / wrong architecture */
    FK_ERR_CUDA = -3,       /* CUDA runtime failure (message in fk_last_error) */
    FK_ERR_OOM = -4,        /* host or device allocation failed */
    FK_ERR_TOO_LARGE = -5,  /* problem does not fit the selected path */
    FK_ERR_INTERNAL = -6
} fk_status;

/* Expression kinds in the order of `enum Expression`, fiksi/src/constraints/expressions.rs:28-40. */
typedef enum fk_kind {
    FK_VARIABLE_VARIABLE_EQUALITY = 0,      /* idx: v1, v2                     slots 2 */
    FK_POINT_POINT_DISTANCE = 1,            /* idx: p1, p2          param dist  slots 4 */
    FK_POINT_POINT_POINT_ANGLE = 2,         /* idx: p1, p2, p3      param angle slots 6 */
    FK_POINT_LINE_INCIDENCE = 3,            /* idx: p, l1, l2                  slots 6 */
    FK_POINT_LINE_DISTANCE = 4,             /* idx: p, l1, l2       param dist  slots 6 */
    FK_POINT_CIRCLE_INCIDENCE = 5,          /* idx: p, center, radius_var      slots 5 */
    FK_SEGMENT_SEGMENT_LENGTH_EQUALITY = 6, /* idx: s1p1, s1p2, s2p1, s2p2     slots 8 */
    FK_LINE_LINE_ANGLE = 7,                 /* idx: l1p1, l1p2, l2p1, l2p2 param angle  8 */
    FK_LINE_LINE_PARALLELISM = 8,           /* same idx                        slots 8 */
    FK_LINE_LINE_PERPENDICULARITY = 9,      /* same idx                        slots 8 */
    FK_LINE_CIRCLE_TANGENCY = 10,           /* idx: l1, l2, center, radius_var slots 7 */
    /* The two coincidence rows `ClusteredSystem` adds per (cluster, frontier point) for Decomposer::RecursiveAssembly
     * (fiksi/src/assemble/mod.rs:538-585, Pose2D: constraints/expressions.rs:1094-1159); not members of the
     * reference's `enum Expression`.  idx: pose (rotation, tx, ty: three consecutive variables), the updated
     * coordinate (one variable), the point before the step (u, v: two consecutive variables, fixed).
     * residual x: tx + u cos - v sin - updated;  y: ty + u sin + v cos - updated. */
    FK_POSE_POINT_X = 11,                   /* idx: pose, updated_x, point             slots 6 */
    FK_POSE_POINT_Y = 12,                   /* idx: pose, updated_y, point             slots 6 */
    FK_NUM_KINDS = 13
} fk_kind;

/*
 * The flattened problem == the arguments of `Subsystem::new` (fiksi/src/assemble/mod.rs:132-146):
 *   vars      system.variables_transformed: scaled, free ones already perturbed; fixed variables
 *             are read from here (fiksi/src/variable_map.rs:57-72)
 *   kind/idx/param   system.expressions_transformed as SoA; idx holds the base indices exactly as
 *             stored in the Expression structs (a point index p expands to slots p, p+1,
 *             expressions.rs:48-182); param is the scaled distance or the angle, 0 if none
 *   free_vars ascending global variable indices == IndexSet order (fiksi/src/subsystem.rs:22,35)
 *   rows      expression ids of this problem in row order (assemble/mod.rs:136-145)
 */
typedef struct fk_problem {
    uint32_t n_vars;
    const double* vars;
    uint32_t n_expr;
    const uint8_t* kind;   /* [n_expr] */
    const uint32_t* idx;   /* [n_expr][4] */
    const double* param;   /* [n_expr] */
    uint32_t n_free;
    const uint32_t* free_vars; /* [n_free] */
    uint32_t n_rows;
    const uint32_t* rows;  /* [n_rows] */
} fk_problem;

/* Exit reasons == the four exits of fiksi/src/solve/lm.rs plus the guard for its unbounded loop. */
typedef enum fk_exit {
    FK_EXIT_CONVERGED_RESIDUAL = 0, /* sum r^2 < 1e-8                       lm.rs:110-112 */
    FK_EXIT_SMALL_STEP = 1,         /* sum delta^2 < 1e-12                  lm.rs:139-142 */
    FK_EXIT_STALLED = 2,            /* relative decrease <= 1e-6            lm.rs:164-168 */
    FK_EXIT_MAX_OUTER = 3,          /* 100 outer iterations                 lm.rs:109     */
    FK_EXIT_LAMBDA_OVERFLOW = 4     /* lambda reached +inf: the reference would spin forever */
} fk_exit;

/* New output (the reference returns `()`, fiksi/src/lib.rs:464-466). 40 bytes. */
typedef struct fk_report {
    uint32_t exit_reason;    /* fk_exit */
    uint32_t outer_iters;    /* outer iterations that entered the damping loop */
    uint32_t factorizations; /* damping-loop iterations (one factor + solve each) */
    uint32_t accepted;       /* accepted steps */
    double ssr;              /* sum of squared residuals at the returned variables (scaled units) */
    double lambda;           /* final damping factor */
    uint64_t trace_hash;     /* h = 3h + code + 1 per decision; code 0 unsolved, 1 accept, 2 reject */
} fk_report;

/* ---- library / device ------------------------------------------------------------------- */
FK_API int fk_version(void);
FK_API const char* fk_last_error(void);          /* thread-local, never NULL */
FK_API int fk_device_count(void);                /* usable CUDA devices, 0 if none */

/* ---- symbolic analysis, computed once per topology --------------------------------------- */
/* A topology is a problem without its numbers: kinds, indices, free set and row list.  Creating
 * it runs the host symbolic pipeline that replaces, per LM call in the reference,
 *   SparseColMat::from_triplet_mat   solvi/src/sparse_col_mat.rs:690-737   (augmented CSC pattern)
 *   colamd_rs::colamd                colamd_rs/src/colamd.rs:354-494       (column permutation)
 *   elimination_tree / post_order / CholeskyCounts / CholeskyStructure
 *                                    solvi/src/decomposition/sparse/cholesky.rs:31-595
 * `vars` and `param` of the problem are ignored. */
typedef struct fk_topology fk_topology;

typedef struct fk_topology_info {
    uint32_t n_vars, n_expr, n_free, n_rows;
    uint32_t jac_nnz;      /* structural entries of J (duplicates merged), without damping rows */
    uint32_t aug_nnz;      /* jac_nnz + n_free */
    uint32_t r_nnz;        /* entries of R = L^T including the diagonal */
    uint32_t etree_height; /* longest root-to-leaf path, in columns */
    uint32_t path;         /* 0 tile-per-sketch (shared memory), 1 CTA-per-sketch, 2 global sparse */
    uint32_t tile;         /* lanes per sketch on path 0/1 */
    uint32_t smem_bytes;   /* shared memory per sketch on path 0/1 */
    uint32_t eval_bytes;   /* algorithmic bytes of one residual+Jacobian evaluation of one sketch (SURVEY 8d) */
    uint64_t chol_flops;   /* sum over columns of colcount^2: flops of one sparse factorisation */
} fk_topology_info;

FK_API int fk_topology_create(const fk_problem* problem, fk_topology** out);
FK_API void fk_topology_destroy(fk_topology* topo);
FK_API int fk_topology_info_get(const fk_topology* topo, fk_topology_info* info);

/* Parity probes.  Each output may be NULL.  Sizes: aug_colptr[n_free+1], aug_rowidx[aug_nnz],
 * colamd_perm[n_free], etree_parent[n_free] (-1 == root; of the permuted matrix), r_colptr[n_free+1],
 * r_rowidx[r_nnz] (pattern of R, per column ascending rows, diagonal last — identical to
 * SymbolicQr::r_structure, solvi/src/decomposition/sparse/qr.rs:80-82). */
FK_API int fk_topology_symbolic(const fk_topology* topo, uint32_t* aug_colptr, uint32_t* aug_rowidx,
                                int32_t* colamd_perm, int32_t* etree_parent, uint32_t* r_colptr,
                                uint32_t* r_rowidx);
/* Convenience: create + probe + destroy. */
FK_API int fk_symbolic(const fk_problem* problem, uint32_t* aug_colptr, uint32_t* aug_rowidx,
                       int32_t* colamd_perm, int32_t* etree_parent, uint32_t* r_colptr,
                       uint32_t* r_rowidx);

/* Solve one system with an existing topology (symbolic analysis reused across calls).  Takes the
 * batched shared-memory kernel with n = 1 or, for large systems (info.path == 2), the global
 * sparse path: K1/K2 evaluation, K3 normal-equation assembly and K5 sparse LDL^T on the device with
 * a thin host loop for the accept/reject decisions.  On the shared-memory path the first call builds a
 * twin of the topology with 32 lanes per sketch (single systems are latency bound; the topology's own
 * lane count is chosen for batch throughput); results do not depend on the lane count. */
FK_API int fk_topology_lm_solve(fk_topology* topo, const double* vars, const double* param,
                                double* free_values, fk_report* report);
/* Large systems only: one residual + Jacobian evaluation at free_values (out_r[n_rows],
 * out_j[jac_nnz] in CSC order, either may be NULL), timed over `repeats` launches. */
FK_API int fk_topology_eval(fk_topology* topo, const double* vars, const double* param,
                            const double* free_values, double* out_r, double* out_j, int repeats,
                            float* ms_per_eval);
/* Phase times of the last large-system solve: out8 = {eval ms, assemble ms, factor ms,
 * triangular-solve ms, evaluations, factorisations, forward ms, backward ms}. */
FK_API int fk_topology_last_timing(fk_topology* topo, float* out8);

/* Parity / structure probe of the large-system path (host only, no device needed): the supernodal
 * multifrontal analysis built on top of the R pattern of SymbolicQr::build (qr.rs:118-206).
 * Call once with all array pointers NULL to get the sizes, then with arrays of
 *   sn_first[n_supernodes+1]  first permuted column of every supernode (last entry = n_free)
 *   front[n_supernodes]       order of the frontal matrix (= column count of the first column of L)
 *   sn_parent[n_supernodes]   supernodal elimination tree (-1 root)
 *   rows[rows_total]          row lists of the fronts, concatenated in supernode order
 *   rel[rel_total]            for every update row of every supernode its position in the parent's front
 *   big[n_supernodes]         1: level-scheduled tiled path, 0: member of a one-warp subtree
 *   level[n_supernodes]       level of a big supernode (0 = no big child)
 *   tasks[4*n_tasks], launches[3*n_launches]  static task lists {supernode,row0,col0,packed} and the
 *                             launch sequence {kind (0 asm,1 diag,2 panel,3 update), first task, count}. */
typedef struct fk_supernodal_info {
    uint32_t n_supernodes, n_small_subtrees, n_big, n_levels, max_front, n_tasks, n_launches, pad0;
    uint64_t rows_total, rel_total, panel_doubles, update_doubles;
} fk_supernodal_info;
FK_API int fk_topology_supernodal(const fk_topology* topo, fk_supernodal_info* info, uint32_t* sn_first, uint32_t* front,
                                  int32_t* sn_parent, uint32_t* rows, uint32_t* rel, uint8_t* big, uint32_t* level,
                                  uint32_t* tasks, uint32_t* launches);

/* ---- Levenberg–Marquardt ----------------------------------------------------------------- */
/* == levenberg_marquardt(problem, variables), fiksi/src/solve/lm.rs:21.  free_values in/out,
 * length n_free.  Picks the batched kernel (n = 1) or the large sparse path by size. */
FK_API int fk_lm_solve(const fk_problem* problem, double* free_values, fk_report* report);

/* n independent problems (one per sketch or connected component).  Problems with identical
 * topology are grouped and solved by one batched launch per group and device; contiguous ranges
 * of each group go to the n_gpus devices (0 == all visible), no inter-GPU traffic. */
FK_API int fk_lm_solve_batch(uint32_t n, const fk_problem* const* problems,
                             double* const* free_values, fk_report* reports, int n_gpus);

/* Uniform batch: n sketches sharing one topology.  vars[n][n_vars], param[n][n_expr] (row-major,
 * one sketch after another), free_out[n][n_free], reports[n].  This is the throughput entry
 * point for configs 2, 4 and 5.  The batched entry points (this one, fk_batch_solve_device[_begin/_wait],
 * fk_batch_system_solve[_begin/_wait] and the batch plan) also take topologies on the global sparse path
 * (info.path == 2) whose largest supernodal front has at most 236 rows: one CTA per sketch runs the LM loop over
 * the supernodal tree with the front in shared memory (fk_topology_batch_kernel returns 3), with the decisions of
 * fk_topology_lm_solve.  Larger fronts: FK_ERR_TOO_LARGE naming the front order; solve such systems with
 * fk_topology_lm_solve. */
FK_API int fk_batch_solve(const fk_topology* topo, uint32_t n, const double* vars,
                          const double* param, double* free_out, fk_report* reports, int n_gpus);

/* Same on one explicit device (one process per GPU launches, e.g. under torchrun). */
FK_API int fk_batch_solve_device(const fk_topology* topo, int device, uint32_t n, const double* vars,
                                 const double* param, double* free_out, fk_report* reports);
/* The same call in two halves (see fk_batch_system_solve_begin / _wait: same token rules, the two kinds of call share the pipeline of a
 * (topology, device) and may be mixed). */
FK_API int fk_batch_solve_device_begin(const fk_topology* topo, int device, uint32_t n, const double* vars, const double* param,
                                       double* free_out, fk_report* reports, uint64_t* token);
FK_API int fk_batch_solve_device_wait(const fk_topology* topo, int device, uint64_t token);

/* System::solve for a batch of single-component sketches that share one topology, pre- and post-processing
 * included (fiksi/src/assemble/mod.rs:32-44,58-79,113-124,161-166): per sketch the RMS scale over all variables
 * and distance parameters, variables and distances divided by it, the seeded perturbation of the listed variables
 * (the reference re-seeds its generator with 42 on every solve, so every sketch sees the same draws), the LM solve,
 * and the solved free variables multiplied by the scale again.  All of it runs on `device`; the host only copies
 * raw_vars[n][n_vars] and raw_param ([n][n_expr], or ONE row with FK_PREP_SHARED_PARAM) in and free_out[n][n_free]
 * (UNSCALED values, i.e. what System::solve writes into system.variables), scales_out[n] (optional) and reports out.
 * Restriction: the sketch is one connected component whose problem names every variable and expression of the
 * system (the scale is a property of the whole system); fk_system_batch_solve takes any drawing of the fk_system mirror. */
enum { FK_PREP_SHARED_PARAM = 1, FK_PREP_PERTURB = 2 };
typedef struct {
    uint32_t flags;               /* FK_PREP_* */
    uint32_t n_perturb;           /* variables that draw from the generator, ascending; with perturb_vars == NULL: */
    const uint32_t* perturb_vars; /* the topology's free variables */
    uint32_t seed;                /* 42 in the reference (assemble/mod.rs:47) */
    uint32_t pad;
} fk_prepare_opts;
FK_API int fk_batch_system_solve(const fk_topology* topo, int device, uint32_t n, const double* raw_vars,
                                 const double* raw_param, const fk_prepare_opts* opts, double* free_out,
                                 double* scales_out, fk_report* reports);
/* The same call in two halves, so that a caller streaming batch after batch keeps the device busy across calls (the first chunk's
 * upload of the next batch and the last chunk's download of this one overlap the kernels of the other): _begin returns when every
 * chunk of the batch is enqueued (it waits, chunk by chunk, for a free slot of the pipeline) and hands out a token; _wait returns
 * when that batch's results are in its host buffers (kernel / copy errors surface there).  Up to two batches may be in flight per
 * (topology, device): begin(A), begin(B), wait(A), begin(C), wait(B), ...  Buffers of a batch in flight must not be reused
 * (inputs may be shared between batches, outputs not); pinned host memory is what makes the copies asynchronous. */
FK_API int fk_batch_system_solve_begin(const fk_topology* topo, int device, uint32_t n, const double* raw_vars,
                                       const double* raw_param, const fk_prepare_opts* opts, double* free_out,
                                       double* scales_out, fk_report* reports, uint64_t* token);
FK_API int fk_batch_system_solve_wait(const fk_topology* topo, int device, uint64_t token);

/* Device-resident batch plan (one device; used by bench.py and by fk_batch_solve internally).  Global sparse path
 * topologies are taken up to the front limit of fk_batch_solve (creation fails with FK_ERR_TOO_LARGE above it); their plan
 * also holds the kernel's workspace, one per resident CTA up to `capacity`. */
typedef struct fk_batch_plan fk_batch_plan;
FK_API int fk_batch_plan_create(const fk_topology* topo, uint32_t capacity, int device,
                                fk_batch_plan** out);
FK_API void fk_batch_plan_destroy(fk_batch_plan* plan);
/* Async H2D of n sketches from (ideally pinned) host memory on `stream` (cudaStream_t, may be 0). */
FK_API int fk_batch_plan_upload(fk_batch_plan* plan, uint32_t n, const double* vars,
                                const double* param, void* stream);
/* Launch the LM kernel over the n resident sketches.  Inputs are not modified, so the call can be
 * repeated on the same resident data. */
FK_API int fk_batch_plan_run(fk_batch_plan* plan, void* stream);
/* Async D2H of results of the last run. */
FK_API int fk_batch_plan_download(fk_batch_plan* plan, double* free_out, fk_report* reports,
                                  void* stream);
/* Device pointers of the resident buffers (any may be NULL): vars, param, free_out, reports. */
FK_API int fk_batch_plan_device_ptrs(fk_batch_plan* plan, void** vars, void** param,
                                     void** free_out, void** reports);
/* Number of kernel launches issued by this plan so far / name of the LM kernel. */
FK_API uint64_t fk_batch_plan_launches(const fk_batch_plan* plan);

/* Measured FP64 DFMA throughput of `device` in TFLOP/s (roofline denominator for the
 * factorisation; MEASURED_PEAKS.json carries no FP64 figure). */
FK_API int fk_fp64_peak_tflops(int device, double* out);

/* Which batched LM kernel fk_batch_plan_run / fk_batch_solve* launch: -1 automatic (the
 * sketch-per-thread kernel for batches that fill the device, the tile kernel otherwise), 0 always the
 * tile kernel, 1 the sketch-per-thread kernel whenever the topology has one (2: always its one-warp-per-32-sketches
 * shape, 3: always its warp-pair shape when that fits).  Process-wide; meant for tests and A/B measurements
 * (environment: FK_LM_KERNEL=tile|sketch, FK_SK_PAIR=0|1). */
FK_API void fk_set_lm_kernel(int choice);
FK_API int fk_get_lm_kernel(void);
/* Sketch-per-thread kernel of a topology: *available = 0/1, *state_doubles = shared-memory doubles per
 * sketch, *table_words = 16-bit words of its parameter block.  Any pointer may be null. */
FK_API int fk_topology_sketch_kernel_info(const fk_topology* topo, int* available, uint32_t* state_doubles, uint32_t* table_words);

/* Which kernel a batched LM solve of n_sketches sketches of this topology launches under the current
 * fk_set_lm_kernel choice: 0 tile kernel, 1 sketch-per-thread (one warp per 32 sketches), 2 sketch-per-thread in its
 * warp-pair shape, 3 the one-CTA-per-sketch kernel of the global sparse path (negative: error, FK_ERR_TOO_LARGE when a
 * global sparse path topology has a front of more than 236 rows). */
FK_API int fk_topology_batch_kernel(const fk_topology* topo, uint32_t n_sketches);

/* Topology cache of fk_lm_solve / fk_lm_solve_batch / fk_system_solve*: the symbolic analysis of a flattened
 * problem (the reference repeats it on every LM call, fiksi/src/solve/lm.rs:98-104) is kept in a process-wide
 * LRU keyed by the problem's structure, so that re-solving a sketch costs no analysis.  Default capacity 1024
 * topologies (environment FK_TOPOLOGY_CACHE; 0 disables).  Cached topologies keep their device tables and
 * staging buffers; _clear releases them. */
FK_API void fk_topology_cache_configure(uint32_t capacity);
FK_API void fk_topology_cache_clear(void);
FK_API void fk_topology_cache_stats(uint64_t* hits, uint64_t* misses, uint32_t* entries);

/* Blocks until all work issued for this plan's device has finished. */
FK_API int fk_batch_plan_sync(fk_batch_plan* plan);

/* Pinned host memory helpers (so that callers without a CUDA binding can stage inputs). */
FK_API void* fk_host_alloc(size_t bytes);
FK_API void fk_host_free(void* p);

/* ---- residual / Jacobian evaluation kernels on their own (assembly GB/s metric) ----------- */
/* Evaluates all rows of n sketches of a topology once: residuals out_r[n][n_rows] and Jacobian
 * values scattered into the precomputed CSC pattern out_j[n][jac_nnz] (device-resident plan
 * buffers).  == Subsystem::calculate_residuals_and_sparse_jacobian, fiksi/src/subsystem.rs:126-166
 * followed by SparseColMat::from_triplet_mat.  mode 0: residuals + Jacobian (K1); mode 1:
 * residuals only (K2, subsystem.rs:93-104).  Shared-memory paths only: FK_ERR_TOO_LARGE on a global sparse path
 * plan (fk_topology_eval evaluates those). */
FK_API int fk_batch_plan_eval(fk_batch_plan* plan, int mode, void* stream);
FK_API int fk_batch_plan_eval_download(fk_batch_plan* plan, double* out_r, double* out_j, void* stream);

/* ---- Decomposer::SinglePass on a uniform batch (SURVEY 8f-1) ------------------------------------------ */
/* The loop of fiksi/src/assemble/mod.rs:169-210 for n sketches sharing one topology whose free set is one
 * connected component: the plan (maximum matching + strongly connected expression sets,
 * analyze/graph/equations.rs, over ALL n_expr expressions of the topology) is computed once on the host,
 * then every set is ONE batched LM launch over all n sketches, later sets seeing earlier results as fixed
 * values.  vars[n][n_vars] is updated in place (scaled / perturbed by the caller as for fk_batch_solve);
 * reports[n][steps] (may be NULL), *n_steps receives the number of sets. */
FK_API int fk_batch_solve_single_pass(const fk_topology* topo, uint32_t n, double* vars, const double* param,
                                      fk_report* reports, uint32_t* n_steps, int n_gpus);

/* ---- L-BFGS (SURVEY 8f-3) ----------------------------------------------------------------------------- */
/* == lbfgs(problem, variables), fiksi/src/solve/lbfgs.rs:20 (Optimizer::LBfgs, assemble/mod.rs:155-157)
 * for n sketches sharing one topology: vars[n][n_vars] / param[n][n_expr] scaled and perturbed exactly
 * as for the LM entry points, free_out[n][n_free].  reports[k]: exit_reason 0 initial sum of squares
 * < 1e-4 (lbfgs.rs:53-56), 1 change < 1e-10 (:177-179), 2 sum of squares < 1e-6 (:180-182), 3 100
 * iterations, 4 guard (the reference's unbounded bisection loop, :338-351, would not return);
 * outer_iters = line searches, factorizations = residual+Jacobian evaluations, ssr, lambda = last step
 * size, trace_hash = h*31 + evaluations per line search.  Shared-memory tile paths only
 * (FK_ERR_TOO_LARGE otherwise); fk_lbfgs_solve_batch takes systems of every size. */
FK_API int fk_batch_solve_lbfgs(const fk_topology* topo, int device, uint32_t n, const double* vars, const double* param,
                                double* free_out, fk_report* reports);
/* Same on the resident sketches of a batch plan (fk_batch_plan_upload / _download around it).  Tile paths only, as
 * fk_batch_solve_lbfgs; fk_batch_plan_run_lbfgs_global runs any plan. */
FK_API int fk_batch_plan_run_lbfgs(fk_batch_plan* plan, void* stream);
/* Same with the CTA kernel on any plan: one CTA of 256 threads per sketch, the sketch's L-BFGS state in global memory,
 * bit-identical to the tile kernel.  The plan grows its workspace on first use (at most 1 GiB: a large system gets
 * fewer CTAs in flight) and frees it with the plan. */
FK_API int fk_batch_plan_run_lbfgs_global(fk_batch_plan* plan, void* stream);
/* L-BFGS kernel the batch calls use for a topology: 0 the tile kernel (every topology fk_batch_solve_lbfgs takes),
 * 1 the CTA kernel (every other topology; no size limit but device memory).  Host only. */
FK_API int fk_topology_lbfgs_kernel(const fk_topology* topo, uint32_t n_sketches);
/* The L-BFGS counterparts of fk_lm_solve / fk_lm_solve_batch, for systems of every size: problems grouped by structure
 * through the topology cache, one launch per group (the kernel of fk_topology_lbfgs_kernel), groups placed on or
 * sharded over n_gpus devices as fk_lm_solve_batch does.  Reports as fk_batch_solve_lbfgs. */
FK_API int fk_lbfgs_solve(const fk_problem* problem, double* free_values, fk_report* report);
FK_API int fk_lbfgs_solve_batch(uint32_t n, const fk_problem* const* problems, double* const* free_values, fk_report* reports,
                                int n_gpus);

/* ---- System::analyze: over-constraint detection (SURVEY 8f-2) -------------------------------------- */
/* == find_overconstraints (fiksi/src/analyze/numerical/mod.rs:123-163) for n sketches sharing one
 * topology: the dense Jacobian of ALL n_expr expressions with respect to ALL n_vars variables (the
 * reference treats every variable as free here, :124) at the UNSCALED variables vars[n][n_vars] /
 * parameters param[n][n_expr], reduced by incremental_gauss_jordan_elimination (:33-117, epsilon 1e-8).
 * independent[n][n_expr] receives 1 for an expression that increases the rank, 0 for a dependent one
 * (the constraint owning a dependent expression is what System::analyze reports as overconstrained).
 * The topology's free set and row list are not used.  Kernels on `device` (fk_topology_analyze_kernel): one warp per
 * sketch with the matrix in shared memory where it fits (at most 200 KiB with the column order and the flags); otherwise
 * the matrix in global memory, one CTA per sketch when the batch fills the device and a cooperative group of CTAs per
 * sketch below that.  Limit: n_vars <= 26,624 (the row being reduced is held in shared memory) and one sketch's
 * min(n_expr, n_vars) x n_vars matrix within the 4 GiB workspace of a (topology, device), which a large sketch shares
 * with fewer sketches in flight.  Above it, FK_ERR_TOO_LARGE with the sizes in fk_last_error(), before any allocation. */
FK_API int fk_batch_analyze(const fk_topology* topo, int device, uint32_t n, const double* vars, const double* param,
                            uint8_t* independent);
/* Which kernel fk_batch_analyze launches for n_sketches sketches of this topology on the current device: 0 one warp per
 * sketch, 1 one CTA per sketch, 2 groups of CTAs per sketch; negative on error (FK_ERR_TOO_LARGE above the limit of
 * fk_batch_analyze).  Environment FK_ANALYZE_KERNEL=warp|cta|group forces one wherever it can take the shape (tests,
 * A/B measurements); a forced warp kernel on a matrix it cannot hold is FK_ERR_TOO_LARGE. */
FK_API int fk_topology_analyze_kernel(const fk_topology* topo, uint32_t n_sketches);

/* ---- fiksi::System mirror (host side above the solve boundary) ------------------------------- */
/* Same operations, argument meaning and ordering rules as fiksi::System (fiksi/src/lib.rs:252-467):
 * elements and constraints are created in order and get consecutive ids; lines and circles are
 * flattened to their points / lengths at creation (constraints/mod.rs:481-487); connected
 * components are maintained incrementally exactly as fiksi/src/graph.rs:178-225 does (including
 * its stale-index behaviour); fk_system_solve == System::solve(SolvingOptions { optimizer:
 * LevenbergMarquardt, decomposer: None, perturb }) with the scale, seeded perturbation and
 * write-back of fiksi/src/assemble/mod.rs:32-167.  All components go to the GPU in one
 * fk_lm_solve_batch call.  Functions returning an id return UINT32_MAX on invalid arguments. */
typedef struct fk_system fk_system;
typedef enum fk_constraint_tag { /* ConstraintTag order, fiksi/src/constraints/mod.rs:893-905 */
    FK_C_POINT_POINT_COINCIDENCE = 0,       /* elements: point, point */
    FK_C_POINT_POINT_DISTANCE = 1,          /* point, point; param = distance */
    FK_C_POINT_POINT_POINT_ANGLE = 2,       /* point, point, point; param = angle (radians) */
    FK_C_POINT_LINE_INCIDENCE = 3,          /* point, line */
    FK_C_POINT_LINE_DISTANCE = 4,           /* point, line; param = signed distance */
    FK_C_POINT_CIRCLE_INCIDENCE = 5,        /* point, circle */
    FK_C_SEGMENT_SEGMENT_LENGTH_EQUALITY = 6, /* point, point, point, point */
    FK_C_LINE_LINE_ANGLE = 7,               /* line, line; param = angle */
    FK_C_LINE_LINE_PARALLELISM = 8,         /* line, line */
    FK_C_LINE_LINE_PERPENDICULARITY = 9,    /* line, line */
    FK_C_LINE_CIRCLE_TANGENCY = 10          /* line, circle */
} fk_constraint_tag;

FK_API int fk_system_create(fk_system** out);
FK_API void fk_system_destroy(fk_system* s);
FK_API uint32_t fk_system_add_length(fk_system* s, double length);               /* elements::Length::create */
FK_API uint32_t fk_system_add_point(fk_system* s, double x, double y);           /* elements::Point::create */
FK_API uint32_t fk_system_add_line(fk_system* s, uint32_t p1, uint32_t p2);      /* elements::Line::create */
FK_API uint32_t fk_system_add_circle(fk_system* s, uint32_t center, uint32_t radius);
FK_API int fk_system_fix(fk_system* s, uint32_t element, int fix);               /* ElementHandle::fix / unfix */
FK_API uint32_t fk_system_add_constraint(fk_system* s, int tag, const uint32_t* elements,
                                         uint32_t n_elements, double param);
FK_API uint32_t fk_system_num_variables(const fk_system* s);
FK_API uint32_t fk_system_num_constraints(const fk_system* s);
FK_API uint32_t fk_system_element_variable(const fk_system* s, uint32_t element); /* first variable index */
FK_API int fk_system_get_variables(const fk_system* s, double* out);
FK_API int fk_system_set_variable(fk_system* s, uint32_t var, double value);     /* update_value */
FK_API int fk_system_set_parameter(fk_system* s, uint32_t constraint, double value); /* update_parameter */
FK_API int fk_system_solve(fk_system* s, int perturb, fk_report* reports, uint32_t cap, uint32_t* n_solved);
/* == System::solve(SolvingOptions { optimizer: LevenbergMarquardt, decomposer, perturb }), lib.rs:205-237.
 * decomposer 0: Decomposer::None (== fk_system_solve); 1: Decomposer::SinglePass (assemble/mod.rs:169-210;
 * maximum matching + strongly connected expression sets of analyze/graph/equations.rs on the host, every
 * set solved by the GPU LM in sequence); 2: Decomposer::RecursiveAssembly (assemble/mod.rs:212-277: the
 * recombination plan of analyze/graph/recursive_assembly.rs on the host -- hash-set iteration orders, which the
 * reference leaves to its hasher's seed, taken in ascending id order --, every step a `ClusteredSystem`
 * (assemble/mod.rs:282-590: cluster poses + the step's elements, FK_POSE_POINT_X/Y rows) solved by the GPU LM,
 * owned points moved with their cluster's pose afterwards).  reports: one per solved sub-problem, up to `cap`. */
FK_API int fk_system_solve_opts(fk_system* s, int decomposer, int perturb, fk_report* reports, uint32_t cap, uint32_t* n_solved);
/* SolvingOptions (lib.rs:205-237).  optimizer 0: LevenbergMarquardt, 1: LBfgs; decomposer as fk_system_solve_opts;
 * perturb 0 / 1; pad must be 0. */
typedef struct fk_solving_options {
    uint32_t optimizer, decomposer, perturb, pad;
} fk_solving_options;
/* == System::solve(options).  optimizer 0 is fk_system_solve_opts(decomposer).  optimizer 1 with Decomposer::None: the
 * scale, seeded perturbation and per-component problems of fk_system_solve, every component solved by L-BFGS in one
 * fk_lbfgs_solve_batch call, write-back as assemble/mod.rs:161-166; reports as fk_batch_solve_lbfgs.  The reference
 * dispatches on the optimizer only under Decomposer::None (assemble/mod.rs:148-158): SinglePass and RecursiveAssembly
 * call levenberg_marquardt directly (:191, :224), so optimizer 1 with decomposer 1 or 2 runs LM, identically to
 * optimizer 0.  Any other value: FK_ERR_INVALID. */
FK_API int fk_system_solve_options(fk_system* s, const fk_solving_options* opts, fk_report* reports, uint32_t cap, uint32_t* n_solved);
/* == System::solve(options) (lib.rs:464, assemble/mod.rs:46-167) applied to n variants of the drawing `s`: variant v is `s`
 * with every variable set to vars[v][i] (fk_system_set_variable) and every constraint parameter set to params[v][c]
 * (fk_system_set_parameter), then solved.  vars == NULL: every variant starts from s's variables; params == NULL: from s's
 * parameters.  vars_out[n][n_vars] receives what fk_system_get_variables would return after that solve, bit for bit what
 * fk_system_solve_options gives on a copy of `s` with the variant's numbers (LM on the global sparse path: the decisions of
 * that call, coordinates within the documented difference between the sparse batch kernel and the single-system path).
 * reports[v][k] (row stride reports_per_variant, may be NULL): the report of the k-th solved component (component order, as
 * fk_system_solve), the first reports_per_variant of them; *n_solved = solved components per variant (the same for every
 * variant).  Only Decomposer::None: opts->decomposer != 0 is FK_ERR_INVALID.  Variants are sharded over n_gpus devices
 * (0 == all visible) as fk_batch_solve does.  `s` is not modified.
 * On the device: one kernel scales, perturbs and gathers every component's input rows straight into the batch buffers of its
 * structure (components of identical shape share one topology: sketch = variant * multiplicity + member), one batched launch
 * per structure (the kernels of fk_batch_solve / fk_lbfgs_solve_batch), one kernel writes the unscaled rows back.  The plan
 * (components, structures, their topologies and device tables) is kept on `s` until a structural edit (an add_*, fix / unfix).
 * Variants go in chunks whose device buffers stay within about 1 GiB (at least one variant per chunk).  Refusals come before
 * any device work and leave vars_out untouched: FK_ERR_INVALID for bad arguments, FK_ERR_TOO_LARGE with LM when a
 * component's largest supernodal front exceeds the 236 rows of fk_batch_solve (the message names the component and the
 * front's order; L-BFGS takes every size). */
FK_API int fk_system_batch_solve(const fk_system* s, const fk_solving_options* opts, uint32_t n, const double* vars,
                                 const double* params, double* vars_out, fk_report* reports, uint32_t reports_per_variant,
                                 uint32_t* n_solved, int n_gpus);
/* Host-only probe of fk_system_batch_solve's plan (no device needed): solved components, distinct component structures,
 * and the components per structure in order of first appearance (multiplicity[n_structures], may be NULL). */
FK_API int fk_system_batch_layout(const fk_system* s, uint32_t* n_components, uint32_t* n_structures, uint32_t* multiplicity);
/* == System::solve(*opts) (lib.rs:464, assemble/mod.rs:46-167) on each of n different drawings, in one call.  systems[i] is
 * solved in place exactly as fk_system_solve_options(systems[i], opts, ...) would solve it: after the call it holds bit for bit
 * what that call gives on an identically built copy, and so do its reports -- for both optimizers, with and without
 * perturbation, fixed variables, stale-index components (SURVEY F7), empty drawings and NaN / inf inputs (which stay inside
 * their own drawing).  One exception: an LM component on the global sparse path runs the sparse batch kernel, with the
 * decisions, traces and counters of that call and coordinates within the 1e-11 relative difference of fk_system_batch_solve.
 * reports: the solved components of systems[0] in component order, then those of systems[1], ...; at most reports_cap are
 * written.  n_solved[i] (may be NULL) = components solved in systems[i].
 * Only Decomposer::None.  Refusals come before any device work and modify no system: FK_ERR_INVALID for null `systems` or
 * `opts`, a null entry, the same fk_system twice (the results would depend on the order), opts->decomposer != 0 or other bad
 * options; FK_ERR_TOO_LARGE with LM when a component's largest supernodal front exceeds the 236 rows of fk_batch_solve (the
 * message names the drawing's index, the component and the front's order).  n == 0 returns FK_OK.  All or nothing: the systems
 * are written only after every chunk on every device has succeeded, so a device error leaves every system as it was.
 * Each drawing's plan is fk_system_batch_solve's, kept on the system until a structural edit.  Per call, the structures of
 * all drawings are merged (same structure, whatever the drawing) and each goes to one launch kind: under LM, fk_lm_solve_batch's
 * rule (path 0 with fewer than 64 instances, 32-lane tables and at most 48 KiB of state: the one heterogeneous launch of the
 * chunk), the uniform batch kernels for the other path-0 / 1 structures, the sparse batch kernel on path 2; under L-BFGS one
 * uniform launch per structure.  On the device, per chunk of drawings on one stream per device: one copy up of the drawings'
 * raw rows and the call's tables, one kernel computes every drawing's scale and gathers every component's input rows, the
 * solve launches, one kernel writes the unscaled rows and the reports, one copy down.  Drawings go in order in chunks of about
 * 1 GiB of device buffers (FK_SYSTEM_BATCH_CHUNK caps the drawings per chunk), sharded by count over n_gpus devices (0 == all
 * visible). */
FK_API int fk_systems_solve(uint32_t n, fk_system* const* systems, const fk_solving_options* opts, fk_report* reports,
                            uint32_t reports_cap, uint32_t* n_solved, int n_gpus);
/* Host-only probe of fk_systems_solve's plan (no device needed): total solved components, distinct structures across the
 * drawings, and per structure (order of first appearance) its instance count and launch kind (0 heterogeneous, 1 uniform
 * batch, 2 sparse batch).  instances[n_structures] and launch_kind[n_structures] may be NULL; refusals as fk_systems_solve's
 * FK_ERR_INVALID. */
FK_API int fk_systems_layout(uint32_t n, fk_system* const* systems, const fk_solving_options* opts, uint32_t* n_components,
                             uint32_t* n_structures, uint32_t* instances, uint32_t* launch_kind);
/* == System::solve(SolvingOptions { decomposer: SinglePass, perturb }) (assemble/mod.rs:169-210; the reference runs LM here
 * whatever the optimizer, :191) applied to n variants of `s`; argument meaning as fk_system_batch_solve.  vars_out[v] and
 * reports[v] are bit for bit what fk_system_solve_opts(decomposer = 1, perturb) gives on a copy of `s` with the variant's
 * numbers (a set on the global sparse path runs the sparse batch kernel: the decisions of that call, coordinates within the
 * documented difference).  reports[v][k]: the k-th solved set in the order fk_system_solve_opts(decomposer = 1) reports them,
 * the first reports_per_variant of them; *n_solved = sets per variant.  `s` is not modified.
 * The plan is kept on `s` until a structural edit, like fk_system_batch_solve's: the strongly connected sets, grouped by
 * structure through the topology cache, and their waves.  A set's wave is one more than the latest wave of the sets it must
 * follow in the host loop's order (one writes what the other reads or writes, or reads what it writes), directly or through
 * a component's perturbation; a perturbation runs in the prepare kernel, or at the start of the wave after the last set that
 * reads its component's variables before it.  On the device, per chunk of variants: one prepare kernel (scale, resident scaled
 * rows), then per wave one gather / scatter kernel and one batched LM launch per structure present in the wave, and a last
 * gather / scatter kernel that writes the unscaled rows.  perturb 0 or 1; refusals come before any device work and leave
 * vars_out untouched: FK_ERR_INVALID for bad arguments, FK_ERR_TOO_LARGE when a set on the global sparse path has a largest
 * supernodal front above the 236 rows of fk_batch_solve (the message names the set, its first expression and the front).
 * Variants are chunked (about 1 GiB of device buffers, FK_SYSTEM_BATCH_CHUNK overrides) and sharded over n_gpus devices. */
FK_API int fk_system_batch_solve_single_pass(const fk_system* s, int perturb, uint32_t n, const double* vars, const double* params,
                                             double* vars_out, fk_report* reports, uint32_t reports_per_variant,
                                             uint32_t* n_solved, int n_gpus);
/* Host-only probe of its plan (no device needed): sets, waves, distinct set structures, and per set its wave and structure
 * (structures in order of first appearance; step_wave[n_steps] and step_structure[n_steps] may be NULL). */
FK_API int fk_system_single_pass_batch_layout(const fk_system* s, uint32_t* n_steps, uint32_t* n_waves, uint32_t* n_structures,
                                              uint32_t* step_wave, uint32_t* step_structure);
/* == System::solve(SolvingOptions { decomposer: RecursiveAssembly, perturb }) (assemble/mod.rs:212-277; the reference runs LM
 * here whatever the optimizer, :224) applied to n variants of `s`; arguments as fk_system_batch_solve_single_pass.
 * reports[v][k]: step k in the order fk_system_solve_opts(decomposer = 2) reports them (components in order, then the steps
 * of each component's plan), the first reports_per_variant of them; *n_solved = steps per variant.  vars_out[v][i] is
 * scale * the solved value for a variable some step writes (a variable of the step's elements, or a point a moved cluster
 * owns), and the raw input for every other variable, even where the call perturbed it.  `s` is not modified.
 * The plan is kept on `s` until a structural edit (add_*, fix / unfix): the recombination steps of every component, each
 * as its clustered problem (pose columns, element variables, the fixed point copies behind them) grouped by structure
 * through the topology cache, the points each step moves in the host loop's order, and the waves of
 * fk_system_batch_solve_single_pass's rule (a step reads its variables and the points it moves, and writes its element
 * variables and the points it moves).  On the device, per chunk of variants: one prepare kernel, then per wave one gather /
 * scatter kernel (previous wave's solutions, its moves, its reports, perturbations, this wave's input rows with every pose at
 * the identity) and one batched LM launch per structure present, and a last gather / scatter kernel with the write-back.
 * Numerical contract: each step's LM runs the kernels of the host loop, so a drawing whose plan moves no point gives bit
 * for bit what fk_system_solve_opts(decomposer = 2, perturb) gives on a copy of `s` with the variant's numbers.  A move is
 * Pose2D::transform_point with CUDA's sincos on the device and glibc's sin / cos in the host loop, which may differ in
 * the last place: with moves, every step's exit, iterations, factorisations and trace agree, and coordinates agree within
 * 1e-11 relative to the variant's largest |value| unless a step's decisions flip on that last place.  perturb 0 or 1;
 * refusals come before any device work and leave vars_out untouched: FK_ERR_INVALID for bad arguments, for a system the
 * reference panics on and for an expression that reads a variable outside its step (the host loop's messages),
 * FK_ERR_TOO_LARGE when a step on the global sparse path has a largest supernodal front above the 236 rows of
 * fk_batch_solve (the message names the step, its first constraint and the front).  Chunks and devices as
 * fk_system_batch_solve_single_pass. */
FK_API int fk_system_batch_solve_recursive_assembly(const fk_system* s, int perturb, uint32_t n, const double* vars,
                                                    const double* params, double* vars_out, fk_report* reports,
                                                    uint32_t reports_per_variant, uint32_t* n_solved, int n_gpus);
/* Host-only probe of its plan (no device needed): steps, waves, distinct step structures, and per step its wave and
 * structure (structures in order of first appearance; step_wave[n_steps] and step_structure[n_steps] may be NULL). */
FK_API int fk_system_recursive_assembly_batch_layout(const fk_system* s, uint32_t* n_steps, uint32_t* n_waves,
                                                     uint32_t* n_structures, uint32_t* step_wave, uint32_t* step_structure);
/* Host-only probe of the RecursiveAssembly plan (no device needed) as a stream of 32-bit words: per step
 * n_constraints, constraints..., n_elements, elements..., n_free, free elements..., then the maps on_frontiers,
 * owned_elements, frontier_elements (recursive_assembly.rs:75-114) as n_keys and per key (ascending) key, n,
 * values....  *n_words = length of the stream (at most `cap` words are written), *n_steps = steps. */
FK_API int fk_system_recursive_assembly_plan(const fk_system* s, uint32_t* out, uint32_t cap, uint32_t* n_words, uint32_t* n_steps);
/* Host-only probe of the SinglePass plan (no device needed): call with NULL arrays for
 * sizes3 = {steps, total free variables, total expressions}; then free_ptr[steps+1], free_vars (ascending
 * per step), expr_ptr[steps+1], exprs (row order per step). */
FK_API int fk_system_single_pass_plan(const fk_system* s, uint32_t* sizes3, uint32_t* free_ptr, uint32_t* free_vars,
                                      uint32_t* expr_ptr, uint32_t* exprs);
FK_API int fk_system_residuals(fk_system* s, double* out /* [num_constraints] */); /* calculate_residual */
/* == System::analyze (lib.rs:454-458): ids of the constraints that own a dependent expression, in
 * expression order, up to `cap`; *n_found receives their number.  All variables and expressions of the system go
 * through fk_batch_analyze as one sketch on device 0 (a group of CTAs once its matrix leaves shared memory), under
 * the same size limit. */
FK_API int fk_system_analyze(fk_system* s, uint32_t* constraints, uint32_t cap, uint32_t* n_found);
/* == System::analyze on n variants of `s` (variant v: every variable set to vars[v][i], every constraint parameter to
 * params[v][c]; NULL = s's own values, as fk_system_batch_solve).  dependent[v][c] = number of constraint c's expressions
 * the elimination found dependent (0 up to its expression count).  A constraint's expressions are consecutive and
 * expression ids ascend with constraint ids, so the list fk_system_analyze returns for variant v is every c
 * ascending, repeated dependent[v][c] times.
 * Bit for bit per variant: dependent[v] gives exactly that list on a copy of `s` with the variant's numbers, quirks
 * included (rows beyond min(n_expressions, n_variables) are never examined and count as dependent; every variable is a
 * column, fixed or not).  All three analyze kernels repeat the reference's floating-point operations, so the flags do not
 * depend on which one runs.  `s` is not modified; NaN and inf stay inside their own variant.
 * The plan (expression kinds, slot tables, the constraints' expression ranges; per device those tables and a grow-only
 * workspace within the 4 GiB of fk_batch_analyze) is built on first use and kept until a structural edit (add_*, fix /
 * unfix); new variable or parameter values keep it, and the NULL rows are s's values at call time.  No topology is built.
 * On the device, per chunk of variants on one stream per device: upload (or broadcast s's rows), one kernel expands the
 * parameters per expression, the analyze kernel choose_analyze picks for the chunk's size (FK_ANALYZE_KERNEL honoured), one
 * kernel counts each constraint's dependent expressions, download.  Chunks keep their buffers within about 1 GiB
 * (FK_SYSTEM_BATCH_CHUNK overrides); variants are sharded over n_gpus devices (0 == all visible).
 * Refusals come before any device work and leave `dependent` untouched: FK_ERR_INVALID for a null `s` or a null output with
 * n > 0, FK_ERR_TOO_LARGE with choose_analyze's message for a drawing beyond the analyze limit (n_variables > 26,624, or one
 * sketch's matrix beyond the 4 GiB workspace).  n = 0 and a drawing without constraints return FK_OK. */
FK_API int fk_system_batch_analyze(const fk_system* s, uint32_t n, const double* vars, const double* params,
                                   uint8_t* dependent /* [n][n_constraints] */, int n_gpus);
/* == calculate_residual of every constraint for n variants: out[v][c] is what fk_system_residuals writes on a copy of s
 * with the variant's numbers (unscaled; 2-norm of the two equalities of a coincidence), bit for bit on both of its paths
 * (the batch plan's K2 evaluation and fk_topology_eval on the global sparse path: both evaluate with the same device
 * formulas).  Arguments, plan, chunks, devices and FK_ERR_INVALID as fk_system_batch_analyze; one kernel evaluates every
 * constraint of every variant from the plan's slot tables (q += r * r in expression order, then sqrt, as
 * fk_system_residuals combines a coincidence).  Every drawing size is taken: no topology, batch plan or front limit. */
FK_API int fk_system_batch_residuals(const fk_system* s, uint32_t n, const double* vars, const double* params,
                                     double* out /* [n][n_constraints] */, int n_gpus);
/* == System::analyze on each of n different drawings in one call.  dependent[]: the constraints of systems[0] in constraint
 * order, then those of systems[1], ... (sum of fk_system_num_constraints entries); entry = how many of that constraint's
 * expressions were found dependent.  For drawing i, every constraint c ascending, repeated its entry times, is exactly the
 * list fk_system_analyze(systems[i]) returns: bit for bit, quirks included (rows beyond min(n_expressions, n_variables) are
 * never examined and count as dependent; every variable is a column, fixed or not).  NaN and inf stay inside their own
 * drawing.  No system is modified, so the same system may appear more than once.
 * Each drawing keeps fk_system_batch_analyze's plan.  Per call, drawings with equal plans (variables, expression kinds, slot
 * tables, constraint ranges: fixing an element changes none of them) are one structure.  A structure of fewer than 64
 * drawings whose matrix fits one warp (200 KiB of shared memory) joins the heterogeneous warp launch of its chunk (one warp per
 * drawing, one launch per footprint class: the warp's bytes rounded up to a power of two); any other gets one launch of the
 * kernel choose_analyze picks for its drawings in the chunk (FK_ANALYZE_KERNEL honoured: cta or group sends every structure
 * there).  On the device, per chunk of
 * drawings on one stream per device: one copy up of the descriptors, tables and rows, the analyze launches, one kernel counts
 * each constraint's dependent expressions, one copy down.  Drawings go in order in chunks of about 1 GiB of device buffers
 * (FK_SYSTEM_BATCH_CHUNK caps the drawings per chunk), sharded by count over n_gpus devices (0 == all visible).
 * Refusals come before any device work and leave `dependent` untouched: FK_ERR_INVALID for null `systems` with n > 0, a null
 * entry (the message names its index), a null `dependent` with a non-empty total, or `cap` below the total (the message names
 * it); FK_ERR_TOO_LARGE for a drawing beyond choose_analyze's limit, with "drawing i: " and choose_analyze's message.  n == 0
 * and drawings without constraints return FK_OK. */
FK_API int fk_systems_analyze(uint32_t n, const fk_system* const* systems, uint8_t* dependent, uint64_t cap, int n_gpus);
/* == calculate_residual of every constraint of each of n different drawings in one call, in fk_systems_analyze's ragged
 * layout: out[] holds bit for bit what fk_system_residuals(systems[i]) writes, on both of its paths.  Plan, chunks, devices,
 * no modification and FK_ERR_INVALID as fk_systems_analyze; one kernel evaluates every constraint of the chunk (q += r * r in
 * expression order, then sqrt, as fk_system_batch_residuals).  Every drawing size is taken. */
FK_API int fk_systems_residuals(uint32_t n, const fk_system* const* systems, double* out, uint64_t cap, int n_gpus);
/* Host-only probe of fk_systems_analyze's plan (no device needed): distinct analyze structures across the drawings, and per
 * structure (order of first appearance) its instance count and launch kind (0 heterogeneous warp launch, 1 one launch of the
 * kernel choose_analyze picks).  instances[n_structures] and launch_kind[n_structures] may be NULL; refusals as
 * fk_systems_analyze's for null systems. */
FK_API int fk_systems_analyze_layout(uint32_t n, const fk_system* const* systems, uint32_t* n_structures, uint32_t* instances,
                                     uint32_t* launch_kind);
FK_API uint32_t fk_system_num_components(const fk_system* s);
FK_API int fk_system_component(const fk_system* s, uint32_t index, uint32_t* n_elements, uint32_t* elements,
                               uint32_t* n_constraints, uint32_t* constraints);

#ifdef __cplusplus
}
#endif
#endif /* FIKSI_B200_H */
