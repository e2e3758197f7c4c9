// fk_system_batch_solve: System::solve over n variants of one drawing, every component solved in batches on the device.
// system.cpp describes the drawing (SystemBatchLayout), capi.cu groups its components by structure and runs the chunks,
// system_batch.cu holds the prepare / gather and scatter kernels.  fk_system_batch_solve_single_pass (Decomposer::SinglePass)
// shares the layout, the prepare kernel and the structure grouping, and adds the waves of strongly connected sets;
// fk_system_batch_solve_recursive_assembly (Decomposer::RecursiveAssembly) runs on the same waves with the recombination steps
// in place of the sets, plus the owned-point moves that follow each step.
#pragma once
#include <cstdint>
#include <memory>
#include <string>
#include <vector>

#include "../../include/fiksi_b200.h"

namespace fk {

constexpr uint32_t kSbNone = 0xFFFFFFFFu;

// The drawing as System::solve sees it, values aside (those come with every call).
struct SystemBatchLayout {
    uint32_t n_vars = 0, n_constraints = 0;
    std::vector<uint8_t> kind;              // [n_expr] expression kinds of the system
    std::vector<uint32_t> expr_constraint;  // [n_expr] constraint whose parameter the expression holds, kSbNone for none
    std::vector<double> draws;              // the solve's generator (seed 42): two draws per free variable, component order
    struct Component {                      // one per non-empty component, in component order
        std::vector<uint32_t> slot_var;     // local variable -> system variable (LocalProblem numbering)
        std::vector<uint32_t> slot_draw;    // local variable -> draw pair already applied at the component's snapshot, or kSbNone
        std::vector<uint32_t> expr;         // local expression -> system expression
        std::vector<uint32_t> free_var;     // local free column -> system variable
        // Decomposer::RecursiveAssembly: pairs (first variable of a point the step's cluster moves, the cluster's first pose
        // column) in the host loop's order.  A pose column has slot_var and free_var kSbNone (gathered as 0.0, never
        // scattered), a pose row expr kSbNone (parameter 0.0).
        std::vector<uint32_t> moves;
    };
    std::vector<Component> comps;
    // Decomposer::SinglePass (fk_system_batch_solve_single_pass): comps are the strongly connected sets in the order of the host
    // loop (slot_draw unused), comp_wave their waves.  Per system variable: var_draw, the draw pair of its component's
    // perturbation, and var_wave, the wave at whose start that perturbation runs (0: in the prepare kernel); kSbNone for a
    // variable of no non-empty component's free set.
    std::vector<uint32_t> comp_wave, var_draw, var_wave;
    uint32_t n_waves = 0;
    // Decomposer::RecursiveAssembly: comps are the steps, step_constraint[k] the first constraint of step k (refusals name it).
    std::vector<uint32_t> step_constraint;
};

// Device descriptor of one structure (components of identical shape) for the two kernels: its batch buffers hold sketch
// variant * mult + member.
struct SbStructure {
    double* vars;                  // [sketches][nv]
    double* params;                // [sketches][ne]
    const double* out;             // [sketches][nf]
    const fk_report* reps;         // [sketches]
    const uint32_t* slot_var;      // [mult][nv]
    const uint32_t* slot_draw;     // [mult][nv]
    const uint32_t* expr;          // [mult][ne]
    uint32_t nv, ne, nf, mult;
};

// Per variant: the scale over raw_vars[v] (stride 0: one row for all) and the parameters (raw_param[v][constraint] where
// the expression holds a constraint's parameter and raw_param is given, tmpl_param otherwise), then every structure's input
// rows; scales[v].  perturb 0: no draws applied.
int launch_system_batch_prepare(uint32_t n, uint32_t n_vars, uint32_t n_expr, uint32_t n_constraints, const uint8_t* kinds,
                                const uint32_t* expr_constraint, const double* draws, int perturb, const double* raw_vars,
                                uint32_t raw_vars_stride, const double* raw_param, const double* tmpl_param, uint32_t n_structures,
                                const SbStructure* structures, double* scales, void* stream);
// vars_out[v][i] = raw_vars[v][i], or scales[v] * x for a solved free variable (var_struct[i] != kSbNone: structure, var_off[i]:
// offset in the variant's block of that structure's free values); reports_out[v][k] = the report of component k
// (comp_struct[k], comp_member[k]) for k < n_reports.
int launch_system_batch_scatter(uint32_t n, uint32_t n_vars, const double* raw_vars, uint32_t raw_vars_stride, const double* scales,
                                const uint32_t* var_struct, const uint32_t* var_off, uint32_t n_reports, const uint32_t* comp_struct,
                                const uint32_t* comp_member, const SbStructure* structures, double* vars_out, fk_report* reports_out,
                                void* stream);

// fk_system_batch_solve_single_pass: the sets of one structure inside one wave.  s.vars / s.params / s.out / s.reps are the
// structure's batch buffers (sketch = variant * mult + member), s.slot_var [mult][nv] and s.expr [mult][ne] the members' rows
// (s.slot_draw unused; kSbNone gathers 0.0); free_var [mult][nf]: system variable of each solved column (kSbNone: not
// scattered); step [mult]: the member's set index.  fk_system_batch_solve_recursive_assembly: the members are steps and member
// m moves the points of moves[2k] (variable of x, y follows) with the pose in its solved columns moves[2k + 1] .. + 2, for
// move_off[m] <= k < move_off[m + 1] (all empty under SinglePass).
struct SpGroup {
    SbStructure s;
    const uint32_t* free_var;
    const uint32_t* step;
    const uint32_t* move_off;
    const uint32_t* moves;
};

// One launch between two waves of fk_system_batch_solve_single_pass / _recursive_assembly, per variant v < n on the resident
// rows vt[v][n_vars] (scaled variables) and pt[v][n_expr] (scaled parameters), in this order: the solved values of the
// `scatter` groups into vt; their owned-point moves (Pose2D::transform_point); their reports into reports_out[v][step]
// (step < n_reports); the perturbations perturb_var[k] with draw pair
// perturb_draw[k]; the input rows of the `gather` groups.  vars_out != null: then vars_out[v][i] = scales[v] * vt[v][i] for a
// variable some set solves (solved[i] != 0), raw_vars[v][i] otherwise.
int launch_system_sp_gather_scatter(uint32_t n, uint32_t n_vars, uint32_t n_expr, double* vt, const double* pt, uint32_t n_scatter,
                                    const SpGroup* scatter, uint32_t n_reports, fk_report* reports_out, uint32_t n_perturb,
                                    const uint32_t* perturb_var, const uint32_t* perturb_draw, const double* draws, uint32_t n_gather,
                                    const SpGroup* gather, const uint8_t* solved, const double* raw_vars, uint32_t raw_vars_stride,
                                    const double* scales, double* vars_out, void* stream);

// Host plan of a drawing (capi.cu): components grouped by structure through the topology cache, device state per device.
struct SystemBatch;
int system_batch_create(SystemBatchLayout&& layout, const std::vector<const fk_problem*>& problems, std::shared_ptr<SystemBatch>* out);
// (n_components, n_structures, multiplicity per structure in order of first appearance)
void system_batch_layout(const SystemBatch& b, uint32_t* n_components, uint32_t* n_structures, std::vector<uint32_t>* multiplicity);
struct SystemBatchCall {
    int optimizer = 0, perturb = 1, n_gpus = 1;
    uint32_t n = 0;
    const double* vars = nullptr;        // [n][n_vars] or null
    const double* params = nullptr;      // [n][n_constraints] or null
    const double* tmpl_vars = nullptr;   // [n_vars]
    const double* tmpl_param = nullptr;  // [n_expr]
    double* vars_out = nullptr;
    fk_report* reports = nullptr;
    uint32_t reports_per_variant = 0;
};
// Refusals (checked before any device work) and the solve.  Errors leave a message for fk_last_error().
int system_batch_solve(SystemBatch& b, const SystemBatchCall& call);

// The same for Decomposer::SinglePass: layout.comps are the sets (problems: one per set), grouped by structure; per wave one
// launch per structure present.  (call.optimizer is ignored: the reference runs LM under SinglePass.)  Decomposer::
// RecursiveAssembly uses the same plan and calls with layout.comps the steps (layout.step_constraint set, moves per step).
struct SystemSpBatch;
int system_sp_batch_create(SystemBatchLayout&& layout, const std::vector<const fk_problem*>& problems, std::shared_ptr<SystemSpBatch>* out);
// (n_sets, n_waves, n_structures, wave and structure of each set)
void system_sp_batch_layout(const SystemSpBatch& b, uint32_t* n_sets, uint32_t* n_waves, uint32_t* n_structures,
                            std::vector<uint32_t>* set_wave, std::vector<uint32_t>* set_structure);
int system_sp_batch_solve(SystemSpBatch& b, const SystemBatchCall& call);

// fk_system_batch_analyze / fk_system_batch_residuals: System::analyze and calculate_residual over n variants of one drawing.
// The drawing's expressions as analyze and the residuals read them; no topology, ordering or symbolic analysis.
struct SystemAnLayout {
    uint32_t n_vars = 0;
    std::vector<uint8_t> kind;              // [n_expr]
    std::vector<uint32_t> slot_var;         // [n_expr][8] expand_slots of every expression, as fk_batch_analyze builds it
    std::vector<uint32_t> expr_constraint;  // [n_expr] constraint whose parameter the expression holds, kSbNone for none
    std::vector<uint32_t> con_off;          // [n_constraints + 1] constraint c owns expressions [con_off[c], con_off[c + 1])
};
// pt[v][e] = variant_param(raw_param, ..., v, e) (prepare.cuh) for v < n; tmpl_vars != null: vt[v] = tmpl_vars too.
int launch_system_an_expand(uint32_t n, uint32_t n_vars, uint32_t n_expr, uint32_t n_constraints, const double* tmpl_vars, double* vt,
                            const uint32_t* expr_constraint, const double* raw_param, const double* tmpl_param, double* pt, void* stream);
// dependent[v][c] = number of expressions of constraint c with independent[v][e] == 0.
int launch_system_an_reduce(uint32_t n, uint32_t n_expr, uint32_t n_constraints, const uint8_t* independent, const uint32_t* con_off,
                            uint8_t* dependent, void* stream);
// out[v][c] = fk_system_residuals of variant v (rows vt[v][n_vars], pt[v][n_expr]).
int launch_system_residuals(uint32_t n, uint32_t n_vars, uint32_t n_expr, uint32_t n_constraints, const uint8_t* kinds, const uint32_t* slot_var,
                            const uint32_t* con_off, const double* vt, const double* pt, double* out, void* stream);
// fk_systems_analyze / fk_systems_residuals over the chunk's n drawings (SysAnJob, lm_kernels.cuh: its tables in `tabs`, its rows
// and flags), the chunk's constraints in drawing order: drawing d owns constraints [con_base[d], con_base[d + 1]), total =
// con_base[n].  dependent[i] = the dependent expressions of constraint i (zero flags); out[i] = its residual, as
// launch_system_residuals evaluates it.
struct SysAnJob;
int launch_systems_an_reduce(uint32_t n, uint64_t total, const uint64_t* con_base, const SysAnJob* drawings, const uint32_t* tabs,
                             const uint8_t* flags, uint8_t* dependent, void* stream);
int launch_systems_residuals(uint32_t n, uint64_t total, const uint64_t* con_base, const SysAnJob* drawings, const uint32_t* tabs,
                             const double* vars, const double* params, double* out, void* stream);
struct SystemAnBatch;
int system_an_batch_create(SystemAnLayout&& layout, std::shared_ptr<SystemAnBatch>* out);
struct SystemAnCall {
    int n_gpus = 1;
    uint32_t n = 0;
    const double* vars = nullptr;        // [n][n_vars] or null
    const double* params = nullptr;      // [n][n_constraints] or null
    const double* tmpl_vars = nullptr;   // [n_vars]
    const double* tmpl_param = nullptr;  // [n_expr]
    uint8_t* dependent = nullptr;        // fk_system_batch_analyze: [n][n_constraints]
    double* residuals = nullptr;         // fk_system_batch_residuals: [n][n_constraints] (exactly one of the two is set)
};
// Refusals (analyze: choose_analyze's size limit) before any device work, then the chunks on every device.
int system_an_batch_run(SystemAnBatch& b, const SystemAnCall& call);

// fk_systems_analyze / fk_systems_residuals: System::analyze and calculate_residual over n different drawings, each with its own
// SystemAnBatch plan.  capi.cu merges equal plans into structures, runs chunks of drawings and returns every drawing's counts or
// residuals (drawing after drawing, constraint order); system.cpp validates the call.
struct SystemsAnDrawing {
    const SystemAnBatch* plan;
    const double* vars;   // [plan n_vars]
    const double* param;  // [plan n_expr]
};
// Host-only: per distinct structure (order of first appearance) its instances and analyze launch kind (0 heterogeneous warp
// launch, 1 one launch of the kernel choose_analyze picks).
void systems_an_layout(const std::vector<SystemsAnDrawing>& d, std::vector<uint32_t>* instances, std::vector<uint32_t>* launch_kind);
// Exactly one of dependent / residuals is set, with room for every constraint of every drawing.  Refusals (analyze: a drawing
// beyond choose_analyze's limit) before any device work.
int systems_an_run(const std::vector<SystemsAnDrawing>& d, uint8_t* dependent, double* residuals, int n_gpus);

// fk_systems_solve: System::solve over n different drawings, each with its own SystemBatch plan (its components, grouped by
// structure inside the drawing).  capi.cu merges the structures of all drawings, runs chunks of drawings and returns every
// drawing's variables and reports; system.cpp validates the call and writes the results into the systems.
//
// One instance per solved component of a chunk's drawings, in drawing order and component order inside a drawing, so that the
// k-th instance's report is the k-th report of the chunk.  vars / params: where the prepare kernel writes its input rows (its
// structure's batch rows, or its heterogeneous job's rows); out / rep: its solution.  tab: offset in the chunk's u32 table of
// the component's slot_var[nv], slot_draw[nv], expr[ne] and free_var[nf] (SystemBatchLayout::Component).
struct SysInst {
    double* vars;
    double* params;
    const double* out;
    const fk_report* rep;
    uint64_t tab;
    uint32_t drawing;  // in the chunk
    uint32_t nv, ne, nf;
};
// Ragged rows of the chunk's n drawings: drawing d owns raw_vars[var_off[d] .. var_off[d + 1]) and raw_param / kinds
// [expr_off[d] .. expr_off[d + 1]) (s->vars, s->param, s->kind), and the instances [inst_off[d], inst_off[d + 1]).
// Per drawing: scales[d] = prepare_scale of its rows, then every instance's input rows (perturb 0: no draws applied; draws: the
// one table of the call, pair k is the same in every drawing).
int launch_systems_prepare(uint32_t n, const uint64_t* var_off, const uint64_t* expr_off, const uint32_t* inst_off, const uint8_t* kinds,
                           const double* raw_vars, const double* raw_param, const double* draws, int perturb, const SysInst* inst,
                           const uint32_t* tabs, double* scales, void* stream);
// vars_out[var_off[d] + i] = raw_vars[var_off[d] + i], then scales[d] * x for every solved free variable; reports_out[k] = the
// k-th instance's report.
int launch_systems_scatter(uint32_t n, const uint64_t* var_off, const uint32_t* inst_off, const double* raw_vars, const double* scales,
                           const SysInst* inst, const uint32_t* tabs, double* vars_out, fk_report* reports_out, void* stream);

struct SystemsDrawing {
    const SystemBatch* plan;
    const double* vars;   // [plan n_vars]
    const double* param;  // [plan n_expr]
};
// Host-only: solved components, distinct structures across the drawings (order of first appearance), per structure its
// instances and launch kind (0 heterogeneous, 1 uniform batch, 2 sparse batch) under `optimizer`.
void systems_layout(const std::vector<SystemsDrawing>& d, int optimizer, uint32_t* n_components, std::vector<uint32_t>* instances,
                    std::vector<uint32_t>* launch_kind);
// The solve: vars_out receives every drawing's variables after the solve (drawing after drawing), reports every solved
// component's report (drawing after drawing, component order).  Refusals before any device work; vars_out and reports are only
// complete when FK_OK is returned.
int systems_solve(const std::vector<SystemsDrawing>& d, int optimizer, int perturb, int n_gpus, double* vars_out, fk_report* reports);

// fk_last_error()'s message for errors found outside capi.cu.
int system_batch_fail(int code, const std::string& msg);

}  // namespace fk
