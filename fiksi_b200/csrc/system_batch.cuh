// fk_system_batch_solve: System::solve over n variants of one drawing, every component solved in batches on the device.
// system.cpp describes the drawing (SystemBatchLayout), capi.cu groups its components by structure and runs the chunks,
// system_batch.cu holds the prepare / gather and scatter kernels.
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
    };
    std::vector<Component> comps;
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
// fk_last_error()'s message for errors found outside capi.cu.
int system_batch_fail(int code, const std::string& msg);

}  // namespace fk
