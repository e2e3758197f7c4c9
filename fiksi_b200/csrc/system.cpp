// fk_system: the host-side mirror of fiksi::System (fiksi/src/lib.rs:252-467) above the solve
// boundary — element / constraint creation, the incidence graph with its incremental connected
// components, fix / unfix, and assemble::solve's scale, perturbation and write-back
// (fiksi/src/assemble/mod.rs:32-167).  All numerics (residuals, Jacobians, ordering,
// factorisation, LM) happen behind fk_lm_solve_batch / the evaluation kernels on the GPU.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <set>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/fiksi_b200.h"
#include "recursive_assembly.hpp"
#include "single_pass.hpp"
#include "symbolic.hpp"
#include "system_batch.cuh"

namespace {

enum ElemTag : uint8_t { kLength = 0, kPoint = 1, kLine = 2, kCircle = 3 };

struct Elem {
    uint8_t tag;
    uint32_t a, b;  // Length/Point: a = first variable; Line: a, b = point variables; Circle: a = centre var, b = radius var
};
struct Constr {
    uint8_t tag;         // ConstraintTag order (constraints/mod.rs:893-905)
    uint32_t first_expr; // index of its first expression
    uint8_t n_expr;      // valency: 2 for PointPointCoincidence, else 1 (constraints/mod.rs:992-1034)
    uint8_t n_inc;       // incident primitive elements (graph.rs:112-117), in the order the reference lists them
    uint32_t inc[4];
};

// Knuth/Lewis LCG of fiksi/src/rand.rs:24-39.
struct Lcg {
    uint32_t s;
    double next() {
        s = s * 1664525u + 1013904223u;
        return (1.0 / 4294967295.0) * (double)s;
    }
};

}  // namespace

struct fk_system {
    std::vector<Elem> elems;
    std::vector<double> vars;
    std::vector<uint32_t> var_owner;  // variable -> primitive element (lib.rs variable_to_primitive)
    std::vector<uint8_t> fixed;       // per variable
    std::vector<Constr> constrs;
    std::vector<uint8_t> kind;
    std::vector<uint32_t> idx;        // 4 per expression
    std::vector<double> param;
    // incidence graph: incremental connected components exactly as graph.rs:178-225 builds them —
    // only the elements incident to the new constraint are re-pointed on a merge, members of a
    // merged-away component keep their old (now empty) slot.
    std::vector<uint32_t> comp_of;    // per element, 0 = none, else 1-based slot
    struct Comp { std::set<uint32_t> elements, constraints; };
    std::vector<Comp> comps;
    std::string error;
    std::unique_ptr<fk_topology, void (*)(fk_topology*)> eval_topo{nullptr, fk_topology_destroy};
    // fk_system_batch_solve's plan (components grouped by structure, device tables): built on first use, dropped by every
    // structural edit (elements, constraints, fix / unfix); new variable or parameter values keep it.
    mutable std::mutex batch_mu;
    mutable std::shared_ptr<fk::SystemBatch> batch;
    mutable std::shared_ptr<fk::SystemSpBatch> sp_batch;  // fk_system_batch_solve_single_pass's plan, kept and dropped alike
    mutable std::shared_ptr<fk::SystemSpBatch> ra_batch;  // fk_system_batch_solve_recursive_assembly's plan, kept and dropped alike
    mutable std::shared_ptr<fk::SystemAnBatch> an_batch;  // fk_system_batch_analyze / _residuals' plan, kept and dropped alike

    uint32_t new_element(uint8_t tag, uint32_t a, uint32_t b, const double* v, int nv) {
        uint32_t id = (uint32_t)elems.size();
        uint32_t first = (uint32_t)vars.size();
        for (int k = 0; k < nv; k++) {
            vars.push_back(v[k]);
            var_owner.push_back(id);
            fixed.push_back(0);
        }
        elems.push_back({tag, nv ? first : a, b});
        comp_of.push_back(0);
        eval_topo.reset();
        drop_batch_plan();
        return id;
    }
    int element_vars(uint32_t e, uint32_t out[4]) const {
        const Elem& el = elems[e];
        switch (el.tag) {
            case kLength: out[0] = el.a; return 1;
            case kPoint: out[0] = el.a; out[1] = el.a + 1; return 2;
            case kLine: out[0] = el.a; out[1] = el.a + 1; out[2] = el.b; out[3] = el.b + 1; return 4;
            default: out[0] = el.a; out[1] = el.a + 1; out[2] = el.b; return 3;
        }
    }
    void connect(uint32_t constraint, const uint32_t* inc, int n) {
        uint32_t target = 0;
        size_t best = 0;
        for (int k = 0; k < n; k++) {
            uint32_t c = comp_of[inc[k]];
            if (c && comps[c - 1].elements.size() > best) {
                best = comps[c - 1].elements.size();
                target = c;
            }
        }
        if (!target) {
            comps.emplace_back();
            target = (uint32_t)comps.size();
        }
        Comp merged;
        merged.elements.swap(comps[target - 1].elements);
        merged.constraints.swap(comps[target - 1].constraints);
        for (int k = 0; k < n; k++) {
            uint32_t c = comp_of[inc[k]];
            if (c) {
                Comp& src = comps[c - 1];  // already emptied if it is the target (or a stale slot)
                merged.elements.insert(src.elements.begin(), src.elements.end());
                merged.constraints.insert(src.constraints.begin(), src.constraints.end());
                src.elements.clear();
                src.constraints.clear();
            } else {
                merged.elements.insert(inc[k]);
            }
            comp_of[inc[k]] = target;
        }
        merged.constraints.insert(constraint);
        comps[target - 1].elements.swap(merged.elements);
        comps[target - 1].constraints.swap(merged.constraints);
    }
    void drop_batch_plan() {
        std::lock_guard<std::mutex> lock(batch_mu);
        batch.reset();
        sp_batch.reset();
        ra_batch.reset();
        an_batch.reset();
    }
    void push_expr(uint8_t k, uint32_t i0, uint32_t i1, uint32_t i2, uint32_t i3, double p) {
        kind.push_back(k);
        idx.push_back(i0); idx.push_back(i1); idx.push_back(i2); idx.push_back(i3);
        param.push_back(p);
    }
};

extern "C" {

int fk_system_create(fk_system** out) {
    if (!out) return FK_ERR_INVALID;
    *out = new (std::nothrow) fk_system();
    return *out ? FK_OK : FK_ERR_OOM;
}
void fk_system_destroy(fk_system* s) { delete s; }

// elements/mod.rs:280-454
uint32_t fk_system_add_length(fk_system* s, double length) { return s->new_element(kLength, 0, 0, &length, 1); }
uint32_t fk_system_add_point(fk_system* s, double x, double y) {
    double v[2] = {x, y};
    return s->new_element(kPoint, 0, 0, v, 2);
}
uint32_t fk_system_add_line(fk_system* s, uint32_t p1, uint32_t p2) {
    if (p1 >= s->elems.size() || p2 >= s->elems.size() || s->elems[p1].tag != kPoint || s->elems[p2].tag != kPoint) return UINT32_MAX;
    return s->new_element(kLine, s->elems[p1].a, s->elems[p2].a, nullptr, 0);
}
uint32_t fk_system_add_circle(fk_system* s, uint32_t center, uint32_t radius) {
    if (center >= s->elems.size() || radius >= s->elems.size() || s->elems[center].tag != kPoint || s->elems[radius].tag != kLength) return UINT32_MAX;
    return s->new_element(kCircle, s->elems[center].a, s->elems[radius].a, nullptr, 0);
}

// elements/mod.rs:60-86
int fk_system_fix(fk_system* s, uint32_t element, int fix) {
    if (!s || element >= s->elems.size()) return FK_ERR_INVALID;
    uint32_t v[4];
    int n = s->element_vars(element, v);
    for (int k = 0; k < n; k++) s->fixed[v[k]] = fix ? 1 : 0;
    s->drop_batch_plan();
    return FK_OK;
}

// constraints/mod.rs:317-891.  `tag` in ConstraintTag order; `elements` are the handles the
// reference's constructor takes (e.g. {point, line} for PointLineIncidence).
uint32_t fk_system_add_constraint(fk_system* s, int tag, const uint32_t* el, uint32_t n_el, double p) {
    static const uint8_t want[11][4] = {
        {kPoint, kPoint, 255, 255}, {kPoint, kPoint, 255, 255}, {kPoint, kPoint, kPoint, 255}, {kPoint, kLine, 255, 255},
        {kPoint, kLine, 255, 255},  {kPoint, kCircle, 255, 255}, {kPoint, kPoint, kPoint, kPoint}, {kLine, kLine, 255, 255},
        {kLine, kLine, 255, 255},   {kLine, kLine, 255, 255},   {kLine, kCircle, 255, 255}};
    if (!s || tag < 0 || tag > 10 || !el) return UINT32_MAX;
    uint32_t need = 0;
    while (need < 4 && want[tag][need] != 255) need++;
    if (n_el != need) return UINT32_MAX;
    for (uint32_t k = 0; k < need; k++)
        if (el[k] >= s->elems.size() || s->elems[el[k]].tag != want[tag][k]) return UINT32_MAX;
    auto var = [&](uint32_t e) { return s->elems[e].a; };
    auto own = [&](uint32_t v) { return s->var_owner[v]; };
    const uint32_t id = (uint32_t)s->constrs.size();
    const uint32_t first = (uint32_t)s->kind.size();
    uint32_t inc[4];
    int n_inc = 0;
    uint8_t n_expr = 1;
    switch (tag) {
        case 0: {  // PointPointCoincidence: x and y equalities
            inc[0] = el[0]; inc[1] = el[1]; n_inc = 2; n_expr = 2;
            s->push_expr(FK_VARIABLE_VARIABLE_EQUALITY, var(el[0]), var(el[1]), 0, 0, 0.0);
            s->push_expr(FK_VARIABLE_VARIABLE_EQUALITY, var(el[0]) + 1, var(el[1]) + 1, 0, 0, 0.0);
        } break;
        case 1:
            inc[0] = el[0]; inc[1] = el[1]; n_inc = 2;
            s->push_expr(FK_POINT_POINT_DISTANCE, var(el[0]), var(el[1]), 0, 0, p);
            break;
        case 2:
            inc[0] = el[0]; inc[1] = el[1]; inc[2] = el[2]; n_inc = 3;
            s->push_expr(FK_POINT_POINT_POINT_ANGLE, var(el[0]), var(el[1]), var(el[2]), 0, p);
            break;
        case 3: case 4: {
            const Elem& l = s->elems[el[1]];
            inc[0] = el[0]; inc[1] = own(l.a); inc[2] = own(l.b); n_inc = 3;
            s->push_expr(tag == 3 ? FK_POINT_LINE_INCIDENCE : FK_POINT_LINE_DISTANCE, var(el[0]), l.a, l.b, 0, tag == 4 ? p : 0.0);
        } break;
        case 5: {
            const Elem& c = s->elems[el[1]];
            inc[0] = el[0]; inc[1] = own(c.a); inc[2] = own(c.b); n_inc = 3;
            s->push_expr(FK_POINT_CIRCLE_INCIDENCE, var(el[0]), c.a, c.b, 0, 0.0);
        } break;
        case 6:
            for (int k = 0; k < 4; k++) inc[k] = own(var(el[k]));
            n_inc = 4;
            s->push_expr(FK_SEGMENT_SEGMENT_LENGTH_EQUALITY, var(el[0]), var(el[1]), var(el[2]), var(el[3]), 0.0);
            break;
        case 7: case 8: case 9: {
            const Elem& l1 = s->elems[el[0]];
            const Elem& l2 = s->elems[el[1]];
            inc[0] = own(l1.a); inc[1] = own(l1.b); inc[2] = own(l2.a); inc[3] = own(l2.b); n_inc = 4;
            const uint8_t k = tag == 7 ? FK_LINE_LINE_ANGLE : (tag == 8 ? FK_LINE_LINE_PARALLELISM : FK_LINE_LINE_PERPENDICULARITY);
            s->push_expr(k, l1.a, l1.b, l2.a, l2.b, tag == 7 ? p : 0.0);
        } break;
        default: {  // 10 LineCircleTangency
            const Elem& l = s->elems[el[0]];
            const Elem& c = s->elems[el[1]];
            inc[0] = own(l.a); inc[1] = own(l.b); inc[2] = own(c.a); inc[3] = own(c.b); n_inc = 4;
            s->push_expr(FK_LINE_CIRCLE_TANGENCY, l.a, l.b, c.a, c.b, 0.0);
        } break;
    }
    s->connect(id, inc, n_inc);
    Constr rec{(uint8_t)tag, first, n_expr, (uint8_t)n_inc, {0, 0, 0, 0}};
    for (int k = 0; k < n_inc; k++) rec.inc[k] = inc[k];
    s->constrs.push_back(rec);
    s->eval_topo.reset();
    s->drop_batch_plan();
    return id;
}

uint32_t fk_system_num_variables(const fk_system* s) { return s ? (uint32_t)s->vars.size() : 0; }
uint32_t fk_system_num_constraints(const fk_system* s) { return s ? (uint32_t)s->constrs.size() : 0; }
uint32_t fk_system_element_variable(const fk_system* s, uint32_t e) { return (s && e < s->elems.size()) ? s->elems[e].a : UINT32_MAX; }
int fk_system_get_variables(const fk_system* s, double* out) {
    if (!s || !out) return FK_ERR_INVALID;
    std::memcpy(out, s->vars.data(), s->vars.size() * sizeof(double));
    return FK_OK;
}
// elements/mod.rs:558-579 (update_value) for any variable
int fk_system_set_variable(fk_system* s, uint32_t var, double value) {
    if (!s || var >= s->vars.size()) return FK_ERR_INVALID;
    s->vars[var] = value;
    return FK_OK;
}
// constraints/mod.rs:992-1046 (update_parameter)
int fk_system_set_parameter(fk_system* s, uint32_t constraint, double value) {
    if (!s || constraint >= s->constrs.size()) return FK_ERR_INVALID;
    s->param[s->constrs[constraint].first_expr] = value;
    return FK_OK;
}

}  // extern "C"

namespace {

// One compact fk_problem: `free_sorted` free, `exprs` as rows (in that order), every other referenced
// variable fixed at its current value in `vt`.  Referenced variables are renumbered ascending, so x/y of a point
// stay adjacent, and sub-problems of the same shape share one topology inside the batch calls.
struct LocalProblem {
    std::vector<double> vars, param, x;
    std::vector<uint8_t> kind;
    std::vector<uint32_t> idx, free_local, rows, free_global;
    std::vector<uint32_t> slot_global;  // local variable -> system variable
    fk_problem prob;
};
void build_local(const fk_system* s, const std::vector<double>& vt, const std::vector<double>& pt, const std::vector<uint32_t>& free_sorted,
                 const std::vector<uint32_t>& exprs, LocalProblem& L) {
    std::set<uint32_t> used(free_sorted.begin(), free_sorted.end());
    for (uint32_t e : exprs) {
        uint32_t sv[8];
        const int a = fk::expand_slots(s->kind[e], &s->idx[4 * (size_t)e], sv);
        for (int k = 0; k < a; k++) used.insert(sv[k]);
    }
    std::map<uint32_t, uint32_t> local;
    for (uint32_t g : used) {
        local.emplace(g, (uint32_t)L.vars.size());
        L.vars.push_back(vt[g]);
        L.slot_global.push_back(g);
    }
    for (uint32_t g : free_sorted) {
        L.free_global.push_back(g);
        L.free_local.push_back(local[g]);
        L.x.push_back(vt[g]);
    }
    static const int stored[FK_NUM_KINDS] = {2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 4, 3, 3};
    for (uint32_t e : exprs) {
        L.rows.push_back((uint32_t)L.kind.size());
        L.kind.push_back(s->kind[e]);
        L.param.push_back(pt[e]);
        for (int q = 0; q < 4; q++) L.idx.push_back(q < stored[s->kind[e]] ? local[s->idx[4 * (size_t)e + q]] : 0);
    }
    fk_problem& p = L.prob;
    p.n_vars = (uint32_t)L.vars.size(); p.vars = L.vars.data();
    p.n_expr = (uint32_t)L.kind.size(); p.kind = L.kind.data(); p.idx = L.idx.data(); p.param = L.param.data();
    p.n_free = (uint32_t)L.free_local.size(); p.free_vars = L.free_local.data();
    p.n_rows = (uint32_t)L.rows.size(); p.rows = L.rows.data();
}

struct PreparedSystem {
    double scale = 1.0;
    std::vector<std::unique_ptr<LocalProblem>> locals;  // one per non-empty component, in component order
};

// assemble/mod.rs:32-124: scale, seeded perturbation and the per-component problems.
void prepare_components(const fk_system* s, int perturb, PreparedSystem& out) {
    const size_t nv = s->vars.size();
    // assemble/mod.rs:32-44,58-79: RMS of all variables and of the distance parameters (sequential sums)
    double sum = 0.0;
    size_t cnt = 0;
    for (double v : s->vars) { sum += v * v; cnt++; }
    for (size_t e = 0; e < s->kind.size(); e++)
        if (s->kind[e] == FK_POINT_POINT_DISTANCE || s->kind[e] == FK_POINT_LINE_DISTANCE) { sum += s->param[e] * s->param[e]; cnt++; }
    const double scale = out.scale = std::sqrt(sum / (double)cnt);
    const double recip = 1.0 / scale;
    std::vector<double> vt(nv);
    for (size_t i = 0; i < nv; i++) vt[i] = s->vars[i] * recip;
    std::vector<double> pt(s->param);
    for (size_t e = 0; e < pt.size(); e++)
        if (s->kind[e] == FK_POINT_POINT_DISTANCE || s->kind[e] == FK_POINT_LINE_DISTANCE) pt[e] = recip * s->param[e];
    Lcg rng{42};  // assemble/mod.rs:47: one generator per solve, consumed by the components in order
    for (const fk_system::Comp& c : s->comps) {
        if (c.elements.empty()) continue;  // assemble/mod.rs:87-89
        std::set<uint32_t> free_set;
        for (uint32_t e : c.elements) {
            uint32_t v[4];
            int n = s->element_vars(e, v);
            for (int k = 0; k < n; k++)
                if (!s->fixed[v[k]]) free_set.insert(v[k]);
        }
        if (perturb) {  // assemble/mod.rs:113-124
            for (uint32_t fv : free_set) {
                const double r1 = rng.next();
                const double r2 = rng.next();
                vt[fv] += vt[fv] * (1.0 / 8196.0) * r1 + (1.0 / 65568.0) * r2;
            }
        }
        std::vector<uint32_t> exprs;
        for (uint32_t ci : c.constraints)
            for (uint8_t k = 0; k < s->constrs[ci].n_expr; k++) exprs.push_back(s->constrs[ci].first_expr + k);
        std::unique_ptr<LocalProblem> L(new LocalProblem());
        // (values as of now: later components have not been perturbed yet)
        build_local(s, vt, pt, std::vector<uint32_t>(free_set.begin(), free_set.end()), exprs, *L);
        out.locals.push_back(std::move(L));
    }
}

// == System::solve(SolvingOptions { optimizer, decomposer: None, perturb }) (lib.rs:464, assemble/mod.rs:46-167): every
// component in one batch call of the optimizer (0 LM, 1 L-BFGS, assemble/mod.rs:148-158).
int solve_components(fk_system* s, int optimizer, int perturb, fk_report* reports, uint32_t cap, uint32_t* n_solved) {
    if (n_solved) *n_solved = 0;
    PreparedSystem ps;
    prepare_components(s, perturb, ps);
    std::vector<std::unique_ptr<LocalProblem>>& locals = ps.locals;
    if (locals.empty()) return FK_OK;
    std::vector<const fk_problem*> probs;
    std::vector<double*> xs;
    for (auto& L : locals) {
        probs.push_back(&L->prob);
        xs.push_back(L->x.data());
    }
    std::vector<fk_report> reps(locals.size());
    const uint32_t n = (uint32_t)locals.size();
    int rc = optimizer == 1 ? fk_lbfgs_solve_batch(n, probs.data(), xs.data(), reps.data(), 1)
                            : fk_lm_solve_batch(n, probs.data(), xs.data(), reps.data(), 1);
    if (rc != FK_OK) return rc;
    // assemble/mod.rs:161-166
    for (auto& L : locals)
        for (size_t k = 0; k < L->free_global.size(); k++) s->vars[L->free_global[k]] = ps.scale * L->x[k];
    for (size_t k = 0; k < locals.size() && reports && k < cap; k++) reports[k] = reps[k];
    if (n_solved) *n_solved = n;
    return FK_OK;
}

}  // namespace

extern "C" {

// == System::solve(SolvingOptions { optimizer: LevenbergMarquardt, decomposer: None, perturb })
// (lib.rs:464, assemble/mod.rs:46-167).  reports: one per solved component in component order, up
// to `cap`; *n_solved receives the number of components solved.
int fk_system_solve(fk_system* s, int perturb, fk_report* reports, uint32_t cap, uint32_t* n_solved) {
    if (!s) return FK_ERR_INVALID;
    return solve_components(s, 0, perturb, reports, cap, n_solved);
}

// ---- Decomposer::SinglePass (SURVEY 8f-1) ------------------------------------------------------------
namespace {

// The equation graph of lib.rs:262,395,434.
void equation_graph(const fk_system* s, std::vector<std::vector<uint32_t>>& var_exprs, std::vector<std::vector<uint32_t>>& expr_vars) {
    var_exprs.assign(s->vars.size(), {});
    expr_vars.assign(s->kind.size(), {});
    for (uint32_t e = 0; e < s->kind.size(); e++) {
        uint32_t sv[8];
        const int a = fk::expand_slots(s->kind[e], &s->idx[4 * (size_t)e], sv);
        expr_vars[e].assign(sv, sv + a);
        for (int k = 0; k < a; k++) var_exprs[sv[k]].push_back(e);
    }
}

std::vector<uint32_t> component_free_variables(const fk_system* s, const fk_system::Comp& c) {
    std::set<uint32_t> free_set;
    for (uint32_t e : c.elements) {
        uint32_t v[4];
        const int n = s->element_vars(e, v);
        for (int k = 0; k < n; k++)
            if (!s->fixed[v[k]]) free_set.insert(v[k]);
    }
    return std::vector<uint32_t>(free_set.begin(), free_set.end());
}

}  // namespace

// The sequence of sub-problems SinglePass solves, all components in order (host only, no device):
// call with NULL arrays for sizes3 = {steps, total free variables, total expressions}, then with
// free_ptr[steps+1], free_vars, expr_ptr[steps+1], exprs.
int fk_system_single_pass_plan(const fk_system* s, uint32_t* sizes3, uint32_t* free_ptr, uint32_t* free_vars, uint32_t* expr_ptr,
                               uint32_t* exprs) {
    if (!s) return FK_ERR_INVALID;
    std::vector<std::vector<uint32_t>> var_exprs, expr_vars;
    equation_graph(s, var_exprs, expr_vars);
    fk::SinglePassPlanner planner(var_exprs, expr_vars);
    std::vector<fk::SinglePassStep> all;
    for (const fk_system::Comp& c : s->comps) {
        if (c.elements.empty()) continue;
        for (fk::SinglePassStep& st : planner.plan(component_free_variables(s, c))) all.push_back(std::move(st));
    }
    uint32_t nf = 0, ne = 0;
    for (const auto& st : all) { nf += (uint32_t)st.free_variables.size(); ne += (uint32_t)st.expressions.size(); }
    if (sizes3) { sizes3[0] = (uint32_t)all.size(); sizes3[1] = nf; sizes3[2] = ne; }
    if (!free_ptr || !free_vars || !expr_ptr || !exprs) return FK_OK;
    uint32_t af = 0, ae = 0;
    for (size_t k = 0; k < all.size(); k++) {
        free_ptr[k] = af; expr_ptr[k] = ae;
        for (uint32_t v : all[k].free_variables) free_vars[af++] = v;
        for (uint32_t e : all[k].expressions) exprs[ae++] = e;
    }
    free_ptr[all.size()] = af; expr_ptr[all.size()] = ae;
    return FK_OK;
}


// ---- Decomposer::RecursiveAssembly (SURVEY 8f-4) -------------------------------------------------------
namespace {

// graph.rs:98-117 as the planner wants it: dof = variables an element adds (lib.rs:372-403), valency = expressions
// of the constraint (constraints/mod.rs:331-334 and the like).
fk::RaGraph constraint_graph(const fk_system* s) {
    fk::RaGraph g;
    for (const Elem& e : s->elems) g.add_vertex(e.tag == kLength ? 1 : (e.tag == kPoint ? 2 : 0));
    for (const Constr& c : s->constrs) g.add_edge(c.n_expr, c.inc, c.n_inc);
    return g;
}

std::vector<fk::RaStep> component_plan(const fk_system* s, const fk_system::Comp& c) {
    fk::RecursiveAssemblyPlanner planner(constraint_graph(s));
    return planner.plan(std::vector<uint32_t>(c.elements.begin(), c.elements.end()),
                        std::vector<uint32_t>(c.constraints.begin(), c.constraints.end()));
}

const std::vector<uint32_t>* find_list(const fk::RaLists& m, uint32_t key) {
    auto it = m.find(key);
    return it == m.end() ? nullptr : &it->second;
}

// One step of the plan as a flattened problem (ClusteredSystem, assemble/mod.rs:282-590): free variables = the poses
// of the clusters the step moves (three each, starting at 0) followed by the variables of the step's elements; rows =
// two FK_POSE_POINT rows per (cluster, frontier point), then the step's expressions with their variables renumbered.
// The points' positions before the step enter as fixed variables behind the free ones.
struct ClusteredProblem {
    std::vector<uint32_t> elements;                                        // step_plus_frontier_elements
    std::vector<std::pair<uint32_t, std::vector<uint32_t>>> clusters;      // cluster key -> frontier points, in first-seen order
    std::map<uint32_t, uint32_t> slot;                                     // system variable -> free variable of the step
    std::vector<uint32_t> var_global, expr_global;  // local variable / expression -> system one, fk::kSbNone for a pose's
    std::vector<double> vars, param, x;
    std::vector<uint8_t> kind;
    std::vector<uint32_t> idx, free_vars, rows;
    fk_problem prob{};
    std::string error;

    bool build(const fk_system* s, const fk::RaStep& step, const std::vector<double>& vt, const std::vector<double>& pt) {
        auto has = [](const std::vector<uint32_t>& v, uint32_t x) { return std::find(v.begin(), v.end(), x) != v.end(); };
        elements = step.elements;
        // clusters reachable through shared frontier points (:355-398)
        std::vector<uint32_t> reach;
        auto add_clusters_of = [&](uint32_t el) -> size_t {
            const std::vector<uint32_t>* l = find_list(step.on_frontiers, el);
            if (!l) return 0;
            for (uint32_t c : *l)
                if (!has(reach, c)) reach.push_back(c);
            return l->size();
        };
        for (uint32_t el : step.elements)
            if (s->elems[el].tag == kPoint) add_clusters_of(el);
        for (size_t i = 0; i < reach.size(); i++) {
            const std::vector<uint32_t>* fr = find_list(step.frontier_elements, reach[i]);
            if (!fr) { error = "recursive assembly: cluster without a frontier list"; return false; }
            for (uint32_t el : *fr) {
                if (s->elems[el].tag != kPoint) continue;
                const size_t n_frontiers = add_clusters_of(el);
                if (!has(elements, el) && n_frontiers > 1) elements.push_back(el);
            }
        }
        // pose rows: one pair per (cluster, point on its frontier) (:401-429)
        for (uint32_t el : elements) {
            const std::vector<uint32_t>* l = find_list(step.on_frontiers, el);
            if (!l || s->elems[el].tag != kPoint) continue;
            for (uint32_t c : *l) {
                auto it = std::find_if(clusters.begin(), clusters.end(), [&](const std::pair<uint32_t, std::vector<uint32_t>>& p) { return p.first == c; });
                if (it == clusters.end()) {
                    clusters.emplace_back(c, std::vector<uint32_t>());
                    it = clusters.end() - 1;
                }
                it->second.push_back(el);
            }
        }
        // free variables (:432-477)
        vars.assign(clusters.size() * 3, 0.0);
        var_global.assign(clusters.size() * 3, fk::kSbNone);
        for (uint32_t el : elements) {
            const Elem& e = s->elems[el];
            const int n = e.tag == kLength ? 1 : (e.tag == kPoint ? 2 : 0);
            for (int k = 0; k < n; k++) {
                slot[e.a + k] = (uint32_t)vars.size();
                vars.push_back(vt[e.a + k]);
                var_global.push_back(e.a + k);
            }
        }
        const uint32_t n_free = (uint32_t)vars.size();
        x = vars;
        for (uint32_t k = 0; k < n_free; k++) free_vars.push_back(k);
        // rows
        for (size_t ci = 0; ci < clusters.size(); ci++)
            for (uint32_t point : clusters[ci].second) {
                const uint32_t pv = s->elems[point].a;
                const uint32_t at = (uint32_t)vars.size();
                vars.push_back(vt[pv]);      // the point before the step: constant of the two rows
                vars.push_back(vt[pv + 1]);
                var_global.push_back(pv);
                var_global.push_back(pv + 1);
                for (int y = 0; y < 2; y++) {
                    expr_global.push_back(fk::kSbNone);
                    rows.push_back((uint32_t)kind.size());
                    kind.push_back(y ? FK_POSE_POINT_Y : FK_POSE_POINT_X);
                    param.push_back(0.0);
                    idx.push_back((uint32_t)(3 * ci)); idx.push_back(slot.at(pv) + (uint32_t)y); idx.push_back(at); idx.push_back(0);
                }
            }
        static const int stored[FK_NUM_KINDS] = {2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 4, 3, 3};
        for (uint32_t c : step.constraints)
            for (uint8_t k = 0; k < s->constrs[c].n_expr; k++) {
                const uint32_t e = s->constrs[c].first_expr + k;
                expr_global.push_back(e);
                rows.push_back((uint32_t)kind.size());
                kind.push_back(s->kind[e]);
                param.push_back(pt[e]);
                for (int q = 0; q < 4; q++) {
                    uint32_t v = 0;
                    if (q < stored[s->kind[e]]) {
                        auto it = slot.find(s->idx[4 * (size_t)e + q]);
                        if (it == slot.end()) { error = "recursive assembly: an expression reads a variable outside its step"; return false; }
                        v = it->second;
                    }
                    idx.push_back(v);
                }
            }
        prob.n_vars = (uint32_t)vars.size(); prob.vars = vars.data();
        prob.n_expr = (uint32_t)kind.size(); prob.kind = kind.data(); prob.idx = idx.data(); prob.param = param.data();
        prob.n_free = n_free; prob.free_vars = free_vars.data();
        prob.n_rows = (uint32_t)rows.size(); prob.rows = rows.data();
        return true;
    }
};

// the reference panics here: unwrap on a missing cluster entry (recursive_assembly.rs:352-373)
const char kRaPanic[] = "recursive assembly: the decomposition reaches a cluster without bookkeeping (the reference panics on this system)";

// == System::solve(SolvingOptions { optimizer: LevenbergMarquardt, decomposer: RecursiveAssembly, perturb })
// (assemble/mod.rs:212-277): every step of every component's plan is one LM solve on the GPU; afterwards the points a
// moved cluster owns (and the step did not solve for) follow the cluster's pose on the host.  As in the reference,
// `fix` has no effect on this decomposer (ClusteredSystem takes every variable of the step's elements).
int solve_recursive_assembly(fk_system* s, int perturb, fk_report* reports, uint32_t cap, uint32_t* n_solved) {
    if (n_solved) *n_solved = 0;
    const size_t nv = s->vars.size();
    double sum = 0.0;
    size_t cnt = 0;
    for (double v : s->vars) { sum += v * v; cnt++; }
    for (size_t e = 0; e < s->kind.size(); e++)
        if (s->kind[e] == FK_POINT_POINT_DISTANCE || s->kind[e] == FK_POINT_LINE_DISTANCE) { sum += s->param[e] * s->param[e]; cnt++; }
    const double scale = std::sqrt(sum / (double)cnt);
    const double recip = 1.0 / scale;
    std::vector<double> vt(nv);
    for (size_t i = 0; i < nv; i++) vt[i] = s->vars[i] * recip;
    std::vector<double> pt(s->param);
    for (size_t e = 0; e < pt.size(); e++)
        if (s->kind[e] == FK_POINT_POINT_DISTANCE || s->kind[e] == FK_POINT_LINE_DISTANCE) pt[e] = recip * s->param[e];
    Lcg rng{42};
    uint32_t solved = 0;
    for (const fk_system::Comp& c : s->comps) {
        if (c.elements.empty()) continue;
        if (perturb) {
            for (uint32_t fv : component_free_variables(s, c)) {
                const double r1 = rng.next();
                const double r2 = rng.next();
                vt[fv] += vt[fv] * (1.0 / 8196.0) * r1 + (1.0 / 65568.0) * r2;
            }
        }
        std::vector<fk::RaStep> steps;
        try {
            steps = component_plan(s, c);
        } catch (const std::out_of_range&) {
            s->error = kRaPanic;
            return FK_ERR_INVALID;
        }
        for (const fk::RaStep& step : steps) {
            ClusteredProblem P;
            if (!P.build(s, step, vt, pt)) {
                s->error = P.error;
                return FK_ERR_INVALID;
            }
            fk_report rep{};
            const int rc = fk_lm_solve(&P.prob, P.x.data(), &rep);
            if (rc != FK_OK) return rc;
            for (const auto& kv : P.slot) {  // :226-233
                vt[kv.first] = P.x[kv.second];
                s->vars[kv.first] = scale * P.x[kv.second];
            }
            for (size_t ci = 0; ci < P.clusters.size(); ci++) {  // :235-273
                const std::vector<uint32_t>* owned = find_list(step.owned_elements, P.clusters[ci].first);
                if (!owned) continue;
                const double rot = P.x[3 * ci], tx = P.x[3 * ci + 1], ty = P.x[3 * ci + 2];
                const double sn = std::sin(rot), cs = std::cos(rot);  // Pose2D::transform_point, expressions.rs:1122-1136
                for (uint32_t el : *owned) {
                    if (std::find(P.elements.begin(), P.elements.end(), el) != P.elements.end() || s->elems[el].tag != kPoint) continue;
                    const uint32_t pv = s->elems[el].a;
                    const double u = vt[pv], w = vt[pv + 1];
                    const double uc = u * cs, us = u * sn, vc = w * cs, vs = w * sn;
                    const double nx = tx + uc - vs, ny = ty + us + vc;
                    vt[pv] = nx; vt[pv + 1] = ny;
                    s->vars[pv] = scale * nx; s->vars[pv + 1] = scale * ny;
                }
            }
            if (reports && solved < cap) reports[solved] = rep;
            solved++;
        }
    }
    if (n_solved) *n_solved = solved;
    return FK_OK;
}

}  // namespace

// == System::solve(SolvingOptions { optimizer: LevenbergMarquardt, decomposer, perturb }).
// decomposer 0: None (== fk_system_solve); 1: SinglePass (assemble/mod.rs:169-210): the strongly
// connected expression sets of every component are solved one after the other on the GPU, each seeing
// the variables solved before it as fixed values.  reports: one per solved sub-problem.
int fk_system_solve_opts(fk_system* s, int decomposer, int perturb, fk_report* reports, uint32_t cap, uint32_t* n_solved) {
    if (!s) return FK_ERR_INVALID;
    if (decomposer == 0) return fk_system_solve(s, perturb, reports, cap, n_solved);
    if (decomposer == 2) return solve_recursive_assembly(s, perturb, reports, cap, n_solved);
    if (decomposer != 1) return FK_ERR_INVALID;
    if (n_solved) *n_solved = 0;
    const size_t nv = s->vars.size();
    double sum = 0.0;
    size_t cnt = 0;
    for (double v : s->vars) { sum += v * v; cnt++; }
    for (size_t e = 0; e < s->kind.size(); e++)
        if (s->kind[e] == FK_POINT_POINT_DISTANCE || s->kind[e] == FK_POINT_LINE_DISTANCE) { sum += s->param[e] * s->param[e]; cnt++; }
    const double scale = std::sqrt(sum / (double)cnt);
    const double recip = 1.0 / scale;
    std::vector<double> vt(nv);
    for (size_t i = 0; i < nv; i++) vt[i] = s->vars[i] * recip;
    std::vector<double> pt(s->param);
    for (size_t e = 0; e < pt.size(); e++)
        if (s->kind[e] == FK_POINT_POINT_DISTANCE || s->kind[e] == FK_POINT_LINE_DISTANCE) pt[e] = recip * s->param[e];
    std::vector<std::vector<uint32_t>> var_exprs, expr_vars;
    equation_graph(s, var_exprs, expr_vars);
    fk::SinglePassPlanner planner(var_exprs, expr_vars);
    Lcg rng{42};
    uint32_t solved = 0;
    for (const fk_system::Comp& c : s->comps) {
        if (c.elements.empty()) continue;
        const std::vector<uint32_t> free_sorted = component_free_variables(s, c);
        if (perturb) {
            for (uint32_t fv : free_sorted) {
                const double r1 = rng.next();
                const double r2 = rng.next();
                vt[fv] += vt[fv] * (1.0 / 8196.0) * r1 + (1.0 / 65568.0) * r2;
            }
        }
        for (const fk::SinglePassStep& st : planner.plan(free_sorted)) {
            LocalProblem L;
            build_local(s, vt, pt, st.free_variables, st.expressions, L);
            fk_report rep{};
            const int rc = fk_lm_solve(&L.prob, L.x.data(), &rep);
            if (rc != FK_OK) return rc;
            for (size_t k = 0; k < L.free_global.size(); k++) {  // assemble/mod.rs:201-208
                vt[L.free_global[k]] = L.x[k];
                s->vars[L.free_global[k]] = scale * L.x[k];
            }
            if (reports && solved < cap) reports[solved] = rep;
            solved++;
        }
    }
    if (n_solved) *n_solved = solved;
    return FK_OK;
}

// == System::solve(options).  The reference dispatches on the optimizer only under Decomposer::None (assemble/mod.rs:148-158);
// SinglePass and RecursiveAssembly call levenberg_marquardt directly (:191, :224) whatever the optimizer.
int fk_system_solve_options(fk_system* s, const fk_solving_options* opts, fk_report* reports, uint32_t cap, uint32_t* n_solved) {
    if (!s || !opts || opts->optimizer > 1 || opts->decomposer > 2 || opts->perturb > 1 || opts->pad != 0) return FK_ERR_INVALID;
    if (opts->optimizer == 1 && opts->decomposer == 0) return solve_components(s, 1, (int)opts->perturb, reports, cap, n_solved);
    return fk_system_solve_opts(s, (int)opts->decomposer, (int)opts->perturb, reports, cap, n_solved);
}

// The recombination plan of all components as one stream of 32-bit words (host only, no device): per step
// n_constraints, constraints..., n_elements, elements..., n_free, free elements..., then on_frontiers, owned_elements,
// frontier_elements, each as n_keys and per key (ascending)  key, n, values....  Returns FK_OK; *n_words receives the
// stream's length (at most `cap` words are written), *n_steps the number of steps.
int fk_system_recursive_assembly_plan(const fk_system* s, uint32_t* out, uint32_t cap, uint32_t* n_words, uint32_t* n_steps) {
    if (!s) return FK_ERR_INVALID;
    std::vector<uint32_t> w;
    auto list = [&](const std::vector<uint32_t>& v) {
        w.push_back((uint32_t)v.size());
        w.insert(w.end(), v.begin(), v.end());
    };
    auto lists = [&](const fk::RaLists& m) {
        w.push_back((uint32_t)m.size());
        for (const auto& kv : m) {
            w.push_back(kv.first);
            list(kv.second);
        }
    };
    uint32_t steps = 0;
    for (const fk_system::Comp& c : s->comps) {
        if (c.elements.empty()) continue;
        std::vector<fk::RaStep> plan;
        try {
            plan = component_plan(s, c);
        } catch (const std::out_of_range&) {  // (the reference panics on this system, see solve_recursive_assembly)
            return FK_ERR_INVALID;
        }
        for (const fk::RaStep& st : plan) {
            list(st.constraints); list(st.elements); list(st.free_elements);
            lists(st.on_frontiers); lists(st.owned_elements); lists(st.frontier_elements);
            steps++;
        }
    }
    if (n_words) *n_words = (uint32_t)w.size();
    if (n_steps) *n_steps = steps;
    for (size_t k = 0; k < w.size() && k < cap && out; k++) out[k] = w[k];
    return FK_OK;
}

// == System::analyze (lib.rs:454-458, analyze/numerical/mod.rs:123-163): the dense Jacobian + the
// incremental Gauss-Jordan run on the GPU (fk_batch_analyze with a batch of one); the host maps
// dependent expressions back to their constraints (:149-160).
int fk_system_analyze(fk_system* s, uint32_t* constraints, uint32_t cap, uint32_t* n_found) {
    if (!s) return FK_ERR_INVALID;
    if (n_found) *n_found = 0;
    const uint32_t ne = (uint32_t)s->kind.size();
    if (ne == 0) return FK_OK;
    std::vector<uint32_t> all_vars(s->vars.size()), all_rows(ne);
    for (uint32_t i = 0; i < all_vars.size(); i++) all_vars[i] = i;
    for (uint32_t i = 0; i < ne; i++) all_rows[i] = i;
    fk_problem p{};
    p.n_vars = (uint32_t)s->vars.size(); p.vars = s->vars.data();
    p.n_expr = ne; p.kind = s->kind.data(); p.idx = s->idx.data(); p.param = s->param.data();
    p.n_free = p.n_vars; p.free_vars = all_vars.data();
    p.n_rows = ne; p.rows = all_rows.data();
    fk_topology* t = nullptr;
    int rc = fk_topology_create(&p, &t);
    if (rc != FK_OK) return rc;
    std::vector<uint8_t> independent(ne, 0);
    rc = fk_batch_analyze(t, 0, 1, s->vars.data(), s->param.data(), independent.data());
    fk_topology_destroy(t);
    if (rc != FK_OK) return rc;
    std::vector<uint32_t> expr_to_constraint(ne, 0);
    for (uint32_t c = 0; c < s->constrs.size(); c++)
        for (uint8_t k = 0; k < s->constrs[c].n_expr; k++) expr_to_constraint[s->constrs[c].first_expr + k] = c;
    uint32_t found = 0;
    for (uint32_t e = 0; e < ne; e++)
        if (!independent[e]) {
            if (constraints && found < cap) constraints[found] = expr_to_constraint[e];
            found++;
        }
    if (n_found) *n_found = found;
    return FK_OK;
}

// Residual of every constraint at the current (unscaled) variables == ConstraintHandle::
// calculate_residual (constraints/mod.rs:88-110): the expression residual, or the 2-norm of the two
// equalities of a coincidence.  Evaluated by the K2 kernel.
int fk_system_residuals(fk_system* s, double* out) {
    if (!s || !out) return FK_ERR_INVALID;
    const uint32_t ne = (uint32_t)s->kind.size();
    if (ne == 0) return FK_OK;
    std::vector<double> r(ne);
    std::vector<uint32_t> all_vars(s->vars.size()), all_rows(ne);
    for (uint32_t i = 0; i < all_vars.size(); i++) all_vars[i] = i;
    for (uint32_t i = 0; i < ne; i++) all_rows[i] = i;
    if (!s->eval_topo) {
        fk_problem p{};
        p.n_vars = (uint32_t)s->vars.size(); p.vars = s->vars.data();
        p.n_expr = ne; p.kind = s->kind.data(); p.idx = s->idx.data(); p.param = s->param.data();
        p.n_free = p.n_vars; p.free_vars = all_vars.data();
        p.n_rows = ne; p.rows = all_rows.data();
        fk_topology* t = nullptr;
        int rc = fk_topology_create(&p, &t);
        if (rc != FK_OK) return rc;
        s->eval_topo.reset(t);
    }
    fk_topology_info info;
    fk_topology_info_get(s->eval_topo.get(), &info);
    int rc;
    if (info.path == 2) {
        rc = fk_topology_eval(s->eval_topo.get(), s->vars.data(), s->param.data(), s->vars.data(), r.data(), nullptr, 0, nullptr);
    } else {
        fk_batch_plan* plan = nullptr;
        int dev = 0;
        rc = fk_batch_plan_create(s->eval_topo.get(), 1, dev, &plan);
        if (rc == FK_OK) rc = fk_batch_plan_upload(plan, 1, s->vars.data(), s->param.data(), nullptr);
        if (rc == FK_OK) rc = fk_batch_plan_eval(plan, 1, nullptr);
        if (rc == FK_OK) rc = fk_batch_plan_eval_download(plan, r.data(), nullptr, nullptr);
        if (rc == FK_OK) rc = fk_batch_plan_sync(plan);
        fk_batch_plan_destroy(plan);
    }
    if (rc != FK_OK) return rc;
    for (size_t c = 0; c < s->constrs.size(); c++) {
        const Constr& k = s->constrs[c];
        if (k.n_expr > 1) {
            double q = 0.0;
            for (uint8_t e = 0; e < k.n_expr; e++) q += r[k.first_expr + e] * r[k.first_expr + e];
            out[c] = std::sqrt(q);
        } else {
            out[c] = r[k.first_expr];
        }
    }
    return FK_OK;
}

// Connected components as the reference's graph holds them (including element-less slots).
uint32_t fk_system_num_components(const fk_system* s) { return s ? (uint32_t)s->comps.size() : 0; }
int fk_system_component(const fk_system* s, uint32_t ci, uint32_t* n_elements, uint32_t* elements, uint32_t* n_constraints, uint32_t* constraints) {
    if (!s || ci >= s->comps.size()) return FK_ERR_INVALID;
    const fk_system::Comp& c = s->comps[ci];
    if (n_elements) *n_elements = (uint32_t)c.elements.size();
    if (n_constraints) *n_constraints = (uint32_t)c.constraints.size();
    if (elements) std::copy(c.elements.begin(), c.elements.end(), elements);
    if (constraints) std::copy(c.constraints.begin(), c.constraints.end(), constraints);
    return FK_OK;
}

}  // extern "C"

// ---- System::solve over n variants of one drawing ------------------------------------------------------------------
namespace {

// The parts of a batch plan that do not depend on the decomposer: the expressions and, per variable, no draw or wave yet.
fk::SystemBatchLayout batch_layout(const fk_system* s) {
    fk::SystemBatchLayout lay;
    lay.n_vars = (uint32_t)s->vars.size();
    lay.n_constraints = (uint32_t)s->constrs.size();
    lay.kind = s->kind;
    lay.expr_constraint.assign(s->kind.size(), fk::kSbNone);
    for (uint32_t c = 0; c < s->constrs.size(); c++) lay.expr_constraint[s->constrs[c].first_expr] = c;  // update_parameter
    lay.var_draw.assign(s->vars.size(), fk::kSbNone);
    lay.var_wave.assign(s->vars.size(), fk::kSbNone);
    return lay;
}

// A component's draws from the solve's generator: two per free variable, in the ascending free set; var_draw their pair.
int component_draws(fk::SystemBatchLayout& lay, Lcg& rng, const std::vector<uint32_t>& free_sorted) {
    for (uint32_t fv : free_sorted) {
        if (lay.var_draw[fv] != fk::kSbNone) return fk::system_batch_fail(FK_ERR_INTERNAL, "a variable is free in two components");
        lay.var_draw[fv] = (uint32_t)(lay.draws.size() / 2);
        lay.draws.push_back(rng.next());
        lay.draws.push_back(rng.next());
    }
    return FK_OK;
}

// The drawing's batch plan: per non-empty component (component order) its LocalProblem numbering, the draws of the solve's
// generator and, per local variable, the draw already applied at the component's snapshot -- prepare_components perturbs
// component by component, so a variable of a later component is read unperturbed and one of an earlier component perturbed.
int batch_plan_for(const fk_system* s, std::shared_ptr<fk::SystemBatch>* out) {
    std::lock_guard<std::mutex> lock(s->batch_mu);
    if (!s->batch) {
        fk::SystemBatchLayout lay = batch_layout(s);
        std::vector<std::unique_ptr<LocalProblem>> locals;
        Lcg rng{42};
        for (const fk_system::Comp& c : s->comps) {
            if (c.elements.empty()) continue;  // assemble/mod.rs:87-89
            const std::vector<uint32_t> free_sorted = component_free_variables(s, c);
            const int rc = component_draws(lay, rng, free_sorted);
            if (rc != FK_OK) return rc;
            std::vector<uint32_t> exprs;
            for (uint32_t ci : c.constraints)
                for (uint8_t k = 0; k < s->constrs[ci].n_expr; k++) exprs.push_back(s->constrs[ci].first_expr + k);
            std::unique_ptr<LocalProblem> L(new LocalProblem());
            build_local(s, s->vars, s->param, free_sorted, exprs, *L);
            fk::SystemBatchLayout::Component comp;
            comp.slot_var = L->slot_global;
            for (uint32_t g : L->slot_global) comp.slot_draw.push_back(lay.var_draw[g]);
            comp.expr = exprs;
            comp.free_var = free_sorted;
            lay.comps.push_back(std::move(comp));
            locals.push_back(std::move(L));
        }
        std::vector<const fk_problem*> probs;
        for (const auto& L : locals) probs.push_back(&L->prob);
        const int rc = fk::system_batch_create(std::move(lay), probs, &s->batch);
        if (rc != FK_OK) return rc;
    }
    *out = s->batch;
    return FK_OK;
}

// The waves of the batched SinglePass and RecursiveAssembly plans.  The host loop is a sequence of nodes: per non-empty
// component its perturbation (reads and writes the component's free variables) followed by its sets or steps.  Node b follows
// an earlier node a when a writes what b reads or writes, or reads what b writes.  Times: a set or step of wave w at 2w + 1, a
// perturbation at the start of wave w at 2w; every node goes to the earliest time after all nodes it follows (ASAP).  The
// perturbation nodes count whether or not the call perturbs, so the waves do not depend on it.  Any schedule that respects
// the edges computes the host loop's values.
struct WaveScheduler {
    std::vector<int64_t> last_write, last_read;  // per system variable: latest time of a writer / reader
    explicit WaveScheduler(size_t n_vars) : last_write(n_vars, -1), last_read(n_vars, -1) {}
    // earliest time after every node that the node reading `reads` and writing `writes` (a subset of reads) follows
    int64_t earliest(const std::vector<uint32_t>& reads, const std::vector<uint32_t>& writes) const {
        int64_t t = -1;
        for (uint32_t g : reads) t = std::max(t, last_write[g]);
        for (uint32_t g : writes) t = std::max(t, last_read[g]);
        return t + 1;
    }
    void place(const std::vector<uint32_t>& reads, const std::vector<uint32_t>& writes, int64_t time) {
        for (uint32_t g : reads) last_read[g] = std::max(last_read[g], time);
        for (uint32_t g : writes) last_write[g] = std::max(last_write[g], time);
    }
    // a component's perturbation: the first wave start at or after its earliest time
    uint32_t perturbation(const std::vector<uint32_t>& free_sorted) {
        const uint32_t pw = (uint32_t)((earliest(free_sorted, free_sorted) + 1) / 2);
        place(free_sorted, free_sorted, 2 * (int64_t)pw);
        return pw;
    }
    // a set or step: the first solve time 2w + 1 at or after its earliest time
    uint32_t solve(const std::vector<uint32_t>& reads, const std::vector<uint32_t>& writes) {
        const uint32_t w = (uint32_t)(earliest(reads, writes) / 2);
        place(reads, writes, 2 * (int64_t)w + 1);
        return w;
    }
};

// A component's perturbation node: its wave, and the component's draws.
int perturbation_node(fk::SystemBatchLayout& lay, WaveScheduler& sched, Lcg& rng, const std::vector<uint32_t>& free_sorted) {
    const uint32_t pw = sched.perturbation(free_sorted);
    for (uint32_t fv : free_sorted) lay.var_wave[fv] = pw;
    return component_draws(lay, rng, free_sorted);
}

// fk_system_batch_solve_single_pass's plan: the sets of fk_system_solve_opts(decomposer = 1) in its order, each as its
// LocalProblem numbering (read: its variables, written: its free ones), the draws of batch_plan_for, and the waves.  Sets
// reach across components (SinglePass plans over the equation graph of every expression), so the edges between nodes are
// computed, not assumed.
int single_pass_batch_plan_for(const fk_system* s, std::shared_ptr<fk::SystemSpBatch>* out) {
    std::lock_guard<std::mutex> lock(s->batch_mu);
    if (!s->sp_batch) {
        fk::SystemBatchLayout lay = batch_layout(s);
        WaveScheduler sched(s->vars.size());
        std::vector<std::vector<uint32_t>> var_exprs, expr_vars;
        equation_graph(s, var_exprs, expr_vars);
        fk::SinglePassPlanner planner(var_exprs, expr_vars);
        std::vector<std::unique_ptr<LocalProblem>> locals;
        Lcg rng{42};
        for (const fk_system::Comp& c : s->comps) {
            if (c.elements.empty()) continue;  // assemble/mod.rs:87-89
            const std::vector<uint32_t> free_sorted = component_free_variables(s, c);
            const int rc = perturbation_node(lay, sched, rng, free_sorted);
            if (rc != FK_OK) return rc;
            for (const fk::SinglePassStep& st : planner.plan(free_sorted)) {
                std::unique_ptr<LocalProblem> L(new LocalProblem());
                build_local(s, s->vars, s->param, st.free_variables, st.expressions, *L);
                const uint32_t w = sched.solve(L->slot_global, st.free_variables);
                fk::SystemBatchLayout::Component comp;
                comp.slot_var = L->slot_global;
                comp.expr = st.expressions;
                comp.free_var = st.free_variables;
                lay.comps.push_back(std::move(comp));
                lay.comp_wave.push_back(w);
                lay.n_waves = std::max(lay.n_waves, w + 1);
                locals.push_back(std::move(L));
            }
        }
        std::vector<const fk_problem*> probs;
        for (const auto& L : locals) probs.push_back(&L->prob);
        const int rc = fk::system_sp_batch_create(std::move(lay), probs, &s->sp_batch);
        if (rc != FK_OK) return rc;
    }
    *out = s->sp_batch;
    return FK_OK;
}

// fk_system_batch_solve_recursive_assembly's plan: the steps of fk_system_solve_opts(decomposer = 2) in its order, each as
// its ClusteredProblem (built once on the template values: its structure does not depend on them), the draws of
// batch_plan_for, and the waves.  A step reads its variables (element variables and the point copies behind them) and the
// points it moves, and writes its element variables and the points it moves; the moves are the host loop's, in its order.
int recursive_assembly_batch_plan_for(const fk_system* s, std::shared_ptr<fk::SystemSpBatch>* out) {
    std::lock_guard<std::mutex> lock(s->batch_mu);
    if (!s->ra_batch) {
        fk::SystemBatchLayout lay = batch_layout(s);
        WaveScheduler sched(s->vars.size());
        std::vector<std::unique_ptr<ClusteredProblem>> problems;
        Lcg rng{42};
        for (const fk_system::Comp& c : s->comps) {
            if (c.elements.empty()) continue;  // assemble/mod.rs:87-89
            const int rc = perturbation_node(lay, sched, rng, component_free_variables(s, c));
            if (rc != FK_OK) return rc;
            std::vector<fk::RaStep> steps;
            try {
                steps = component_plan(s, c);
            } catch (const std::out_of_range&) {
                return fk::system_batch_fail(FK_ERR_INVALID, kRaPanic);
            }
            for (const fk::RaStep& step : steps) {
                std::unique_ptr<ClusteredProblem> P(new ClusteredProblem());
                if (!P->build(s, step, s->vars, s->param)) return fk::system_batch_fail(FK_ERR_INVALID, P->error);
                fk::SystemBatchLayout::Component comp;
                comp.slot_var = P->var_global;
                comp.expr = P->expr_global;
                comp.free_var.assign(P->var_global.begin(), P->var_global.begin() + P->prob.n_free);
                for (size_t ci = 0; ci < P->clusters.size(); ci++) {  // as solve_recursive_assembly walks them (:235-273)
                    const std::vector<uint32_t>* owned = find_list(step.owned_elements, P->clusters[ci].first);
                    if (!owned) continue;
                    for (uint32_t el : *owned) {
                        if (std::find(P->elements.begin(), P->elements.end(), el) != P->elements.end() || s->elems[el].tag != kPoint) continue;
                        comp.moves.push_back(s->elems[el].a);
                        comp.moves.push_back((uint32_t)(3 * ci));
                    }
                }
                std::vector<uint32_t> reads, writes;
                for (uint32_t g : comp.slot_var)
                    if (g != fk::kSbNone) reads.push_back(g);
                for (uint32_t g : comp.free_var)
                    if (g != fk::kSbNone) writes.push_back(g);
                for (size_t m = 0; m < comp.moves.size(); m += 2)
                    for (uint32_t y = 0; y < 2; y++) {
                        reads.push_back(comp.moves[m] + y);
                        writes.push_back(comp.moves[m] + y);
                    }
                const uint32_t w = sched.solve(reads, writes);
                lay.comps.push_back(std::move(comp));
                lay.comp_wave.push_back(w);
                lay.step_constraint.push_back(step.constraints[0]);
                lay.n_waves = std::max(lay.n_waves, w + 1);
                problems.push_back(std::move(P));
            }
        }
        std::vector<const fk_problem*> probs;
        for (const auto& P : problems) probs.push_back(&P->prob);
        const int rc = fk::system_sp_batch_create(std::move(lay), probs, &s->ra_batch);
        if (rc != FK_OK) return rc;
    }
    *out = s->ra_batch;
    return FK_OK;
}

// A solve batch call on s's template rows.
fk::SystemBatchCall batch_call(const fk_system* s, int optimizer, int perturb, uint32_t n, const double* vars, const double* params,
                               double* vars_out, fk_report* reports, uint32_t reports_per_variant, int n_gpus) {
    return {optimizer, perturb, n_gpus, n, vars, params, s->vars.data(), s->param.data(), vars_out, reports, reports_per_variant};
}

// The host probe and the call of the two wave plans (SinglePass, RecursiveAssembly), given how to build the plan.
using WavePlanFor = int (*)(const fk_system*, std::shared_ptr<fk::SystemSpBatch>*);

int wave_batch_layout(WavePlanFor plan_for, const fk_system* s, uint32_t* n_steps, uint32_t* n_waves, uint32_t* n_structures,
                      uint32_t* step_wave, uint32_t* step_structure) {
    if (!s) return fk::system_batch_fail(FK_ERR_INVALID, "null system");
    std::shared_ptr<fk::SystemSpBatch> b;
    const int rc = plan_for(s, &b);
    if (rc != FK_OK) return rc;
    std::vector<uint32_t> wave, structure;
    fk::system_sp_batch_layout(*b, n_steps, n_waves, n_structures, &wave, &structure);
    if (step_wave) std::copy(wave.begin(), wave.end(), step_wave);
    if (step_structure) std::copy(structure.begin(), structure.end(), step_structure);
    return FK_OK;
}

int wave_batch_solve(WavePlanFor plan_for, const fk_system* s, int perturb, uint32_t n, const double* vars, const double* params,
                     double* vars_out, fk_report* reports, uint32_t reports_per_variant, uint32_t* n_solved, int n_gpus) {
    if (!s || !vars_out) return fk::system_batch_fail(FK_ERR_INVALID, "null system or vars_out");
    if (perturb != 0 && perturb != 1) return fk::system_batch_fail(FK_ERR_INVALID, "perturb must be 0 or 1");
    std::shared_ptr<fk::SystemSpBatch> b;
    int rc = plan_for(s, &b);
    if (rc != FK_OK) return rc;
    uint32_t n_steps = 0;
    fk::system_sp_batch_layout(*b, &n_steps, nullptr, nullptr, nullptr, nullptr);
    if (n_solved) *n_solved = n_steps;
    return fk::system_sp_batch_solve(*b, batch_call(s, 0, perturb, n, vars, params, vars_out, reports, reports_per_variant, n_gpus));
}

// fk_system_batch_analyze / _residuals' plan: the expressions with their slot tables and the constraints' expression ranges.
int analyze_batch_plan_for(const fk_system* s, std::shared_ptr<fk::SystemAnBatch>* out) {
    std::lock_guard<std::mutex> lock(s->batch_mu);
    if (!s->an_batch) {
        fk::SystemAnLayout lay;
        lay.n_vars = (uint32_t)s->vars.size();
        lay.kind = s->kind;
        lay.slot_var.assign(s->kind.size() * 8, 0);
        for (size_t e = 0; e < s->kind.size(); e++) fk::expand_slots(s->kind[e], &s->idx[4 * e], &lay.slot_var[8 * e]);
        lay.expr_constraint.assign(s->kind.size(), fk::kSbNone);
        lay.con_off.push_back(0);
        for (uint32_t c = 0; c < s->constrs.size(); c++) {
            // (fk_system_add_constraint appends a constraint's expressions: first_expr is the previous constraint's end)
            lay.expr_constraint[s->constrs[c].first_expr] = c;  // update_parameter
            lay.con_off.push_back(s->constrs[c].first_expr + s->constrs[c].n_expr);
        }
        const int rc = fk::system_an_batch_create(std::move(lay), &s->an_batch);
        if (rc != FK_OK) return rc;
    }
    *out = s->an_batch;
    return FK_OK;
}

int an_batch_run(const fk_system* s, uint32_t n, const double* vars, const double* params, uint8_t* dependent, double* residuals,
                 int n_gpus) {
    if (!s || (n && !dependent && !residuals)) return fk::system_batch_fail(FK_ERR_INVALID, "null system or output");
    std::shared_ptr<fk::SystemAnBatch> b;
    const int rc = analyze_batch_plan_for(s, &b);
    if (rc != FK_OK) return rc;
    fk::SystemAnCall c;
    c.n_gpus = n_gpus;
    c.n = n;
    c.vars = vars;
    c.params = params;
    c.tmpl_vars = s->vars.data();
    c.tmpl_param = s->param.data();
    c.dependent = dependent;
    c.residuals = residuals;
    return fk::system_an_batch_run(*b, c);
}

// fk_systems_solve / fk_systems_layout: the refusals of the call (before any device work) and every drawing's batch plan.
int systems_drawings(uint32_t n, fk_system* const* systems, const fk_solving_options* opts, std::vector<fk::SystemsDrawing>& d,
                     std::vector<std::shared_ptr<fk::SystemBatch>>& plans) {
    if (!opts) return fk::system_batch_fail(FK_ERR_INVALID, "null options");
    if (opts->optimizer > 1 || opts->perturb > 1 || opts->pad != 0 || opts->decomposer > 2)
        return fk::system_batch_fail(FK_ERR_INVALID, "invalid solving options");
    if (opts->decomposer != 0) return fk::system_batch_fail(FK_ERR_INVALID, "fk_systems_solve takes Decomposer::None only (decomposer 0)");
    if (n && !systems) return fk::system_batch_fail(FK_ERR_INVALID, "null systems");
    std::set<const fk_system*> seen;
    for (uint32_t i = 0; i < n; i++) {
        if (!systems[i]) return fk::system_batch_fail(FK_ERR_INVALID, "null system at index " + std::to_string(i));
        if (!seen.insert(systems[i]).second)
            return fk::system_batch_fail(FK_ERR_INVALID, "system at index " + std::to_string(i) + " is given twice");
    }
    plans.resize(n);
    d.resize(n);
    for (uint32_t i = 0; i < n; i++) {
        const int rc = batch_plan_for(systems[i], &plans[i]);
        if (rc != FK_OK) return rc;
        d[i] = {plans[i].get(), systems[i]->vars.data(), systems[i]->param.data()};
    }
    return FK_OK;
}

}  // namespace

extern "C" {

int fk_systems_layout(uint32_t n, fk_system* const* systems, const fk_solving_options* opts, uint32_t* n_components, uint32_t* n_structures,
                      uint32_t* instances, uint32_t* launch_kind) {
    std::vector<fk::SystemsDrawing> d;
    std::vector<std::shared_ptr<fk::SystemBatch>> plans;
    const int rc = systems_drawings(n, systems, opts, d, plans);
    if (rc != FK_OK) return rc;
    uint32_t nc = 0;
    std::vector<uint32_t> inst, kind;
    fk::systems_layout(d, (int)opts->optimizer, &nc, &inst, &kind);
    if (n_components) *n_components = nc;
    if (n_structures) *n_structures = (uint32_t)inst.size();
    if (instances) std::copy(inst.begin(), inst.end(), instances);
    if (launch_kind) std::copy(kind.begin(), kind.end(), launch_kind);
    return FK_OK;
}

int fk_systems_solve(uint32_t n, fk_system* const* systems, const fk_solving_options* opts, fk_report* reports, uint32_t reports_cap,
                     uint32_t* n_solved, int n_gpus) {
    std::vector<fk::SystemsDrawing> d;
    std::vector<std::shared_ptr<fk::SystemBatch>> plans;
    int rc = systems_drawings(n, systems, opts, d, plans);
    if (rc != FK_OK || n == 0) return rc;
    std::vector<size_t> var_off(n + 1, 0), rep_off(n + 1, 0);
    for (uint32_t i = 0; i < n; i++) {
        uint32_t nc = 0;
        fk::system_batch_layout(*plans[i], &nc, nullptr, nullptr);
        var_off[i + 1] = var_off[i] + systems[i]->vars.size();
        rep_off[i + 1] = rep_off[i] + nc;
    }
    // all or nothing: the results land in the call's rows, and only a complete call writes them into the systems
    std::vector<double> vars_out(std::max<size_t>(var_off[n], 1));
    std::vector<fk_report> reps(std::max<size_t>(rep_off[n], 1));
    rc = fk::systems_solve(d, (int)opts->optimizer, (int)opts->perturb, n_gpus, vars_out.data(), reps.data());
    if (rc != FK_OK) return rc;
    for (uint32_t i = 0; i < n; i++) {  // assemble/mod.rs:161-166
        std::vector<double>& v = systems[i]->vars;
        if (!v.empty()) std::memcpy(v.data(), vars_out.data() + var_off[i], sizeof(double) * v.size());
        if (n_solved) n_solved[i] = (uint32_t)(rep_off[i + 1] - rep_off[i]);
    }
    if (reports) std::copy(reps.begin(), reps.begin() + std::min<size_t>(reports_cap, rep_off[n]), reports);
    return FK_OK;
}

int fk_system_batch_analyze(const fk_system* s, uint32_t n, const double* vars, const double* params, uint8_t* dependent, int n_gpus) {
    return an_batch_run(s, n, vars, params, dependent, nullptr, n_gpus);
}

int fk_system_batch_residuals(const fk_system* s, uint32_t n, const double* vars, const double* params, double* out, int n_gpus) {
    return an_batch_run(s, n, vars, params, nullptr, out, n_gpus);
}

int fk_system_batch_layout(const fk_system* s, uint32_t* n_components, uint32_t* n_structures, uint32_t* multiplicity) {
    if (!s) return fk::system_batch_fail(FK_ERR_INVALID, "null system");
    std::shared_ptr<fk::SystemBatch> b;
    const int rc = batch_plan_for(s, &b);
    if (rc != FK_OK) return rc;
    std::vector<uint32_t> mult;
    fk::system_batch_layout(*b, n_components, n_structures, &mult);
    if (multiplicity) std::copy(mult.begin(), mult.end(), multiplicity);
    return FK_OK;
}

int fk_system_batch_solve(const fk_system* s, const fk_solving_options* opts, uint32_t n, const double* vars, const double* params,
                          double* vars_out, fk_report* reports, uint32_t reports_per_variant, uint32_t* n_solved, int n_gpus) {
    if (!s || !opts || !vars_out) return fk::system_batch_fail(FK_ERR_INVALID, "null system, options or vars_out");
    if (opts->optimizer > 1 || opts->perturb > 1 || opts->pad != 0) return fk::system_batch_fail(FK_ERR_INVALID, "invalid solving options");
    if (opts->decomposer != 0)
        return fk::system_batch_fail(FK_ERR_INVALID, "fk_system_batch_solve takes Decomposer::None only (decomposer 0)");
    std::shared_ptr<fk::SystemBatch> b;
    int rc = batch_plan_for(s, &b);
    if (rc != FK_OK) return rc;
    uint32_t nc = 0;
    fk::system_batch_layout(*b, &nc, nullptr, nullptr);
    if (n_solved) *n_solved = nc;
    return fk::system_batch_solve(*b, batch_call(s, (int)opts->optimizer, (int)opts->perturb, n, vars, params, vars_out, reports,
                                                 reports_per_variant, n_gpus));
}

int fk_system_single_pass_batch_layout(const fk_system* s, uint32_t* n_steps, uint32_t* n_waves, uint32_t* n_structures,
                                       uint32_t* step_wave, uint32_t* step_structure) {
    return wave_batch_layout(single_pass_batch_plan_for, s, n_steps, n_waves, n_structures, step_wave, step_structure);
}

int fk_system_batch_solve_single_pass(const fk_system* s, int perturb, uint32_t n, const double* vars, const double* params,
                                      double* vars_out, fk_report* reports, uint32_t reports_per_variant, uint32_t* n_solved, int n_gpus) {
    return wave_batch_solve(single_pass_batch_plan_for, s, perturb, n, vars, params, vars_out, reports, reports_per_variant, n_solved, n_gpus);
}

int fk_system_recursive_assembly_batch_layout(const fk_system* s, uint32_t* n_steps, uint32_t* n_waves, uint32_t* n_structures,
                                              uint32_t* step_wave, uint32_t* step_structure) {
    return wave_batch_layout(recursive_assembly_batch_plan_for, s, n_steps, n_waves, n_structures, step_wave, step_structure);
}

int fk_system_batch_solve_recursive_assembly(const fk_system* s, int perturb, uint32_t n, const double* vars, const double* params,
                                             double* vars_out, fk_report* reports, uint32_t reports_per_variant, uint32_t* n_solved,
                                             int n_gpus) {
    return wave_batch_solve(recursive_assembly_batch_plan_for, s, perturb, n, vars, params, vars_out, reports, reports_per_variant,
                            n_solved, n_gpus);
}

}  // extern "C"
