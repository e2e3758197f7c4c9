// Control flow of fiksi/src/solve/lbfgs.rs for one sketch, shared by the tile kernel (fk_batch_lbfgs_kernel, state in
// shared memory, lm_kernels.cu) and the CTA kernel (fk_lbfgs_cta_kernel, state in global memory, lbfgs_global.cu): the
// two-loop recursion with a history of 5 (lbfgs.rs:77-143), the Hager-Zhang line search (mod hager_zhang, :218-506) and
// the three exits (:53-56, :177-182).  Every scalar that steers the control flow (dot products, sums of squares) is a
// sequential sum in index order, exactly as the reference's iterator sums are, so the decisions are the oracle's.  The
// dense row-major Jacobian of the reference is kept in its sparse CSC form; the dense path's "assign per slot" rule
// (expressions.rs:1003-1007) is honoured by eval_row_assign.
//
// The executing group of threads is described by V, the vector primitives:
//   v.sync()                         barrier of the group
//   v.each(cnt, f)                   f(i) for this thread's share of [0, cnt)
//   v.leader()                       true in exactly one thread of the group
//   v.dot(a, b, k)                   Σ a[i]*b[i], i ascending from 0.0, the same value in every thread
//   v.dot2(a1, b1, k1, a2, b2, k2, &o1, &o2)   two independent v.dot (a group may run the two chains side by side)
//   v.evaluate(pt, s)                residuals, Jacobian and gradient at pt, visible to the whole group on return
// The library is built with -fmad=false, so `s += a*b` is a rounded product and an add: a group may form the products
// in parallel first and keep only the chain of adds serial without changing a bit.
#pragma once
#include <cstdint>

#include "../../include/fiksi_b200.h"
#include "expressions.cuh"
#include "lm_kernels.cuh"

namespace fk {

constexpr uint32_t kNop = 0xFFFFFFFFu;

struct LbfgsTables {
    const uint32_t* jcolptr;  // [n+1] CSC of the Jacobian without damping rows
    const uint32_t* jrow;     // [jnnz]
};

// The per-sketch state: x, xs, g, dir [n]; sh, yh [5][n]; r [m]; J [jnnz]; rho, alpha [5].
struct LbfgsVecs {
    double *x, *xs, *g, *dir, *sh, *yh, *r, *J, *rho, *alpha;
};

template <int KIND>
__device__ __forceinline__ void eval_row_assign(const DevProgram& P, uint32_t row, const double* xfree, const double* __restrict__ vars,
                                                const double* __restrict__ params, double* rdst, double* jdst) {
    const uint32_t hdr = __ldg(P.row_hdr + row);
    if (hdr == kNop) return;
    const int kind = KIND >= 0 ? KIND : (int)(hdr & 0xFFu);
    const int a = dev::arity_of(kind);
    uint2 sl[8];
    double v[8], g[8];
#pragma unroll
    for (int s = 0; s < 8; s++) {
        v[s] = 0.0;
        sl[s] = make_uint2(kNop, kNop);
        if (s < a) {
            sl[s] = __ldg(P.row_slots + row * 8 + s);
            v[s] = (int32_t)sl[s].x >= 0 ? xfree[sl[s].x] : __ldg(vars + (sl[s].x & 0x7FFFFFFFu));
        }
    }
    rdst[row] = dev::eval_expression(kind, v, __ldg(params + (hdr >> 8)), g);
#pragma unroll
    for (int s = 0; s < 8; s++)
        if (s < a && sl[s].y != kNop) jdst[sl[s].y & 0xFFFFFFu] = g[s];  // assignment: the later slot wins
}

// g[c] = Σ_q J[q] * r[jrow[q]] over column c's entries, rows ascending, from 0.0 (lbfgs.rs:201-212).
__device__ __forceinline__ double lbfgs_grad_col(const LbfgsTables& T, const double* J, const double* r, uint32_t c) {
    double acc = 0.0;
    for (uint32_t q = __ldg(T.jcolptr + c); q < __ldg(T.jcolptr + c + 1); q++) acc += J[q] * r[__ldg(T.jrow + q)];
    return acc;
}

struct HzParam { double p, phi, dphi; };

// The whole L-BFGS solve of one sketch: x from the sketch's variable row, the solved free values into `out`, the report
// into `*report`.
template <class V>
__device__ __forceinline__ void lbfgs_solve(V& v, const DevProgram& P, const double* __restrict__ vars, const LbfgsVecs& s,
                                            double* __restrict__ out, fk_report* __restrict__ report) {
    const uint32_t n = P.n, m = P.m;
    double *x = s.x, *xs = s.xs, *g = s.g, *dir = s.dir, *sh = s.sh, *yh = s.yh, *r = s.r, *rho = s.rho, *alpha = s.alpha;
    uint32_t evaluations = 0;
    auto evaluate = [&](const double* pt) {
        v.evaluate(pt, s);
        evaluations++;
    };

    v.each(n, [&](uint32_t i) { x[i] = __ldg(vars + __ldg(P.free_vars + i)); });
    v.each(P.jnnz, [&](uint32_t i) { s.J[i] = 0.0; });
    // The histories start as zeros (lbfgs.rs:66-72) and the reference READS not-yet-written slots during
    // the first five iterations (slot (k + i) % 5 for i < min(k, 5), :84-85): they must be zero here too.
    v.each(5 * n, [&](uint32_t i) { sh[i] = 0.0; yh[i] = 0.0; });
    v.each(5, [&](uint32_t i) { rho[i] = 0.0; alpha[i] = 0.0; });
    v.sync();
    evaluate(x);
    double prev = v.dot(r, r, m);
    uint32_t exit_reason = 3, iterations = 0;
    uint64_t trace = 0;
    double last_step = 0.0, ssr = prev;
    bool run = !(prev < 1e-4);
    if (!run) exit_reason = 0;

    for (uint32_t k = 0; run && k < 100; k++) {
        const uint32_t hl = k < 5 ? k : 5;
        v.each(n, [&](uint32_t j) { dir[j] = g[j]; });
        v.sync();
        for (uint32_t ii = hl; ii-- > 0;) {  // lbfgs.rs:83-99
            const uint32_t h = (k + ii) % 5;
            const double a_i = rho[h] * v.dot(sh + h * n, dir, n);
            v.sync();
            if (v.leader()) alpha[ii] = a_i;
            v.each(n, [&](uint32_t j) { dir[j] -= a_i * yh[h * n + j]; });
            v.sync();
        }
        if (k > 0) {  // :101-121
            const uint32_t hp = (k - 1) % 5;
            double sdy, ydy;
            v.dot2(sh + hp * n, yh + hp * n, n, yh + hp * n, yh + hp * n, n, &sdy, &ydy);
            if (ydy > 0.0) {
                const double scale = sdy / ydy;
                v.sync();
                v.each(n, [&](uint32_t j) { dir[j] *= scale; });
                v.sync();
            }
        }
        for (uint32_t ii = 0; ii < hl; ii++) {  // :123-139
            const uint32_t h = (k + ii) % 5;
            const double beta = rho[h] * v.dot(yh + h * n, dir, n);
            const double coef = alpha[ii] - beta;
            v.sync();
            v.each(n, [&](uint32_t j) { dir[j] += sh[h * n + j] * coef; });
            v.sync();
        }
        const uint32_t h = k % 5;
        v.each(n, [&](uint32_t j) {
            dir[j] *= -1.0;          // :141-143
            yh[h * n + j] = g[j];    // :149-150
            xs[j] = x[j];
        });
        v.sync();

        // ---- hager_zhang::line_search (:461-506) --------------------------------------------------------
        const double phi0 = prev, dphi0 = v.dot(g, dir, n);
        const uint32_t evals_before = evaluations;
        bool guard = false;
        auto calculate_phi = [&](double p) -> HzParam {  // :270-286
            v.sync();
            v.each(n, [&](uint32_t j) { xs[j] = x[j] + p * dir[j]; });
            v.sync();
            evaluate(xs);
            HzParam res;
            res.p = p;
            v.dot2(r, r, m, g, dir, n, &res.phi, &res.dphi);
            return res;
        };
        auto secant = [](HzParam a, HzParam b) { return (a.p * b.dphi - b.p * a.dphi) / (b.dphi - a.dphi); };
        auto wolfe = [&](HzParam c) {  // :307-322
            if ((c.phi <= phi0 + c.p * (1e-4 * dphi0)) && (c.dphi >= 0.9 * dphi0)) return true;
            if (c.phi <= phi0 + 1e-6 && (2.0 * 1e-4 - 1.0) * dphi0 >= c.dphi && c.dphi >= 0.9 * dphi0) return true;
            return false;
        };
        auto update = [&](HzParam a, HzParam b, HzParam c, HzParam& oa, HzParam& ob) {  // :325-353
            if (c.p < a.p || c.p > b.p) { oa = a; ob = b; return; }
            if (c.dphi >= 0.0) { oa = a; ob = c; return; }
            if (c.phi <= phi0 + 1e-6) { oa = c; ob = b; return; }
            HzParam aa = a, bb = c;
            for (int it = 0;; it++) {
                if (it >= 200) { guard = true; oa = aa; ob = bb; return; }
                const HzParam d = calculate_phi((1.0 - 0.5) * aa.p + 0.5 * bb.p);
                if (d.dphi >= 0.0) { oa = aa; ob = d; return; }
                else if (d.phi <= phi0 + 1e-6) aa = d;
                else bb = d;
            }
        };
        HzParam res = calculate_phi(1.0);  // :447-452
        if (!wolfe(res)) {
            HzParam a{0.0, phi0, dphi0};
            HzParam b = calculate_phi(5.0);  // bracket, :401-410
            HzParam c = res;
            bool found = false;
            for (int it = 0; it < 100 && !found && !guard; it++) {  // search, :414-443
                // secant2, :360-398
                HzParam a_, b_;
                HzParam cc = calculate_phi(secant(a, b));
                if (wolfe(cc)) { res = cc; found = true; break; }
                update(a, b, cc, a_, b_);
                if (guard) break;
                if (cc.p == b_.p) {
                    const HzParam c2 = calculate_phi(secant(b, b_));
                    if (wolfe(c2)) { res = c2; found = true; break; }
                    HzParam na, nb;
                    update(a_, b_, c2, na, nb);
                    a_ = na; b_ = nb;
                } else if (cc.p == a_.p) {
                    const HzParam c2 = calculate_phi(secant(a, a_));
                    if (wolfe(c2)) { res = c2; found = true; break; }
                    HzParam na, nb;
                    update(a_, b_, c2, na, nb);
                    a_ = na; b_ = nb;
                }
                if (guard) break;
                if (b_.p - a_.p > 0.66 * (b.p - a.p)) {
                    c = calculate_phi(0.5 * (a.p + b.p));
                    if (wolfe(c)) { res = c; found = true; break; }
                    HzParam na, nb;
                    update(a, b, c, na, nb);
                    a = na; b = nb;
                } else {
                    a = a_; b = b_;
                }
            }
            if (!found) res = calculate_phi(c.p);  // :440-442
        }
        v.sync();
        v.each(n, [&](uint32_t j) { x[j] = xs[j]; });  // :169
        iterations++;
        trace = trace * 31ull + (uint64_t)(evaluations - evals_before);
        last_step = res.p;
        ssr = res.phi;
        if (guard) { exit_reason = 4; break; }
        v.each(n, [&](uint32_t j) {  // :171-180
            const double sv = res.p * dir[j];
            sh[h * n + j] = sv;
            yh[h * n + j] = g[j] - yh[h * n + j];
        });
        v.sync();
        const double sdy = v.dot(sh + h * n, yh + h * n, n);
        if (v.leader()) rho[h] = 1.0 / sdy;
        v.sync();
        if (fabs(prev - res.phi) < 1e-10) { exit_reason = 1; break; }
        if (res.phi < 1e-6) { exit_reason = 2; break; }
        prev = res.phi;
    }

    v.sync();
    v.each(n, [&](uint32_t i) { out[i] = x[i]; });
    if (v.leader()) {
        fk_report rep;
        rep.exit_reason = exit_reason;
        rep.outer_iters = iterations;
        rep.factorizations = evaluations;
        rep.accepted = iterations;
        rep.ssr = ssr;
        rep.lambda = last_step;
        rep.trace_hash = trace;
        *report = rep;
    }
}

}  // namespace fk
