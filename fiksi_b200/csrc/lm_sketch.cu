// See lm_sketch.cuh.  Compiled with -fmad=false: a*b+c is two roundings unless it is an explicit fma().
#include "lm_sketch.cuh"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>

#include "expressions.cuh"
#include "lm_kernels.cuh"
#include "symbolic.hpp"

namespace fk {

namespace {

constexpr uint32_t kNone = 0xFFFFFFFFu;

// 1/d for a positive finite pivot (the tile kernel's sequence: hardware seed + two Newton steps).
__device__ __forceinline__ double sk_rcp(double d) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    double e = fma(-d, r, 1.0);
    r = fma(r, e, r);
    e = fma(-d, r, 1.0);
    r = fma(r, e, r);
    return r;
}

// Entry e of a lane's region lives at byte (e << 8) behind the lane's region address (32 lanes x 8 bytes per entry).
// Regions are held as 32-bit shared-window addresses, so a target's address is one 32-bit add of the lane's region address
// and the table word (generic pointers formed it as a 64-bit add folded into a three-input IADD3 with the window base).
// The accesses are asm volatile with a memory clobber: the compiler keeps them in program order (a target's load, its
// store; a later load of the same entry after that store), as it did for the plain loads and stores they replace.
using SmAddr = uint32_t;
__device__ __forceinline__ double lds(SmAddr a) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts(SmAddr a, double v) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory"); }
__device__ __forceinline__ double ldp(SmAddr p, uint32_t off) { return lds(p + off); }
__device__ __forceinline__ void stp(SmAddr p, uint32_t off, double v) { sts(p + off, v); }

__device__ __forceinline__ void cp_async8(SmAddr smem_dst, const void* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_dst), "l"(gmem_src) : "memory");
}

__host__ __device__ constexpr int sk_arity(int kind) {
    return kind == 0 ? 2 : kind == 1 ? 4 : kind <= 4 ? 6 : kind == 5 ? 5 : kind <= 9 ? 8 : kind == 10 ? 7 : 6;  // 11, 12: the pose rows
}
__host__ __device__ constexpr bool sk_has_param(int kind) { return kind == 1 || kind == 2 || kind == 4 || kind == 7; }

// N table words starting at the 16-byte aligned shared-memory address p (every lane reads the same address: one
// broadcast wavefront per 4 words).  wd has room for the padding words of the last load.
template <int N>
__device__ __forceinline__ void ld_words(const uint32_t* p, uint32_t (&wd)[(N + 3) / 4 * 4]) {
#pragma unroll
    for (int i = 0; i < (N + 3) / 4; i++) {
        const uint4 q = reinterpret_cast<const uint4*>(p)[i];
        wd[4 * i] = q.x; wd[4 * i + 1] = q.y; wd[4 * i + 2] = q.z; wd[4 * i + 3] = q.w;
    }
}

// One expression row of fiksi/src/subsystem.rs:143-165 for this thread's sketch, fused with its contributions
// to g = J^T(-r) and H = J^T J (rows arrive in ascending order and every sum starts from zero, so the sums
// keep the tile kernel's order).  All targets of a row are distinct (rows naming a free variable twice stay on
// the tile kernel), so they are fetched before the first FMA and stored afterwards: the accesses overlap
// instead of forming a load-FMA-store chain.  SPECIAL: some slot of the row is a fixed variable.
// rec: the row's record; h0: its first four words (already loaded).
template <int KIND, bool SPECIAL>
__device__ __forceinline__ void sk_eval_row(const uint32_t* rec, const uint4 h0, SmAddr x, SmAddr fx, SmAddr pr, SmAddr w, SmAddr f,
                                            double& ssr) {
    constexpr int A = sk_arity(KIND);
    constexpr int NP = A * (A + 1) / 2;
    constexpr int NW = 2 + 2 * A + NP;
    uint32_t t[(NW + 3) / 4 * 4];
    t[0] = h0.x; t[1] = h0.y; t[2] = h0.z; t[3] = h0.w;
#pragma unroll
    for (int i = 1; i < (NW + 3) / 4; i++) {
        const uint4 q = reinterpret_cast<const uint4*>(rec)[i];
        t[4 * i] = q.x; t[4 * i + 1] = q.y; t[4 * i + 2] = q.z; t[4 * i + 3] = q.w;
    }
    double v[8], g[8];
#pragma unroll
    for (int s = 0; s < 8; s++) v[s] = 0.0;
#pragma unroll
    for (int s = 0; s < A; s++) {
        const uint32_t src = t[2 + s];
        if (SPECIAL) v[s] = (src >> 31) ? ldp(fx, src & 0x7FFFFFFFu) : ldp(x, src);
        else v[s] = ldp(x, src);
    }
    const double param = sk_has_param(KIND) ? ldp(pr, t[1]) : 0.0;
    SmAddr gp[A];
    SmAddr hp[NP];
    double gv[A], hv[NP];
    // the targets do not depend on the row's arithmetic: fetch them before it
#pragma unroll
    for (int s = 0; s < A; s++) {
        const uint32_t o = t[2 + A + s];
        gp[s] = w + o;
        gv[s] = (!SPECIAL || o != kNone) ? lds(gp[s]) : 0.0;
    }
#pragma unroll
    for (int q = 0; q < NP; q++) {
        const uint32_t o = t[2 + 2 * A + q];
        hp[q] = f + o;
        hv[q] = (!SPECIAL || o != kNone) ? lds(hp[q]) : 0.0;
    }
    const double r = dev::eval_expression(KIND, v, param, g);
    ssr = ssr + r * r;  // lm.rs:195-197: sequential, not fused
    const double nr = -r;
#pragma unroll
    for (int s = 0; s < A; s++)
        if (!SPECIAL || t[2 + A + s] != kNone) sts(gp[s], fma(g[s], nr, gv[s]));
    int q = 0;
#pragma unroll
    for (int a = 0; a < A; a++)
#pragma unroll
        for (int b = 0; b <= a; b++, q++)
            if (!SPECIAL || t[2 + 2 * A + q] != kNone) sts(hp[q], fma(g[a], g[b], hv[q]));
}

// Two consecutive rows of one kind without fixed slots: loads and sqrt / divide chains of the two rows are independent
// and issue together; the accumulations stay in row order (row r's stores precede row r+1's target loads).
template <int KIND>
__device__ __forceinline__ void sk_eval_rows2(const uint32_t* rec0, const uint4 h0, const uint32_t* rec1, const uint4 h1, SmAddr x,
                                              SmAddr pr, SmAddr w, SmAddr f, double& ssr) {
    constexpr int A = sk_arity(KIND);
    constexpr int NP = A * (A + 1) / 2;
    constexpr int NW = 2 + 2 * A + NP;
    constexpr int NWD = (NW + 3) / 4 * 4;
    uint32_t t0[NWD], t1[NWD];
    t0[0] = h0.x; t0[1] = h0.y; t0[2] = h0.z; t0[3] = h0.w;
    t1[0] = h1.x; t1[1] = h1.y; t1[2] = h1.z; t1[3] = h1.w;
#pragma unroll
    for (int i = 1; i < NWD / 4; i++) {
        const uint4 q0 = reinterpret_cast<const uint4*>(rec0)[i], q1 = reinterpret_cast<const uint4*>(rec1)[i];
        t0[4 * i] = q0.x; t0[4 * i + 1] = q0.y; t0[4 * i + 2] = q0.z; t0[4 * i + 3] = q0.w;
        t1[4 * i] = q1.x; t1[4 * i + 1] = q1.y; t1[4 * i + 2] = q1.z; t1[4 * i + 3] = q1.w;
    }
    double v0[8], v1[8], g0[8], g1[8];
#pragma unroll
    for (int s = 0; s < 8; s++) v0[s] = v1[s] = 0.0;
#pragma unroll
    for (int s = 0; s < A; s++) {
        v0[s] = ldp(x, t0[2 + s]);
        v1[s] = ldp(x, t1[2 + s]);
    }
    const double p0 = sk_has_param(KIND) ? ldp(pr, t0[1]) : 0.0;
    const double p1 = sk_has_param(KIND) ? ldp(pr, t1[1]) : 0.0;
    SmAddr gp[A];
    SmAddr hp[NP];
    double gv[A], hv[NP];
#pragma unroll
    for (int s = 0; s < A; s++) {
        gp[s] = w + t0[2 + A + s];
        gv[s] = lds(gp[s]);
    }
#pragma unroll
    for (int q = 0; q < NP; q++) {
        hp[q] = f + t0[2 + 2 * A + q];
        hv[q] = lds(hp[q]);
    }
    const double r0 = dev::eval_expression(KIND, v0, p0, g0);
    const double r1 = dev::eval_expression(KIND, v1, p1, g1);
    ssr = ssr + r0 * r0;  // lm.rs:195-197: sequential, not fused
    ssr = ssr + r1 * r1;
    {
        const double nr = -r0;
#pragma unroll
        for (int s = 0; s < A; s++) sts(gp[s], fma(g0[s], nr, gv[s]));
        int q = 0;
#pragma unroll
        for (int a = 0; a < A; a++)
#pragma unroll
            for (int b = 0; b <= a; b++, q++) sts(hp[q], fma(g0[a], g0[b], hv[q]));
    }
    {
        const double nr = -r1;
#pragma unroll
        for (int s = 0; s < A; s++) {
            gp[s] = w + t1[2 + A + s];
            gv[s] = lds(gp[s]);
        }
#pragma unroll
        for (int q = 0; q < NP; q++) {
            hp[q] = f + t1[2 + 2 * A + q];
            hv[q] = lds(hp[q]);
        }
#pragma unroll
        for (int s = 0; s < A; s++) sts(gp[s], fma(g1[s], nr, gv[s]));
        int q = 0;
#pragma unroll
        for (int a = 0; a < A; a++)
#pragma unroll
            for (int b = 0; b <= a; b++, q++) sts(hp[q], fma(g1[a], g1[b], hv[q]));
    }
}

// Right-looking step of column k with C entries below the diagonal: the column is read once into registers,
// every target (C(C+1)/2 entries of later columns, C entries of the right-hand side: the forward substitution
// rides along) is fetched, updated with one FMA and stored.  Same operations as the tile kernel's
// L[dst] = fma(-(L[a] * inv), L[b], L[dst]).  body: C positions in f, C positions in w, C(C+1)/2 targets in f.
template <int C>
__device__ __forceinline__ void sk_column(const uint32_t* body, SmAddr f, SmAddr w, double wk, double inv) {
    constexpr int NP = C * (C + 1) / 2;
    uint32_t t[(2 * C + NP + 3) / 4 * 4];
    ld_words<2 * C + NP>(body, t);
    double l[C], s[C], wv[C], d[NP];
    SmAddr wp[C];
    SmAddr dp[NP];
#pragma unroll
    for (int a = 0; a < C; a++) l[a] = ldp(f, t[a]);
#pragma unroll
    for (int a = 0; a < C; a++) {
        wp[a] = w + t[C + a];
        wv[a] = lds(wp[a]);
    }
#pragma unroll
    for (int q = 0; q < NP; q++) {
        dp[q] = f + t[2 * C + q];
        d[q] = lds(dp[q]);
    }
#pragma unroll
    for (int a = 0; a < C; a++) s[a] = -(l[a] * inv);
    int q = 0;
#pragma unroll
    for (int a = 0; a < C; a++)
#pragma unroll
        for (int b = 0; b <= a; b++, q++) sts(dp[q], fma(s[a], l[b], d[q]));
#pragma unroll
    for (int a = 0; a < C; a++) sts(wp[a], fma(s[a], wk, wv[a]));
}

// Target q of a column record is the pair (a, b), b <= a, of the column's rows: q = a(a+1)/2 + b.
__host__ __device__ constexpr int sk_tri(int a, int b) { return a * (a + 1) / 2 + b; }

// Columns k and k+1 of a pair record (symbolic.hpp): L(:,k) = {k+1} u L(:,k+1), so column k+1's pivot, entries and
// right-hand side entry are column k's targets (0, 0), (a, 0) and w row 0, and its targets are column k's targets
// (a, b), a >= b >= 1.  Every target is loaded once, receives column k's FMA and then column k+1's, and is stored once;
// per entry the operations and their order are those of sk_column for k and then for k+1.  Column k+1's pivot is checked
// after column k's (the caller's), so fstat still records the first bad pivot in column order.
template <int C>
__device__ __forceinline__ void sk_column2(const uint32_t* body, SmAddr f, SmAddr w, double wk, double inv, double lam2, int& fstat) {
    constexpr int NP = C * (C + 1) / 2;
    uint32_t t[(2 * C + NP + 3) / 4 * 4];
    ld_words<2 * C + NP>(body, t);
    double l[C], s[C], wv[C], d[NP];
    SmAddr wp[C];
    SmAddr dp[NP];
#pragma unroll
    for (int a = 0; a < C; a++) l[a] = ldp(f, t[a]);
#pragma unroll
    for (int a = 0; a < C; a++) {
        wp[a] = w + t[C + a];
        wv[a] = lds(wp[a]);
    }
#pragma unroll
    for (int q = 0; q < NP; q++) {
        dp[q] = f + t[2 * C + q];
        d[q] = lds(dp[q]);
    }
#pragma unroll
    for (int a = 0; a < C; a++) s[a] = -(l[a] * inv);
    int q = 0;
#pragma unroll
    for (int a = 0; a < C; a++)
#pragma unroll
        for (int b = 0; b <= a; b++, q++) d[q] = fma(s[a], l[b], d[q]);
#pragma unroll
    for (int a = 0; a < C; a++) wv[a] = fma(s[a], wk, wv[a]);
    // column k+1's entries and right-hand side entry are final now
#pragma unroll
    for (int a = 1; a < C; a++) sts(dp[sk_tri(a, 0)], d[sk_tri(a, 0)]);
    sts(wp[0], wv[0]);
    const double d1 = d[0] + lam2;
    if (fstat == 0 && !(d1 > 0.0 && d1 < INFINITY)) fstat = d1 != d1 ? 2 : 1;
    const double inv1 = sk_rcp(d1);
    sts(dp[0], inv1);
#pragma unroll
    for (int a = 1; a < C; a++) s[a] = -(d[sk_tri(a, 0)] * inv1);
#pragma unroll
    for (int a = 1; a < C; a++)
#pragma unroll
        for (int b = 1; b <= a; b++) sts(dp[sk_tri(a, b)], fma(s[a], d[sk_tri(b, 0)], d[sk_tri(a, b)]));
#pragma unroll
    for (int a = 1; a < C; a++) sts(wp[a], fma(s[a], wv[0], wv[a]));
}

// Columns with more than 8 entries below the diagonal: same operations, one at a time.
__device__ __forceinline__ void sk_column_generic(const uint32_t* t, uint32_t C, SmAddr f, SmAddr w, double wk, double inv) {
    uint32_t q = 0;
    for (uint32_t a = 0; a < C; a++) {
        const double la = ldp(f, t[a]);
        const double sa = -(la * inv);
        for (uint32_t b = 0; b <= a; b++, q++) {
            SmAddr dst = f + t[2 * C + q];
            const double lb = b == a ? la : ldp(f, t[b]);
            sts(dst, fma(sa, lb, lds(dst)));
        }
        SmAddr wr = w + t[C + a];
        sts(wr, fma(sa, wk, lds(wr)));
    }
}

// acc - sum_{a} (L D)(row_a, k) z(row_a), rows descending as the tile kernel's scatter form applies them.
template <int C>
__device__ __forceinline__ double sk_back_column(const uint32_t* body, SmAddr f, SmAddr w, double acc) {
    uint32_t t[(2 * C + 3) / 4 * 4];
    ld_words<2 * C>(body, t);
    double l[C], z[C];
#pragma unroll
    for (int a = 0; a < C; a++) {
        l[a] = ldp(f, t[a]);
        z[a] = ldp(w, t[C + a]);
    }
#pragma unroll
    for (int a = C - 1; a >= 0; a--) acc = fma(-l[a], z[a], acc);
    return acc;
}

// Back substitution of a pair record: column k+1, then column k (acc: column k's right-hand side).  Rows descend and row
// k+1 is column k's last, so both sums run side by side over the rows below k+1 and share their z loads; z(k+1) goes to w
// and to the trial point's slot xs here.  Returns column k's sum, to be multiplied by 1 / d(k).
template <int C>
__device__ __forceinline__ double sk_back_column2(const uint32_t* body, SmAddr f, SmAddr w, SmAddr xs, double acc) {
    uint32_t t[(3 * C + 1 + 3) / 4 * 4];
    ld_words<3 * C + 1>(body, t);  // column k's entries, rows, column k+1's entries, its diagonal, perm[k+1]
    double l[C], l1[C], z[C];
#pragma unroll
    for (int a = 0; a < C; a++) l[a] = ldp(f, t[a]);
#pragma unroll
    for (int a = 1; a < C; a++) {
        z[a] = ldp(w, t[C + a]);
        l1[a] = ldp(f, t[2 * C + a - 1]);
    }
    const SmAddr zp1 = w + t[C];
    double acc1 = lds(zp1);
    const double inv1 = ldp(f, t[3 * C - 1]);
#pragma unroll
    for (int a = C - 1; a >= 1; a--) {
        acc1 = fma(-l1[a], z[a], acc1);
        acc = fma(-l[a], z[a], acc);
    }
    const double z1 = acc1 * inv1;
    sts(zp1, z1);
    stp(xs, t[3 * C], z1);
    return fma(-l[0], z1, acc);
}

// D L^T z = y in place in w (rec: the back section), delta in variable order (qr.rs:354) into the trial point's slots xs.
__device__ __forceinline__ void sk_back_solve(const uint32_t* rec, uint32_t n, SmAddr f, SmAddr w, SmAddr xs) {
    uint4 hn = *reinterpret_cast<const uint4*>(rec);
    for (uint32_t c = 0; c < n;) {
        const uint32_t hx = hn.x, C = hx & (kSkPairFlag - 1), two = hx & kSkPairFlag;
        const double inv = ldp(f, hn.y);
        SmAddr zp = w + hn.z;
        SmAddr xd = xs + hn.w;
        const uint32_t* body = rec + 4;
        rec = body + ((two ? 3 * C + 1 + 3u : 2 * C + 3u) & ~3u);
        hn = *reinterpret_cast<const uint4*>(rec);
        double acc = lds(zp);
        c += two ? 2 : 1;
        switch (hx) {
            case 0: break;
            case 1: acc = sk_back_column<1>(body, f, w, acc); break;
            case 2: acc = sk_back_column<2>(body, f, w, acc); break;
            case 3: acc = sk_back_column<3>(body, f, w, acc); break;
            case 4: acc = sk_back_column<4>(body, f, w, acc); break;
            case 5: acc = sk_back_column<5>(body, f, w, acc); break;
            case 6: acc = sk_back_column<6>(body, f, w, acc); break;
            case 7: acc = sk_back_column<7>(body, f, w, acc); break;
            case 8: acc = sk_back_column<8>(body, f, w, acc); break;
            case kSkPairFlag | 1: acc = sk_back_column2<1>(body, f, w, xs, acc); break;
            case kSkPairFlag | 2: acc = sk_back_column2<2>(body, f, w, xs, acc); break;
            case kSkPairFlag | 3: acc = sk_back_column2<3>(body, f, w, xs, acc); break;
            case kSkPairFlag | 4: acc = sk_back_column2<4>(body, f, w, xs, acc); break;
            case kSkPairFlag | 5: acc = sk_back_column2<5>(body, f, w, xs, acc); break;
            case kSkPairFlag | 6: acc = sk_back_column2<6>(body, f, w, xs, acc); break;
            case kSkPairFlag | 7: acc = sk_back_column2<7>(body, f, w, xs, acc); break;
            case kSkPairFlag | 8: acc = sk_back_column2<8>(body, f, w, xs, acc); break;
            default:  // single columns with more than 8 entries below the diagonal
                for (uint32_t a = C; a-- > 0;) acc = fma(-ldp(f, body[a]), ldp(w, body[C + a]), acc);
                break;
        }
        const double z = acc * inv;
        sts(zp, z);
        sts(xd, z);
    }
}

__device__ __forceinline__ uint64_t sk_trace_push(uint64_t h, uint32_t code) { return h * 3ull + code + 1ull; }

// Stages one sketch's inputs in the interleaved layout; returns the sketch's scale (1 in plain mode).
// Plain mode: the caller's (already scaled and perturbed) rows go straight in with 8-byte asynchronous copies: all of a
// sketch's loads are in flight at once and the thread waits once (with one warp or two per SM nothing else would hide the
// DRAM latency of a load-then-store loop).  Raw mode (SkRaw): the whole variable row (and the parameter row unless shared)
// is staged in the g and H regions first, then scale, scaling and perturbation run exactly as fk_batch_prepare_kernel does.
__device__ __forceinline__ double sk_stage_inputs(const SkProgram& P, const SkRaw& R, const uint32_t* tab, SmAddr base, SmAddr xp, uint32_t sk,
                                                  const double* __restrict__ vars_all, const double* __restrict__ params_all) {
    const uint32_t n = P.n;
    if (R.raw_vars == nullptr) {
        const double* vars = vars_all + (size_t)sk * P.n_vars;
        const double* params = params_all + (size_t)sk * P.n_expr;
        for (uint32_t i = 0; i < n; i++) cp_async8(xp + (i << 8), vars + tab[P.off_free + i]);
        for (uint32_t i = 0; i < P.nfix; i++) cp_async8(base + ((P.fx + i) << 8), vars + tab[P.off_fix + i]);
        for (uint32_t i = 0; i < P.npar; i++) cp_async8(base + ((P.pr + i) << 8), params + tab[P.off_par + i]);
        asm volatile("cp.async.commit_group;\n cp.async.wait_group 0;" ::: "memory");
        return 1.0;
    }
    SmAddr S = base + (P.w << 8);  // scratch: g and H regions, n + nnz(L) entries (sk_raw_fits)
    const double* rv = R.raw_vars + (size_t)sk * P.n_vars;
    const double* rp = R.raw_param + (R.shared_param ? 0 : (size_t)sk * P.n_expr);
    for (uint32_t i = 0; i < P.n_vars; i++) cp_async8(S + (i << 8), rv + i);
    if (!R.shared_param)
        for (uint32_t e = 0; e < P.n_expr; e++) cp_async8(S + ((P.n_vars + e) << 8), rp + e);
    asm volatile("cp.async.commit_group;\n cp.async.wait_group 0;" ::: "memory");
    // assemble/mod.rs:32-44 via utils.rs:12-19: all variables left to right, then the distance parameters in expression order
    double sum = 0.0;
    uint32_t cnt = P.n_vars;
    {
        uint32_t i = 0;
        for (; i + 8 <= P.n_vars; i += 8) {
            double v[8];
#pragma unroll
            for (int u = 0; u < 8; u++) v[u] = ldp(S, (i + u) << 8);
#pragma unroll
            for (int u = 0; u < 8; u++) sum = sum + v[u] * v[u];
        }
        for (; i < P.n_vars; i++) {
            const double v = ldp(S, i << 8);
            sum = sum + v * v;
        }
    }
    // (The loops below work on four or eight items at a time with every load in front of the arithmetic: one warp per 32 sketches
    // does this while nothing else runs in its CTA, and item-by-item each iteration was a chain of two or three dependent L1 / shared
    // loads in front of its FP64 operations -- 21k cycles per CTA: one launch over 65,536 raw trusses took 980 us against 905 us on
    // prepared inputs; 948 us now, fk_batch_system_solve 1,092 -> 1,067 us per call.  Operations and their order per sketch are unchanged.)
    auto is_distance = [](uint32_t kd) { return kd == FK_POINT_POINT_DISTANCE || kd == FK_POINT_LINE_DISTANCE; };
    {
        uint32_t e = 0;
        for (; e + 8 <= P.n_expr; e += 8) {
            uint32_t kd[8];
            double q[8];
#pragma unroll
            for (int u = 0; u < 8; u++) {
                kd[u] = __ldg(R.kinds + e + u);
                q[u] = R.shared_param ? __ldg(rp + e + u) : ldp(S, (P.n_vars + e + u) << 8);
            }
#pragma unroll
            for (int u = 0; u < 8; u++)
                if (is_distance(kd[u])) {
                    sum = sum + q[u] * q[u];
                    cnt++;
                }
        }
        for (; e < P.n_expr; e++) {
            const uint32_t kd = __ldg(R.kinds + e);
            if (is_distance(kd)) {
                const double q = R.shared_param ? __ldg(rp + e) : ldp(S, (P.n_vars + e) << 8);
                sum = sum + q * q;
                cnt++;
            }
        }
    }
    const double scale = sqrt(sum / (double)cnt);
    const double recip = 1.0 / scale;
    auto perturbed = [&](double col, uint32_t j) {  // assemble/mod.rs:113-124
        return j == kNone ? col : col + (col * (1.0 / 8196.0) * __ldg(R.draws + 2 * j) + (1.0 / 65568.0) * __ldg(R.draws + 2 * j + 1));
    };
    // count variables listed at tab[off_tab ..], their draw positions in draw_idx, into entries entry0.. of the region dst
    auto stage_vars = [&](uint32_t count, uint32_t off_tab, const uint32_t* __restrict__ draw_idx, SmAddr dst, uint32_t entry0) {
        uint32_t c = 0;
        for (; c + 4 <= count; c += 4) {
            uint32_t j[4];
            double col[4], d0[4], d1[4], out[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                j[u] = __ldg(draw_idx + c + u);
                col[u] = ldp(S, tab[off_tab + c + u] << 8);
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {  // (no draw: any valid element, unused)
                d0[u] = __ldg(R.draws + (j[u] == kNone ? 0u : 2u * j[u]));
                d1[u] = __ldg(R.draws + (j[u] == kNone ? 0u : 2u * j[u] + 1u));
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const double v = col[u] * recip;
                out[u] = j[u] == kNone ? v : v + (v * (1.0 / 8196.0) * d0[u] + (1.0 / 65568.0) * d1[u]);
            }
#pragma unroll
            for (int u = 0; u < 4; u++) stp(dst, (entry0 + c + u) << 8, out[u]);
        }
        for (; c < count; c++) stp(dst, (entry0 + c) << 8, perturbed(ldp(S, tab[off_tab + c] << 8) * recip, __ldg(draw_idx + c)));
    };
    stage_vars(n, P.off_free, R.free_draw, xp, 0u);
    stage_vars(P.nfix, P.off_fix, R.fix_draw, base, P.fx);
    {
        uint32_t i = 0;
        for (; i + 4 <= P.npar; i += 4) {
            uint32_t kd[4];
            double q[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const uint32_t e = tab[P.off_par + i + u];
                kd[u] = __ldg(R.kinds + e);
                q[u] = R.shared_param ? __ldg(rp + e) : ldp(S, (P.n_vars + e) << 8);
            }
#pragma unroll
            for (int u = 0; u < 4; u++) stp(base, (P.pr + i + u) << 8, is_distance(kd[u]) ? recip * q[u] : q[u]);
        }
        for (; i < P.npar; i++) {
            const uint32_t e = tab[P.off_par + i];
            const uint32_t kd = __ldg(R.kinds + e);
            const double q = R.shared_param ? __ldg(rp + e) : ldp(S, (P.n_vars + e) << 8);
            stp(base, (P.pr + i) << 8, is_distance(kd) ? recip * q : q);
        }
    }
    return scale;
}

constexpr int kSkMaxWarps = 4;

__global__ void __launch_bounds__(32 * kSkMaxWarps)
fk_batch_lm_sketch_kernel(const SkProgram P, const SkRaw R, uint32_t n_sketches, const double* __restrict__ vars_all,
                          const double* __restrict__ params_all, double* __restrict__ free_out, fk_report* __restrict__ reports) {
    extern __shared__ __align__(16) char sk_smem[];
    // the tables, once per CTA
    uint32_t* const tab = reinterpret_cast<uint32_t*>(sk_smem);
    for (uint32_t i = threadIdx.x; i < P.tab_words / 4; i += blockDim.x)
        reinterpret_cast<uint4*>(tab)[i] = __ldg(reinterpret_cast<const uint4*>(P.tab) + i);
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u, warp = __shfl_sync(0xFFFFFFFFu, threadIdx.x >> 5, 0);  // (lane 0's copy: nvcc then knows it is warp-uniform)
    const uint32_t sketch = (blockIdx.x * (blockDim.x >> 5) + warp) * 32u + lane;
    if (sketch - lane >= n_sketches) return;  // a whole warp without work
    const bool valid = sketch < n_sketches;
    const uint32_t sk = valid ? sketch : n_sketches - 1;  // idle lanes shadow the last sketch and store nothing
    const SmAddr base = (SmAddr)__cvta_generic_to_shared(sk_smem) + P.tab_words * 4 + warp * P.entries * 256u + lane * 8u;
    const uint32_t n = P.n;

    // accepted / trial point: the two roles swap per lane on accept (a register exchange instead of a copy)
    SmAddr xp = base + (P.xa << 8);
    SmAddr xsp = base + (P.xb << 8);
    const SmAddr w = base + (P.w << 8);
    const SmAddr f = base + (P.f << 8);
    const SmAddr fx = base + (P.fx << 8);
    const SmAddr pr = base + (P.pr << 8);

    const double scale = sk_stage_inputs(P, R, tab, base, xp, sk, vars_all, params_all);

    double ssr = 0.0, lambda = 0.5, dn = 0.0;  // lm.rs:108
    uint32_t exit_reason = FK_EXIT_MAX_OUTER, outer_iters = 0, factorizations = 0, accepted = 0;
    uint64_t trace = 0;
    bool active = valid;
    int fstat = 0;
    // What the evaluation at the top of the loop is for (warp-uniform): the starting point (lm.rs:80-106), a
    // trial point (lm.rs:148-149 and, for an accepted one, lm.rs:173-185), or the accepted point again after a
    // rejected / unsolved step of some sketch of the warp (its H and g were consumed by the factorisation;
    // sketches that accepted recompute the values they already hold).
    enum { kInit, kTrial, kRestore } mode = kInit;
    SmAddr xe = xp;

    for (;;) {
        // ---- residuals, g = -J^T r (into w), H = J^T J (into f) at xe; s = sum of squared residuals ----------
        double s = 0.0;
        {
            uint32_t i = 0;
            for (; i + 8 <= n; i += 8)
#pragma unroll
                for (int u = 0; u < 8; u++) stp(w, (i + u) << 8, 0.0);
            for (; i < n; i++) stp(w, i << 8, 0.0);
            for (i = 0; i + 8 <= P.lnnz; i += 8)
#pragma unroll
                for (int u = 0; u < 8; u++) stp(f, (i + u) << 8, 0.0);
            for (; i < P.lnnz; i++) stp(f, i << 8, 0.0);
            const uint32_t* rec = tab + P.off_eval;
            uint4 h = *reinterpret_cast<const uint4*>(rec);
            for (uint32_t r = 0; r < P.m;) {
                const uint32_t* cur = rec;
                const uint32_t* rec1 = cur + (h.x >> 16);
                const uint4 h1 = *reinterpret_cast<const uint4*>(rec1);  // next row's header (a padding record follows the last row)
                const bool two = r + 1 < P.m && (h.x & 0x1FFu) <= 1u && (h1.x & 0x1FFu) == (h.x & 0x1FFu);
#define FK_SK_ROW(K)                                                          \
    case K: sk_eval_row<K, false>(cur, h, xe, fx, pr, w, f, s); break;        \
    case 0x100 | K: sk_eval_row<K, true>(cur, h, xe, fx, pr, w, f, s); break;
#define FK_SK_ROW2(K)                                                         \
    case K:                                                                   \
        if (two) sk_eval_rows2<K>(cur, h, rec1, h1, xe, pr, w, f, s);         \
        else sk_eval_row<K, false>(cur, h, xe, fx, pr, w, f, s);              \
        break;                                                                \
    case 0x100 | K: sk_eval_row<K, true>(cur, h, xe, fx, pr, w, f, s); break;
                switch (h.x & 0x1FFu) {  // (pairs of rows only for the kinds whose two-row body fits the register file)
                    FK_SK_ROW2(0) FK_SK_ROW2(1) FK_SK_ROW(2) FK_SK_ROW(3) FK_SK_ROW(4) FK_SK_ROW(5)
                    FK_SK_ROW(6) FK_SK_ROW(7) FK_SK_ROW(8) FK_SK_ROW(9) FK_SK_ROW(10) FK_SK_ROW(11) FK_SK_ROW(12)
                    default: break;
                }
#undef FK_SK_ROW
#undef FK_SK_ROW2
                if (two) {
                    rec = rec1 + (h1.x >> 16);
                    h = *reinterpret_cast<const uint4*>(rec);
                    r += 2;
                } else {
                    rec = rec1;
                    h = h1;
                    r += 1;
                }
            }
        }
        bool restore = false;
        if (mode == kInit) {
            ssr = s;
            if (ssr < 1e-8) {  // lm.rs:110-112 on the first outer iteration
                exit_reason = FK_EXIT_CONVERGED_RESIDUAL;
                active = false;
            } else {
                outer_iters = 1;
            }
        } else if (mode == kTrial && active) {
            factorizations++;
            if (fstat == 1) {  // lm.rs:134-137 (`!solved`)
                lambda *= 8.0;
                trace = sk_trace_push(trace, 0);
                restore = true;
            } else if (fstat == 0 && dn < 1e-12) {  // lm.rs:139-142
                exit_reason = FK_EXIT_SMALL_STEP;
                active = false;
            } else {
                const double ssr_s = fstat == 0 ? s : NAN;
                if (ssr_s < ssr) {  // lm.rs:151 (strict; NaN rejects)
                    lambda *= 0.125;
                    if (lambda < 1e-50) lambda = 1e-50;
                    accepted++;
                    trace = sk_trace_push(trace, 1);
                    SmAddr tmp = xp; xp = xsp; xsp = tmp;
                    const bool stalled = (ssr - ssr_s) / ssr <= 1e-6;  // lm.rs:164-168
                    ssr = ssr_s;
                    if (stalled) {
                        exit_reason = FK_EXIT_STALLED;
                        active = false;
                    } else if (outer_iters == 100) {
                        active = false;  // FK_EXIT_MAX_OUTER: the 100th outer iteration has ended
                    } else if (ssr < 1e-8) {  // lm.rs:109-112
                        exit_reason = FK_EXIT_CONVERGED_RESIDUAL;
                        active = false;
                    } else {
                        outer_iters++;
                    }
                } else {  // lm.rs:187-190
                    lambda *= 2.0;
                    trace = sk_trace_push(trace, 2);
                    restore = true;
                }
            }
        }
        if (mode != kRestore && __any_sync(0xFFFFFFFFu, restore && active)) {
            mode = kRestore;
            xe = xp;
            continue;
        }
        if (active && !isfinite(lambda)) {
            exit_reason = FK_EXIT_LAMBDA_OVERFLOW;
            active = false;
        }
        if (!__any_sync(0xFFFFFFFFu, active)) break;

        // ---- one iteration of the damping loop (lm.rs:115-146) for every sketch of the warp ----------------------
        const double sl = sqrt(lambda);  // lm.rs:119-125
        const double lam2 = sl * sl;
        {   // LDLt of (H + lam2 I) in place (column k keeps (L D)(i,k), and 1 / D(k) on its diagonal slot) and the
            // forward substitution of g in w.  fstat: kind of the FIRST bad pivot in column order (tile kernel's rule).
            fstat = 0;
            const uint32_t* rec = tab + P.off_factor;
            uint4 hn = *reinterpret_cast<const uint4*>(rec);
            for (uint32_t c = 0; c < n;) {
                const uint32_t C = hn.x & (kSkPairFlag - 1), two = hn.x & kSkPairFlag;
                SmAddr dp = f + hn.y;
                const double wk = ldp(w, hn.z);
                const uint32_t* body = rec + 4;
                rec = body + ((2 * C + C * (C + 1) / 2 + 3u) & ~3u);
                hn = *reinterpret_cast<const uint4*>(rec);  // next record's header
                const double d = lds(dp) + lam2;
                if (fstat == 0 && !(d > 0.0 && d < INFINITY)) fstat = d != d ? 2 : 1;
                const double inv = sk_rcp(d);
                sts(dp, inv);
                c += two ? 2 : 1;
                if (two) {
                    switch (C) {
                        case 1: sk_column2<1>(body, f, w, wk, inv, lam2, fstat); break;
                        case 2: sk_column2<2>(body, f, w, wk, inv, lam2, fstat); break;
                        case 3: sk_column2<3>(body, f, w, wk, inv, lam2, fstat); break;
                        case 4: sk_column2<4>(body, f, w, wk, inv, lam2, fstat); break;
                        case 5: sk_column2<5>(body, f, w, wk, inv, lam2, fstat); break;
                        case 6: sk_column2<6>(body, f, w, wk, inv, lam2, fstat); break;
                        case 7: sk_column2<7>(body, f, w, wk, inv, lam2, fstat); break;
                        default: sk_column2<8>(body, f, w, wk, inv, lam2, fstat); break;
                    }
                    continue;
                }
                switch (C) {
                    case 0: break;
                    case 1: sk_column<1>(body, f, w, wk, inv); break;
                    case 2: sk_column<2>(body, f, w, wk, inv); break;
                    case 3: sk_column<3>(body, f, w, wk, inv); break;
                    case 4: sk_column<4>(body, f, w, wk, inv); break;
                    case 5: sk_column<5>(body, f, w, wk, inv); break;
                    case 6: sk_column<6>(body, f, w, wk, inv); break;
                    case 7: sk_column<7>(body, f, w, wk, inv); break;
                    case 8: sk_column<8>(body, f, w, wk, inv); break;
                    default: sk_column_generic(body, C, f, w, wk, inv); break;
                }
            }
        }
        sk_back_solve(tab + P.off_back, n, f, w, xsp);
        {   // lm.rs:139 (sum of squared steps, in variable order) and lm.rs:144-146 (trial point)
            dn = 0.0;
            uint32_t i = 0;
            for (; i + 4 <= n; i += 4) {
                double d[4], x0[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    d[u] = ldp(xsp, (i + u) << 8);
                    x0[u] = ldp(xp, (i + u) << 8);
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    dn = dn + d[u] * d[u];
                    stp(xsp, (i + u) << 8, x0[u] + d[u]);
                }
            }
            for (; i < n; i++) {
                const double d = ldp(xsp, i << 8);
                dn = dn + d * d;
                stp(xsp, i << 8, ldp(xp, i << 8) + d);
            }
        }
        mode = kTrial;
        xe = xsp;
    }

    if (!valid) return;
    double* out = free_out + (size_t)sketch * n;
    if (R.raw_vars == nullptr) {
        for (uint32_t i = 0; i < n; i++) out[i] = ldp(xp, i << 8);
    } else {  // system.variables[var] = system_scale * x[k] (assemble/mod.rs:161-166)
        for (uint32_t i = 0; i < n; i++) out[i] = scale * ldp(xp, i << 8);
        if (R.scales) R.scales[sketch] = scale;
    }
    fk_report rep;
    rep.exit_reason = exit_reason;
    rep.outer_iters = outer_iters;
    rep.factorizations = factorizations;
    rep.accepted = accepted;
    rep.ssr = ssr;
    rep.lambda = lambda;
    rep.trace_hash = trace;
    reports[sketch] = rep;
}

// ---- warp-pair variant ---------------------------------------------------------------------------------------
// When a sketch's state is so large that only one or two warps fit an SM (the 20-point truss: 93 KB per warp), two of
// the SM's four schedulers idle and the one warp per scheduler issues a dependent instruction every ~4 cycles.  Here a
// CTA is TWO warps working on the SAME 32 sketches (thread l of both warps serves sketch l):
//   * evaluation: the leader computes a row (loads, sqrt / divide / atan2) and leaves gradient and residual in a
//     double-buffered staging area; the helper adds them into g and H while the leader is already on the next row;
//   * factorisation: both warps read the pivot column (or column pair) into registers, each applies its share of the
//     updates;
//   * back substitution and the LM bookkeeping stay with the leader (dependent chains), the helper clears g and H
//     for the next evaluation meanwhile.
// One CTA barrier per row and per factorisation step (one column or a column pair) hands the data over.  Operations and
// their order per entry are those of the solo kernel, so the results are bit-identical.
#ifndef FK_SK_LEADER_PCT
#define FK_SK_LEADER_PCT 20  // (30: 71.7, 20: 72.7, 10: 72.5 M sketches/s on the 65,536-truss batch)
#endif
constexpr uint32_t kPairExtra = 38;  // entries behind the solo state: 2 steps x 2 rows x (8 gradients + residual) staging, lambda, pad

template <int KIND, bool SPECIAL>
__device__ __forceinline__ void sk_row_produce(const uint32_t* rec, const uint4 h0, SmAddr x, SmAddr fx, SmAddr pr, SmAddr stage,
                                               double& ssr) {
    constexpr int A = sk_arity(KIND);
    uint32_t t[(2 + A + 3) / 4 * 4];
    t[0] = h0.x; t[1] = h0.y; t[2] = h0.z; t[3] = h0.w;
#pragma unroll
    for (int i = 1; i < (2 + A + 3) / 4; i++) {
        const uint4 q = reinterpret_cast<const uint4*>(rec)[i];
        t[4 * i] = q.x; t[4 * i + 1] = q.y; t[4 * i + 2] = q.z; t[4 * i + 3] = q.w;
    }
    double v[8], g[8];
#pragma unroll
    for (int s = 0; s < 8; s++) v[s] = 0.0;
#pragma unroll
    for (int s = 0; s < A; s++) {
        const uint32_t src = t[2 + s];
        if (SPECIAL) v[s] = (src >> 31) ? ldp(fx, src & 0x7FFFFFFFu) : ldp(x, src);
        else v[s] = ldp(x, src);
    }
    const double param = sk_has_param(KIND) ? ldp(pr, t[1]) : 0.0;
    const double r = dev::eval_expression(KIND, v, param, g);
    ssr = ssr + r * r;  // lm.rs:195-197: sequential, not fused
#pragma unroll
    for (int s = 0; s < A; s++) stp(stage, (uint32_t)s << 8, g[s]);
    stp(stage, 8u << 8, -r);
}

// Two consecutive rows of the same kind without fixed slots: their loads and their sqrt / divide chains are independent,
// so issuing them together hides most of one row's latency behind the other's.
template <int KIND>
__device__ __forceinline__ void sk_rows_produce2(const uint32_t* rec0, const uint4 h0, const uint32_t* rec1, const uint4 h1, SmAddr x,
                                                 SmAddr pr, SmAddr st0, SmAddr st1, double& ssr) {
    constexpr int A = sk_arity(KIND);
    constexpr int NWD = (2 + A + 3) / 4 * 4;
    uint32_t t0[NWD], t1[NWD];
    t0[0] = h0.x; t0[1] = h0.y; t0[2] = h0.z; t0[3] = h0.w;
    t1[0] = h1.x; t1[1] = h1.y; t1[2] = h1.z; t1[3] = h1.w;
#pragma unroll
    for (int i = 1; i < NWD / 4; i++) {
        const uint4 q0 = reinterpret_cast<const uint4*>(rec0)[i], q1 = reinterpret_cast<const uint4*>(rec1)[i];
        t0[4 * i] = q0.x; t0[4 * i + 1] = q0.y; t0[4 * i + 2] = q0.z; t0[4 * i + 3] = q0.w;
        t1[4 * i] = q1.x; t1[4 * i + 1] = q1.y; t1[4 * i + 2] = q1.z; t1[4 * i + 3] = q1.w;
    }
    double v0[8], v1[8], g0[8], g1[8];
#pragma unroll
    for (int s = 0; s < 8; s++) v0[s] = v1[s] = 0.0;
#pragma unroll
    for (int s = 0; s < A; s++) {
        v0[s] = ldp(x, t0[2 + s]);
        v1[s] = ldp(x, t1[2 + s]);
    }
    const double p0 = sk_has_param(KIND) ? ldp(pr, t0[1]) : 0.0;
    const double p1 = sk_has_param(KIND) ? ldp(pr, t1[1]) : 0.0;
    const double r0 = dev::eval_expression(KIND, v0, p0, g0);
    const double r1 = dev::eval_expression(KIND, v1, p1, g1);
    ssr = ssr + r0 * r0;  // lm.rs:195-197: sequential, not fused
    ssr = ssr + r1 * r1;
#pragma unroll
    for (int s = 0; s < A; s++) {
        stp(st0, (uint32_t)s << 8, g0[s]);
        stp(st1, (uint32_t)s << 8, g1[s]);
    }
    stp(st0, 8u << 8, -r0);
    stp(st1, 8u << 8, -r1);
}

template <int KIND, bool SPECIAL>
__device__ __forceinline__ void sk_row_consume(const uint32_t* rec, SmAddr stage, SmAddr w, SmAddr f) {
    constexpr int A = sk_arity(KIND);
    constexpr int NP = A * (A + 1) / 2;
    constexpr int NW = 2 + 2 * A + NP;
    uint32_t t[(NW + 3) / 4 * 4];
    ld_words<NW>(rec, t);
    SmAddr gp[A];
    SmAddr hp[NP];
    double gv[A], hv[NP], g[A];
#pragma unroll
    for (int s = 0; s < A; s++) {
        const uint32_t o = t[2 + A + s];
        gp[s] = w + o;
        gv[s] = (!SPECIAL || o != kNone) ? lds(gp[s]) : 0.0;
    }
#pragma unroll
    for (int q = 0; q < NP; q++) {
        const uint32_t o = t[2 + 2 * A + q];
        hp[q] = f + o;
        hv[q] = (!SPECIAL || o != kNone) ? lds(hp[q]) : 0.0;
    }
#pragma unroll
    for (int s = 0; s < A; s++) g[s] = ldp(stage, (uint32_t)s << 8);
    const double nr = ldp(stage, 8u << 8);
#pragma unroll
    for (int s = 0; s < A; s++)
        if (!SPECIAL || t[2 + A + s] != kNone) sts(gp[s], fma(g[s], nr, gv[s]));
    int q = 0;
#pragma unroll
    for (int a = 0; a < A; a++)
#pragma unroll
        for (int b = 0; b <= a; b++, q++)
            if (!SPECIAL || t[2 + 2 * A + q] != kNone) sts(hp[q], fma(g[a], g[b], hv[q]));
}

// The leader's share of a column's NT targets: less than half, because the leader also carries the pivot checks and,
// alone, the back substitution, during which the helper waits (ncu: the helper spent 21 % of its time at that barrier
// with an even split).
__host__ __device__ constexpr int sk_leader_share(int nt) { return (nt * FK_SK_LEADER_PCT + 50) / 100; }

// One part of a column's updates (HALF 0: the leader's first sk_leader_share(NT) targets in the order "pairs (a, b),
// then the C right-hand-side entries", HALF 1: the rest).  Both parts read the whole column.
template <int C, int HALF>
__device__ __forceinline__ void sk_column_half(const uint32_t* body, SmAddr f, SmAddr w, double wk, double inv) {
    constexpr int NP = C * (C + 1) / 2, NT = NP + C, H0 = sk_leader_share(NT);
    constexpr int LO = HALF ? H0 : 0, HI = HALF ? NT : H0;
    uint32_t t[(2 * C + NP + 3) / 4 * 4];
    ld_words<2 * C + NP>(body, t);
    double l[C], s[C], wv[C], d[NP];
    SmAddr wp[C];
    SmAddr dp[NP];
#pragma unroll
    for (int a = 0; a < C; a++) l[a] = ldp(f, t[a]);
#pragma unroll
    for (int q = 0; q < NP; q++)
        if (q >= LO && q < HI) {
            dp[q] = f + t[2 * C + q];
            d[q] = lds(dp[q]);
        }
#pragma unroll
    for (int a = 0; a < C; a++)
        if (NP + a >= LO && NP + a < HI) {
            wp[a] = w + t[C + a];
            wv[a] = lds(wp[a]);
        }
#pragma unroll
    for (int a = 0; a < C; a++) s[a] = -(l[a] * inv);
    int q = 0;
#pragma unroll
    for (int a = 0; a < C; a++)
#pragma unroll
        for (int b = 0; b <= a; b++, q++)
            if (q >= LO && q < HI) sts(dp[q], fma(s[a], l[b], d[q]));
#pragma unroll
    for (int a = 0; a < C; a++)
        if (NP + a >= LO && NP + a < HI) sts(wp[a], fma(s[a], wk, wv[a]));
}

__device__ __forceinline__ void sk_column_generic_half(const uint32_t* t, uint32_t C, int half, SmAddr f, SmAddr w, double wk, double inv) {
    const uint32_t NP = C * (C + 1) / 2, NT = NP + C, H0 = (uint32_t)sk_leader_share((int)NT);
    const uint32_t lo = half ? H0 : 0, hi = half ? NT : H0;
    uint32_t q = 0;
    for (uint32_t a = 0; a < C; a++) {
        const double la = ldp(f, t[a]);
        const double sa = -(la * inv);
        for (uint32_t b = 0; b <= a; b++, q++) {
            if (q < lo || q >= hi) continue;
            SmAddr dst = f + t[2 * C + q];
            const double lb = b == a ? la : ldp(f, t[b]);
            sts(dst, fma(sa, lb, lds(dst)));
        }
        if (NP + a >= lo && NP + a < hi) {
            SmAddr wr = w + t[C + a];
            sts(wr, fma(sa, wk, lds(wr)));
        }
    }
}

// One part of a pair record's updates (columns k and k+1, see sk_column2).  Both warps read column k's entries and apply
// its update to column k+1's pivot, entries and right-hand side entry, then take 1 / d(k+1); the remaining targets
// ((a, b) with a >= b >= 1, then the w rows a >= 1) receive both updates and are split as sk_column_half splits a column's.
// The step's barrier is part of the body: the helper reads column k+1's values and the pivot of column k during the step,
// so HALF 0 (the leader), which also checks column k+1's pivot, stores them (and 1 / d of both pivots; dpk: column k's
// diagonal) only after the barrier.  Only the back substitution reads them afterwards.
template <int C, int HALF>
__device__ __forceinline__ void sk_column2_half(const uint32_t* body, SmAddr f, SmAddr w, double wk, double inv, double lam2, int& fstat,
                                                SmAddr dpk) {
    constexpr int NP = C * (C + 1) / 2, NP1 = C * (C - 1) / 2, NT = NP1 + C - 1, H0 = sk_leader_share(NT);
    constexpr int LO = HALF ? H0 : 0, HI = HALF ? NT : H0;
    uint32_t t[(2 * C + NP + 3) / 4 * 4];
    ld_words<2 * C + NP>(body, t);
    double l[C], s[C], s1[C], wv[C], d[NP];
    SmAddr wp[C];
    SmAddr dp[NP];
#pragma unroll
    for (int a = 0; a < C; a++) l[a] = ldp(f, t[a]);
#pragma unroll
    for (int a = 0; a < C; a++) {
        dp[sk_tri(a, 0)] = f + t[2 * C + sk_tri(a, 0)];
        d[sk_tri(a, 0)] = lds(dp[sk_tri(a, 0)]);
    }
    wp[0] = w + t[C];
    wv[0] = lds(wp[0]);
#pragma unroll
    for (int a = 1; a < C; a++)
#pragma unroll
        for (int b = 1; b <= a; b++)
            if (sk_tri(a - 1, b - 1) >= LO && sk_tri(a - 1, b - 1) < HI) {
                dp[sk_tri(a, b)] = f + t[2 * C + sk_tri(a, b)];
                d[sk_tri(a, b)] = lds(dp[sk_tri(a, b)]);
            }
#pragma unroll
    for (int a = 1; a < C; a++)
        if (NP1 + a - 1 >= LO && NP1 + a - 1 < HI) {
            wp[a] = w + t[C + a];
            wv[a] = lds(wp[a]);
        }
#pragma unroll
    for (int a = 0; a < C; a++) s[a] = -(l[a] * inv);
#pragma unroll
    for (int a = 0; a < C; a++) {
        d[sk_tri(a, 0)] = fma(s[a], l[0], d[sk_tri(a, 0)]);
#pragma unroll
        for (int b = 1; b <= a; b++)
            if (sk_tri(a - 1, b - 1) >= LO && sk_tri(a - 1, b - 1) < HI) d[sk_tri(a, b)] = fma(s[a], l[b], d[sk_tri(a, b)]);
    }
    wv[0] = fma(s[0], wk, wv[0]);
#pragma unroll
    for (int a = 1; a < C; a++)
        if (NP1 + a - 1 >= LO && NP1 + a - 1 < HI) wv[a] = fma(s[a], wk, wv[a]);
    const double d1 = d[0] + lam2;
    if (HALF == 0 && fstat == 0 && !(d1 > 0.0 && d1 < INFINITY)) fstat = d1 != d1 ? 2 : 1;
    const double inv1 = sk_rcp(d1);
#pragma unroll
    for (int a = 1; a < C; a++) s1[a] = -(d[sk_tri(a, 0)] * inv1);
#pragma unroll
    for (int a = 1; a < C; a++)
#pragma unroll
        for (int b = 1; b <= a; b++)
            if (sk_tri(a - 1, b - 1) >= LO && sk_tri(a - 1, b - 1) < HI) sts(dp[sk_tri(a, b)], fma(s1[a], d[sk_tri(b, 0)], d[sk_tri(a, b)]));
#pragma unroll
    for (int a = 1; a < C; a++)
        if (NP1 + a - 1 >= LO && NP1 + a - 1 < HI) sts(wp[a], fma(s1[a], wv[0], wv[a]));
    __syncthreads();
    if (HALF == 0) {
        sts(dpk, inv);
        sts(dp[0], inv1);
        sts(wp[0], wv[0]);
#pragma unroll
        for (int a = 1; a < C; a++) sts(dp[sk_tri(a, 0)], d[sk_tri(a, 0)]);
    }
}

template <int HALF>
__device__ __forceinline__ void sk_column_dispatch_half(uint32_t C, const uint32_t* body, SmAddr f, SmAddr w, double wk, double inv) {
    switch (C) {
        case 0: break;
        case 1: sk_column_half<1, HALF>(body, f, w, wk, inv); break;
        case 2: sk_column_half<2, HALF>(body, f, w, wk, inv); break;
        case 3: sk_column_half<3, HALF>(body, f, w, wk, inv); break;
        case 4: sk_column_half<4, HALF>(body, f, w, wk, inv); break;
        case 5: sk_column_half<5, HALF>(body, f, w, wk, inv); break;
        case 6: sk_column_half<6, HALF>(body, f, w, wk, inv); break;
        case 7: sk_column_half<7, HALF>(body, f, w, wk, inv); break;
        case 8: sk_column_half<8, HALF>(body, f, w, wk, inv); break;
        default: sk_column_generic_half(body, C, HALF, f, w, wk, inv); break;
    }
}

// A pair record (1 <= C <= kSkPairMaxC); ends with the step's barrier.
template <int HALF>
__device__ __forceinline__ void sk_column2_dispatch_half(uint32_t C, const uint32_t* body, SmAddr f, SmAddr w, double wk, double inv,
                                                         double lam2, int& fstat, SmAddr dpk) {
    switch (C) {
        case 1: sk_column2_half<1, HALF>(body, f, w, wk, inv, lam2, fstat, dpk); break;
        case 2: sk_column2_half<2, HALF>(body, f, w, wk, inv, lam2, fstat, dpk); break;
        case 3: sk_column2_half<3, HALF>(body, f, w, wk, inv, lam2, fstat, dpk); break;
        case 4: sk_column2_half<4, HALF>(body, f, w, wk, inv, lam2, fstat, dpk); break;
        case 5: sk_column2_half<5, HALF>(body, f, w, wk, inv, lam2, fstat, dpk); break;
        case 6: sk_column2_half<6, HALF>(body, f, w, wk, inv, lam2, fstat, dpk); break;
        case 7: sk_column2_half<7, HALF>(body, f, w, wk, inv, lam2, fstat, dpk); break;
        default: sk_column2_half<8, HALF>(body, f, w, wk, inv, lam2, fstat, dpk); break;
    }
}

__global__ void __launch_bounds__(64)
fk_batch_lm_sketch_pair_kernel(const SkProgram P, const SkRaw R, uint32_t n_sketches, const double* __restrict__ vars_all,
                               const double* __restrict__ params_all, double* __restrict__ free_out, fk_report* __restrict__ reports) {
    extern __shared__ __align__(16) char sk_smem[];
    __shared__ int ctrl;  // leader -> helper after an evaluation: 0 iterate, 1 evaluate the accepted point again, 2 done
    uint32_t* const tab = reinterpret_cast<uint32_t*>(sk_smem);
    for (uint32_t i = threadIdx.x; i < P.tab_words / 4; i += blockDim.x)
        reinterpret_cast<uint4*>(tab)[i] = __ldg(reinterpret_cast<const uint4*>(P.tab) + i);
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u, role = __shfl_sync(0xFFFFFFFFu, threadIdx.x >> 5, 0);  // (lane 0's copy: nvcc then knows it is warp-uniform)
    const uint32_t sketch = blockIdx.x * 32u + lane;
    const bool valid = sketch < n_sketches;
    const uint32_t sk = valid ? sketch : n_sketches - 1;
    const SmAddr base = (SmAddr)__cvta_generic_to_shared(sk_smem) + P.tab_words * 4 + lane * 8u;
    const uint32_t n = P.n;
    const SmAddr w = base + (P.w << 8);
    const SmAddr f = base + (P.f << 8);
    const SmAddr stage = base + (P.entries << 8);  // [2 steps][2 rows][9] staging, then lambda

    if (role == 1) {
        // ---- helper ---------------------------------------------------------------------------------------
        if (R.raw_vars != nullptr) __syncthreads();  // raw mode: the leader stages the inputs in the g and H regions first
        for (;;) {
            uint32_t i = 0;
            for (; i + 8 <= n; i += 8)
#pragma unroll
                for (int u = 0; u < 8; u++) stp(w, (i + u) << 8, 0.0);
            for (; i < n; i++) stp(w, i << 8, 0.0);
            for (i = 0; i + 8 <= P.lnnz; i += 8)
#pragma unroll
                for (int u = 0; u < 8; u++) stp(f, (i + u) << 8, 0.0);
            for (; i < P.lnnz; i++) stp(f, i << 8, 0.0);
            // rows are taken one at a time, or two at a time when two consecutive rows share a kind and have no fixed
            // slot (the leader evaluates such a pair together); both warps derive the grouping from the same headers
            const uint32_t* rec = tab + P.off_eval;
            uint32_t hx = rec[0];
            for (uint32_t r = 0, step = 0; r < P.m; step++) {
                const uint32_t* cur = rec;
                const uint32_t h = hx;
                const uint32_t* rec1 = cur + (h >> 16);
                const uint32_t h1 = rec1[0];
                const bool two = r + 1 < P.m && (h & 0x1FFu) < 0x100u && (h1 & 0x1FFu) == (h & 0x1FFu);
                SmAddr st0 = stage + ((step & 1u) * 18u << 8);
                SmAddr st1 = st0 + (9u << 8);
                if (two) {
                    rec = rec1 + (h1 >> 16);
                    r += 2;
                } else {
                    rec = rec1;
                    r += 1;
                }
                hx = rec[0];
                __syncthreads();  // the leader has staged this step's row(s)
#define FK_SK_ROW(K)                                                   \
    case K:                                                            \
        sk_row_consume<K, false>(cur, st0, w, f);                      \
        if (two) sk_row_consume<K, false>(rec1, st1, w, f);            \
        break;                                                         \
    case 0x100 | K: sk_row_consume<K, true>(cur, st0, w, f); break;
                switch (h & 0x1FFu) {
                    FK_SK_ROW(0) FK_SK_ROW(1) FK_SK_ROW(2) FK_SK_ROW(3) FK_SK_ROW(4) FK_SK_ROW(5)
                    FK_SK_ROW(6) FK_SK_ROW(7) FK_SK_ROW(8) FK_SK_ROW(9) FK_SK_ROW(10) FK_SK_ROW(11) FK_SK_ROW(12)
                    default: break;
                }
#undef FK_SK_ROW
            }
            __syncthreads();  // g and H complete; the leader has decided
            const int c = ctrl;
            if (c == 2) break;
            if (c == 1) continue;
            const double lam2 = ldp(stage, 36u << 8);
            const uint32_t* frec = tab + P.off_factor;
            uint4 hn = *reinterpret_cast<const uint4*>(frec);
            int fstat_unused = 0;
            for (uint32_t col = 0; col < n;) {
                const uint32_t hx = hn.x, C = hx & (kSkPairFlag - 1);
                const SmAddr dp = f + hn.y;
                const double wk = ldp(w, hn.z);
                const uint32_t* body = frec + 4;
                frec = body + ((2 * C + C * (C + 1) / 2 + 3u) & ~3u);
                hn = *reinterpret_cast<const uint4*>(frec);
                const double inv = sk_rcp(lds(dp) + lam2);  // (the leader stores 1 / d after the step's barrier)
                if (hx & kSkPairFlag) {
                    sk_column2_dispatch_half<1>(C, body, f, w, wk, inv, lam2, fstat_unused, dp);
                    col += 2;
                } else {
                    sk_column_dispatch_half<1>(C, body, f, w, wk, inv);
                    __syncthreads();
                    col += 1;
                }
            }
            __syncthreads();  // the leader is through with the back substitution
        }
        return;
    }

    // ---- leader ---------------------------------------------------------------------------------------------
    SmAddr xp = base + (P.xa << 8);
    SmAddr xsp = base + (P.xb << 8);
    const SmAddr fx = base + (P.fx << 8);
    const SmAddr pr = base + (P.pr << 8);
    const double scale = sk_stage_inputs(P, R, tab, base, xp, sk, vars_all, params_all);
    if (R.raw_vars != nullptr) __syncthreads();  // the helper may clear g and H now

    double ssr = 0.0, lambda = 0.5, dn = 0.0;  // lm.rs:108
    uint32_t exit_reason = FK_EXIT_MAX_OUTER, outer_iters = 0, factorizations = 0, accepted = 0;
    uint64_t trace = 0;
    bool active = valid;
    int fstat = 0;
    enum { kInit, kTrial, kRestore } mode = kInit;
    SmAddr xe = xp;
    for (;;) {
        double s = 0.0;
        {
            const uint32_t* rec = tab + P.off_eval;
            uint4 h = *reinterpret_cast<const uint4*>(rec);
            for (uint32_t r = 0, step = 0; r < P.m; step++) {
                const uint32_t* cur = rec;
                const uint32_t* rec1 = cur + (h.x >> 16);
                const uint4 h1 = *reinterpret_cast<const uint4*>(rec1);
                const bool two = r + 1 < P.m && (h.x & 0x1FFu) < 0x100u && (h1.x & 0x1FFu) == (h.x & 0x1FFu);
                SmAddr st0 = stage + ((step & 1u) * 18u << 8);
                SmAddr st1 = st0 + (9u << 8);
#define FK_SK_ROW(K)                                                                           \
    case K:                                                                                    \
        if (two) sk_rows_produce2<K>(cur, h, rec1, h1, xe, pr, st0, st1, s);                   \
        else sk_row_produce<K, false>(cur, h, xe, fx, pr, st0, s);                             \
        break;                                                                                 \
    case 0x100 | K: sk_row_produce<K, true>(cur, h, xe, fx, pr, st0, s); break;
                switch (h.x & 0x1FFu) {
                    FK_SK_ROW(0) FK_SK_ROW(1) FK_SK_ROW(2) FK_SK_ROW(3) FK_SK_ROW(4) FK_SK_ROW(5)
                    FK_SK_ROW(6) FK_SK_ROW(7) FK_SK_ROW(8) FK_SK_ROW(9) FK_SK_ROW(10) FK_SK_ROW(11) FK_SK_ROW(12)
                    default: break;
                }
#undef FK_SK_ROW
                if (two) {
                    rec = rec1 + (h1.x >> 16);
                    h = *reinterpret_cast<const uint4*>(rec);
                    r += 2;
                } else {
                    rec = rec1;
                    h = h1;
                    r += 1;
                }
                __syncthreads();  // this step's row(s) are staged
            }
        }
        bool restore = false;
        if (mode == kInit) {
            ssr = s;
            if (ssr < 1e-8) {
                exit_reason = FK_EXIT_CONVERGED_RESIDUAL;
                active = false;
            } else {
                outer_iters = 1;
            }
        } else if (mode == kTrial && active) {
            factorizations++;
            if (fstat == 1) {
                lambda *= 8.0;
                trace = sk_trace_push(trace, 0);
                restore = true;
            } else if (fstat == 0 && dn < 1e-12) {
                exit_reason = FK_EXIT_SMALL_STEP;
                active = false;
            } else {
                const double ssr_s = fstat == 0 ? s : NAN;
                if (ssr_s < ssr) {
                    lambda *= 0.125;
                    if (lambda < 1e-50) lambda = 1e-50;
                    accepted++;
                    trace = sk_trace_push(trace, 1);
                    SmAddr tmp = xp; xp = xsp; xsp = tmp;
                    const bool stalled = (ssr - ssr_s) / ssr <= 1e-6;
                    ssr = ssr_s;
                    if (stalled) {
                        exit_reason = FK_EXIT_STALLED;
                        active = false;
                    } else if (outer_iters == 100) {
                        active = false;
                    } else if (ssr < 1e-8) {
                        exit_reason = FK_EXIT_CONVERGED_RESIDUAL;
                        active = false;
                    } else {
                        outer_iters++;
                    }
                } else {
                    lambda *= 2.0;
                    trace = sk_trace_push(trace, 2);
                    restore = true;
                }
            }
        }
        int c = 0;
        if (mode != kRestore && __any_sync(0xFFFFFFFFu, restore && active)) {
            c = 1;
        } else {
            if (active && !isfinite(lambda)) {
                exit_reason = FK_EXIT_LAMBDA_OVERFLOW;
                active = false;
            }
            if (!__any_sync(0xFFFFFFFFu, active)) c = 2;
        }
        const double sl = sqrt(lambda);  // lm.rs:119-125
        const double lam2 = sl * sl;
        if (c == 0) stp(stage, 36u << 8, lam2);
        if (lane == 0) ctrl = c;
        __syncthreads();  // decision published; g and H complete
        if (c == 1) {
            mode = kRestore;
            xe = xp;
            continue;
        }
        if (c == 2) break;
        {
            fstat = 0;
            SmAddr dp_prev = kNone;
            double inv_prev = 0.0;
            const uint32_t* rec = tab + P.off_factor;
            uint4 hn = *reinterpret_cast<const uint4*>(rec);
            for (uint32_t col = 0; col < n;) {
                const uint32_t hx = hn.x, C = hx & (kSkPairFlag - 1);
                SmAddr dp = f + hn.y;
                const double wk = ldp(w, hn.z);
                const uint32_t* body = rec + 4;
                rec = body + ((2 * C + C * (C + 1) / 2 + 3u) & ~3u);
                hn = *reinterpret_cast<const uint4*>(rec);
                const double d = lds(dp) + lam2;
                if (fstat == 0 && !(d > 0.0 && d < INFINITY)) fstat = d != d ? 2 : 1;
                const double inv = sk_rcp(d);
                if (dp_prev != kNone) sts(dp_prev, inv_prev);  // the helper read that pivot before the last barrier
                if (hx & kSkPairFlag) {
                    sk_column2_dispatch_half<0>(C, body, f, w, wk, inv, lam2, fstat, dp);  // stores 1 / d itself
                    dp_prev = kNone;
                    col += 2;
                } else {
                    sk_column_dispatch_half<0>(C, body, f, w, wk, inv);
                    dp_prev = dp;
                    inv_prev = inv;
                    __syncthreads();
                    col += 1;
                }
            }
            if (dp_prev != kNone) sts(dp_prev, inv_prev);
        }
        sk_back_solve(tab + P.off_back, n, f, w, xsp);
        __syncthreads();  // H and g are consumed: the helper clears them for the trial evaluation
        {
            dn = 0.0;
            uint32_t i = 0;
            for (; i + 4 <= n; i += 4) {
                double d[4], x0[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    d[u] = ldp(xsp, (i + u) << 8);
                    x0[u] = ldp(xp, (i + u) << 8);
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    dn = dn + d[u] * d[u];
                    stp(xsp, (i + u) << 8, x0[u] + d[u]);
                }
            }
            for (; i < n; i++) {
                const double d = ldp(xsp, i << 8);
                dn = dn + d * d;
                stp(xsp, i << 8, ldp(xp, i << 8) + d);
            }
        }
        mode = kTrial;
        xe = xsp;
    }
    if (!valid) return;
    double* out = free_out + (size_t)sketch * n;
    if (R.raw_vars == nullptr) {
        for (uint32_t i = 0; i < n; i++) out[i] = ldp(xp, i << 8);
    } else {  // system.variables[var] = system_scale * x[k] (assemble/mod.rs:161-166)
        for (uint32_t i = 0; i < n; i++) out[i] = scale * ldp(xp, i << 8);
        if (R.scales) R.scales[sketch] = scale;
    }
    fk_report rep;
    rep.exit_reason = exit_reason;
    rep.outer_iters = outer_iters;
    rep.factorizations = factorizations;
    rep.accepted = accepted;
    rep.ssr = ssr;
    rep.lambda = lambda;
    rep.trace_hash = trace;
    reports[sketch] = rep;
}

}  // namespace

// Warps per CTA (they share one copy of the tables) and CTAs per SM: the choice that puts the most warps on an SM; 238
// registers per thread allow 8.  228 KB of shared memory per SM, 1 KB of it reserved per resident CTA.
static void sk_shape(const SkProgram& prog, int* warps_per_cta, int* ctas_per_sm) {
    const size_t tab_bytes = (size_t)prog.tab_words * 4, state = (size_t)prog.entries * 256;
    int best_w = 1, best_warps = 0, best_ctas = 1;
    for (int wpc = 1; wpc <= kSkMaxWarps; wpc++) {
        const size_t per_cta = tab_bytes + wpc * state;
        if (per_cta > 227 * 1024) break;
        const int ctas = std::max(1, std::min((int)std::min<size_t>(32, (228 * 1024) / (per_cta + 1024)), 8 / wpc));
        const int warps = ctas * wpc;
        if (warps > best_warps || (warps == best_warps && wpc <= 2)) { best_warps = warps; best_w = wpc; best_ctas = ctas; }
    }
    static const int forced = [] {  // tuning knob
        const char* e = std::getenv("FK_SK_WARPS");
        return e ? std::atoi(e) : 0;
    }();
    if (forced >= 1 && forced <= kSkMaxWarps && tab_bytes + forced * state <= 227 * 1024) {
        best_w = forced;
        best_ctas = std::max(1, std::min((int)((228 * 1024) / (tab_bytes + forced * state + 1024)), 8 / forced));
    }
    *warps_per_cta = best_w;
    *ctas_per_sm = best_ctas;
}

// The warp-pair variant is used when the solo shape leaves schedulers idle (fewer than four warps per SM) and the
// pair shape keeps as many sketches in flight.  FK_SK_PAIR=0|1 forces the choice (A/B knob).
static bool sk_use_pair(const SkProgram& prog, uint32_t n_sketches, int* ctas_per_sm) {
    const size_t per_cta = (size_t)prog.tab_words * 4 + ((size_t)prog.entries + kPairExtra) * 256;
    if (per_cta > 227 * 1024) return false;
    const int pair_ctas = (int)std::min<size_t>(8, (228 * 1024) / (per_cta + 1024));
    *ctas_per_sm = pair_ctas;
    static const int env_forced = [] {
        const char* e = std::getenv("FK_SK_PAIR");
        return e ? std::atoi(e) : -1;
    }();
    const int choice = lm_kernel_choice().load(std::memory_order_relaxed);  // 2: solo, 3: pair (fk_set_lm_kernel)
    const int forced = choice == 2 ? 0 : (choice == 3 ? 1 : env_forced);
    if (forced == 0) return false;
    if (forced == 1) return true;
    // a batch that does not fill the device anyway: every group of 32 sketches gets its two warps for free, and the pair is
    // the faster shape per group (tools/lm_ab_small.py: 256-3,072 sketches, pair 5-15 % ahead of solo on every topology tried)
    if ((uint64_t)(n_sketches + 31) / 32 <= (uint64_t)pair_ctas * 148u) return true;
    int wpc, ctas;
    sk_shape(prog, &wpc, &ctas);
    const int solo_warps = wpc * ctas;
    // measured (tools/lm_ab.py, M sketches/s solo / pair): 20-point truss (2 solo warps, 2 pair CTAs) 54 / 72; 14-point truss
    // (3 solo warps, 2 pair CTAs) 128 / 117; 10-point truss (5, 3) 215 / 218: the pair pays when it keeps as many groups of 32
    // sketches in flight as the solo shape does warps
    return solo_warps < 4 && pair_ctas >= solo_warps;
}

int sketch_kernel_is_pair(const SkProgram& prog, uint32_t n_sketches) {
    int ctas = 0;
    return sk_use_pair(prog, n_sketches, &ctas) ? 1 : 0;
}

uint32_t sketch_kernel_wave(const SkProgram& prog, int sm_count) {
    int pair_ctas = 0;
    if (sk_use_pair(prog, 0xFFFFFFFFu, &pair_ctas)) return 32u * (uint32_t)pair_ctas * (uint32_t)sm_count;
    int wpc, ctas;
    sk_shape(prog, &wpc, &ctas);
    return 32u * (uint32_t)wpc * (uint32_t)ctas * (uint32_t)sm_count;
}

int launch_batch_lm_sketch(const SkProgram& prog, uint32_t n_sketches, const double* vars, const double* params, double* free_out,
                           fk_report* reports, void* stream, const SkRaw* raw_opt) {
    if (n_sketches == 0) return 0;
    if (!sk_fits(prog.entries, prog.tab_words)) return (int)cudaErrorInvalidConfiguration;
    SkRaw raw{};
    if (raw_opt) {
        if (!sk_raw_fits(prog, raw_opt->shared_param != 0)) return (int)cudaErrorInvalidConfiguration;
        raw = *raw_opt;
    }
    int pair_ctas = 0;
    if (sk_use_pair(prog, n_sketches, &pair_ctas)) {
        const size_t smem = (size_t)prog.tab_words * 4 + ((size_t)prog.entries + kPairExtra) * 256;
        cudaError_t e = cudaFuncSetAttribute(fk_batch_lm_sketch_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        e = cudaFuncSetAttribute(fk_batch_lm_sketch_pair_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return (int)e;
        fk_batch_lm_sketch_pair_kernel<<<(n_sketches + 31) / 32, 64, smem, (cudaStream_t)stream>>>(prog, raw, n_sketches, vars, params, free_out, reports);
        return (int)cudaGetLastError();
    }
    int best_w, ctas;
    sk_shape(prog, &best_w, &ctas);
    const size_t smem = (size_t)prog.tab_words * 4 + (size_t)best_w * prog.entries * 256;
    cudaError_t e = cudaFuncSetAttribute(fk_batch_lm_sketch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    e = cudaFuncSetAttribute(fk_batch_lm_sketch_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return (int)e;
    const uint32_t per_cta = 32u * (uint32_t)best_w;
    const uint32_t grid = (n_sketches + per_cta - 1) / per_cta;
    fk_batch_lm_sketch_kernel<<<grid, per_cta, smem, (cudaStream_t)stream>>>(prog, raw, n_sketches, vars, params, free_out, reports);
    return (int)cudaGetLastError();
}

}  // namespace fk
