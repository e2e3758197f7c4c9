#include "symbolic.hpp"

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <thread>

#include "colamd_order.hpp"

namespace fk {

int expand_slots(uint8_t kind, const uint32_t idx[4], uint32_t out[8]) {
    // Layout per kind: which stored index each slot comes from and whether it is the +1 (y) half.
    // 'p' = point (two slots), 'v' = single variable, 't' = pose (three slots).  expressions.rs:48-182; the pose rows
    // of ClusteredSystem (assemble/mod.rs:538-585): pose, updated coordinate, point before the step.
    static const char* shape[FK_NUM_KINDS] = {"vv", "pp", "ppp", "ppp", "ppp", "ppv", "pppp", "pppp", "pppp", "pppp", "pppv", "tvp", "tvp"};
    if (kind >= FK_NUM_KINDS) return -1;
    int n = 0;
    for (int k = 0; shape[kind][k]; k++) {
        out[n++] = idx[k];
        if (shape[kind][k] != 'v') out[n++] = idx[k] + 1;
        if (shape[kind][k] == 't') out[n++] = idx[k] + 2;
    }
    return n;
}

// Host threads for the phases of the symbolic pipeline that are independent per column / per row
// (large systems only; the reference is single-threaded and repeats this work on every LM call).
static unsigned symbolic_threads(uint64_t work) {
    if (work < (1u << 18)) return 1;
    unsigned t = std::thread::hardware_concurrency();
    if (const char* e = std::getenv("FK_SYM_THREADS")) t = (unsigned)std::max(1, std::atoi(e));
    return std::min(std::max(t, 1u), 32u);
}

// f(thread, begin, end) over [0, n) in chunks handed out dynamically (balanced for uneven work per index).
template <class F>
static void parallel_chunks(uint32_t n, uint32_t chunk, unsigned threads, F&& f) {
    if (threads <= 1 || n <= chunk) {
        f(0u, 0u, n);
        return;
    }
    std::atomic<uint32_t> next{0};
    std::vector<std::thread> pool;
    for (unsigned t = 0; t < threads; t++)
        pool.emplace_back([&, t] {
            for (;;) {
                const uint32_t b = next.fetch_add(chunk);
                if (b >= n) break;
                f(t, b, std::min(n, b + chunk));
            }
        });
    for (auto& th : pool) th.join();
}

static uint64_t mix(uint64_t h, uint64_t v) {
    h ^= v + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2);
    h *= 0xFF51AFD7ED558CCDull;
    return h ^ (h >> 33);
}

int Topology::build(const fk_problem& p, uint32_t lanes) {
    // FK_SYM_TIMING=1: wall time of every phase of the host symbolic pipeline to stderr
    static const bool sym_timing = std::getenv("FK_SYM_TIMING") != nullptr;
    auto sym_t0 = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (!sym_timing) return;
        const auto now = std::chrono::steady_clock::now();
        std::fprintf(stderr, "[symbolic] %-28s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(now - sym_t0).count());
        sym_t0 = now;
    };
    if ((p.n_expr && (!p.kind || !p.idx)) || (p.n_free && !p.free_vars) || (p.n_rows && !p.rows)) {
        error = "null array in fk_problem";
        return FK_ERR_INVALID;
    }
    n_vars = p.n_vars; n_expr = p.n_expr; n_free = p.n_free; n_rows = p.n_rows;
    kind.assign(p.kind, p.kind + n_expr);
    idx.assign(p.idx, p.idx + 4 * (size_t)n_expr);
    free_vars.assign(p.free_vars, p.free_vars + n_free);
    rows.assign(p.rows, p.rows + n_rows);

    signature = mix(mix(mix(0x1234, n_vars), n_free), n_rows);
    for (uint32_t r : rows) {
        if (r >= n_expr) { error = "row references an expression out of range"; return FK_ERR_INVALID; }
        signature = mix(signature, kind[r]);
        for (int q = 0; q < 4; q++) signature = mix(signature, idx[4 * (size_t)r + q]);
    }
    for (uint32_t v : free_vars) signature = mix(signature, v);

    // free-column lookup: rank in free_vars == IndexSet index (subsystem.rs:35,66-68)
    std::vector<int32_t> var_to_free(n_vars, -1);
    for (uint32_t k = 0; k < n_free; k++) {
        uint32_t v = free_vars[k];
        if (v >= n_vars) { error = "free variable out of range"; return FK_ERR_INVALID; }
        if (var_to_free[v] >= 0) { error = "duplicate free variable"; return FK_ERR_INVALID; }
        var_to_free[v] = (int32_t)k;
    }

    // ---- slot tables ------------------------------------------------------------------------
    const uint32_t m = n_rows, n = n_free;
    row_kind.resize(m); row_expr.resize(m);
    slot_var.assign((size_t)m * 8, 0); slot_col.assign((size_t)m * 8, -2);
    slot_pos.assign((size_t)m * 8, -1); slot_dup.assign((size_t)m * 8, 0);
    std::vector<uint32_t> col_count(n + 1, 0);
    eval_bytes = 0;
    static const int stored_idx[FK_NUM_KINDS] = {2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 4, 3, 3};
    for (uint32_t r = 0; r < m; r++) {
        uint32_t e = rows[r];
        uint8_t kd = kind[e];
        uint32_t sv[8];
        int a = expand_slots(kd, &idx[4 * (size_t)e], sv);
        if (a < 0) { error = "unknown expression kind"; return FK_ERR_INVALID; }
        row_kind[r] = kd; row_expr[r] = e;
        int f = 0;
        for (int s = 0; s < a; s++) {
            if (sv[s] >= n_vars) { error = "expression references a variable out of range"; return FK_ERR_INVALID; }
            slot_var[(size_t)r * 8 + s] = sv[s];
            int32_t c = var_to_free[sv[s]];
            slot_col[(size_t)r * 8 + s] = c;
            if (c < 0) continue;
            f++;
            bool dup = false;
            for (int t = 0; t < s; t++) dup |= slot_col[(size_t)r * 8 + t] == c;
            slot_dup[(size_t)r * 8 + s] = dup;
            if (!dup) col_count[c]++;
        }
        // SURVEY §8(d): kind + stored indices + param + gathered vars + scatter slots + r + J
        eval_bytes += 1 + 4 * stored_idx[kd] + 8 + 8 * a + 4 * f + 8 + 8 * f;
    }

    lap("slot tables");
    // ---- augmented CSC pattern ----------------------------------------------------------------
    aug_colptr.assign(n + 1, 0);
    for (uint32_t c = 0; c < n; c++) aug_colptr[c + 1] = aug_colptr[c] + col_count[c] + 1;
    aug_rowidx.assign(aug_colptr[n], 0);
    jac_nnz = aug_colptr[n] - n;
    {
        std::vector<uint32_t> fill(aug_colptr.begin(), aug_colptr.begin() + n);
        for (uint32_t r = 0; r < m; r++)        // rows ascending -> every column list ends up sorted
            for (int s = 0; s < 8; s++) {
                int32_t c = slot_col[(size_t)r * 8 + s];
                if (c < 0 || slot_dup[(size_t)r * 8 + s]) continue;
                aug_rowidx[fill[c]++] = r;
            }
        for (uint32_t c = 0; c < n; c++) aug_rowidx[fill[c]] = m + c;  // damping row last
        // Jacobian value position of a slot = CSC position with the damping entries squeezed out
        std::vector<uint32_t> cursor(n);
        for (uint32_t c = 0; c < n; c++) cursor[c] = aug_colptr[c] - c;
        for (uint32_t r = 0; r < m; r++) {
            for (int s = 0; s < 8; s++) {
                int32_t c = slot_col[(size_t)r * 8 + s];
                if (c < 0) continue;
                if (!slot_dup[(size_t)r * 8 + s]) {
                    slot_pos[(size_t)r * 8 + s] = (int32_t)cursor[c]++;
                } else {
                    for (int t = 0; t < s; t++)
                        if (slot_col[(size_t)r * 8 + t] == c) { slot_pos[(size_t)r * 8 + s] = slot_pos[(size_t)r * 8 + t]; break; }
                }
            }
        }
    }

    lap("augmented pattern");
    // ---- fill-reducing ordering -----------------------------------------------------------------
    perm = ColamdOrder::order((int)(m + n), (int)n, aug_colptr.data(), aug_rowidx.data());
    iperm.assign(n, 0);
    for (uint32_t k = 0; k < n; k++) iperm[perm[k]] = (int32_t)k;

    lap("colamd");
    // ---- column elimination tree of A*P (tree of (AP)ᵀ(AP), never formed) -------------------------
    // Liu's algorithm with path compression; `last_col[i]` links row i to the previous column that
    // held it, which is all of the product's structure that matters.
    parent.assign(n, -1);
    std::vector<int32_t> first_col(m + n, -1);
    {
        std::vector<int32_t> anc(n, -1), last_col(m + n, -1);
        for (uint32_t j = 0; j < n; j++) {
            uint32_t src = (uint32_t)perm[j];
            for (uint32_t q = aug_colptr[src]; q < aug_colptr[src + 1]; q++) {
                uint32_t i = aug_rowidx[q];
                if (first_col[i] < 0) first_col[i] = (int32_t)j;
                for (int32_t k = last_col[i]; k != -1 && k < (int32_t)j;) {
                    int32_t up = anc[k];
                    anc[k] = (int32_t)j;
                    if (up == -1) parent[k] = (int32_t)j;
                    k = up;
                }
                last_col[i] = (int32_t)j;
            }
        }
    }
    {
        std::vector<uint32_t> depth(n, 0);
        etree_height = n ? 1 : 0;
        for (uint32_t jj = n; jj-- > 0;) {  // parents have larger indices
            if (parent[jj] >= 0) depth[jj] = depth[parent[jj]] + 1;
            etree_height = std::max(etree_height, depth[jj] + 1);
        }
    }

    lap("elimination tree");
    // ---- pattern of R = Lᵀ: union of row subtrees (columns of A*P walked up the tree) ------------
    // Columns are independent given the tree: pass 1 counts, pass 2 writes each sorted list in place
    // (threads own private mark arrays; chunks are handed out dynamically).
    r_colptr.assign(n + 1, 0);
    r_rowidx.clear();
    {
        const unsigned T = symbolic_threads((uint64_t)aug_colptr[n] * 8);
        std::vector<std::vector<int32_t>> marks(T);
        std::vector<std::vector<uint32_t>> cols(T);
        auto walk = [&](unsigned t, uint32_t j, std::vector<uint32_t>& col) {
            std::vector<int32_t>& mark = marks[t];
            col.clear();
            mark[j] = (int32_t)j;
            const uint32_t src = (uint32_t)perm[j];
            for (uint32_t q = aug_colptr[src]; q < aug_colptr[src + 1]; q++)
                for (int32_t k = first_col[aug_rowidx[q]]; k != -1 && k < (int32_t)j && mark[k] != (int32_t)j; k = parent[k]) {
                    mark[k] = (int32_t)j;
                    col.push_back((uint32_t)k);
                }
        };
        auto reset = [&](unsigned t) {
            if (marks[t].size() != n) marks[t].assign(n, -1);
            else std::fill(marks[t].begin(), marks[t].end(), -1);
        };
        std::vector<std::atomic<bool>> started(T);
        for (auto& b : started) b = false;
        parallel_chunks(n, 512, T, [&](unsigned t, uint32_t b, uint32_t e) {
            if (!started[t].exchange(true)) reset(t);
            for (uint32_t j = b; j < e; j++) {
                walk(t, j, cols[t]);
                r_colptr[j + 1] = (uint32_t)cols[t].size() + 1;
            }
        });
        for (uint32_t j = 0; j < n; j++) r_colptr[j + 1] += r_colptr[j];
        r_rowidx.resize(r_colptr[n]);
        for (auto& b : started) b = false;
        parallel_chunks(n, 512, T, [&](unsigned t, uint32_t b, uint32_t e) {
            if (!started[t].exchange(true)) reset(t);
            for (uint32_t j = b; j < e; j++) {
                std::vector<uint32_t>& col = cols[t];
                walk(t, j, col);
                std::sort(col.begin(), col.end());
                uint32_t* dst = r_rowidx.data() + r_colptr[j];
                std::copy(col.begin(), col.end(), dst);
                dst[col.size()] = j;
            }
        });
    }
    const uint32_t lnnz = (uint32_t)r_rowidx.size();

    lap("R pattern");
    // ---- L in CSC (transpose of R): diagonal first, then ascending rows ---------------------------
    l_colptr.assign(n + 1, 0);
    for (uint32_t q = 0; q < lnnz; q++) l_colptr[r_rowidx[q] + 1]++;
    for (uint32_t k = 0; k < n; k++) l_colptr[k + 1] += l_colptr[k];
    l_rowidx.assign(lnnz, 0);
    r_lpos.assign(lnnz, 0);
    {
        // transpose by ranges of target columns: a thread owns the L columns [k0, k1) and finds its part of
        // every (sorted) R column by binary search, so no two threads write the same list
        const unsigned T = symbolic_threads(lnnz);
        std::vector<uint32_t> bound(T + 1, n);
        bound[0] = 0;
        for (unsigned t = 1; t < T; t++) {
            const uint32_t want = (uint32_t)((uint64_t)lnnz * t / T);
            bound[t] = (uint32_t)(std::upper_bound(l_colptr.begin(), l_colptr.end(), want) - l_colptr.begin() - 1);
            bound[t] = std::max(bound[t], bound[t - 1]);
        }
        auto part = [&](unsigned t) {
            const uint32_t k0 = bound[t], k1 = bound[t + 1];
            if (k0 >= k1) return;
            std::vector<uint32_t> fill(l_colptr.begin() + k0, l_colptr.begin() + k1);
            for (uint32_t k = k0; k < k1; k++) l_rowidx[fill[k - k0]++] = k;  // diagonal
            for (uint32_t j = k0; j < n; j++) {  // R(i, j) has i <= j: columns before k0 hold nothing of this range
                const uint32_t* b = r_rowidx.data() + r_colptr[j];
                const uint32_t* e = r_rowidx.data() + r_colptr[j + 1];
                const uint32_t* lo = T > 1 ? std::lower_bound(b, e, k0) : b;
                for (const uint32_t* it = lo; it != e && *it < k1; ++it) {
                    const uint32_t i = *it, q = (uint32_t)(it - r_rowidx.data());  // R(i, j) == L(j, i)
                    if (i == j) { r_lpos[q] = l_colptr[j]; continue; }
                    r_lpos[q] = fill[i - k0];
                    l_rowidx[fill[i - k0]++] = j;
                }
            }
        };
        if (T <= 1) part(0);
        else {
            std::vector<std::thread> pool;
            for (unsigned t = 0; t < T; t++) pool.emplace_back(part, t);
            for (auto& th : pool) th.join();
        }
    }
    chol_flops = 0;
    uint64_t n_updates = 0;
    max_col_updates = 0;
    for (uint32_t k = 0; k < n; k++) {
        uint64_t c = l_colptr[k + 1] - l_colptr[k];
        chol_flops += c * c;
        uint64_t u = (c - 1) * c / 2;
        n_updates += u;
        max_col_updates = std::max<uint32_t>(max_col_updates, (uint32_t)std::min<uint64_t>(u, 0xFFFFFFFFu));
    }

    lap("L transpose");
    // ---- path selection -----------------------------------------------------------------------------
    {
        uint64_t work = std::max<uint64_t>(jac_nnz, lnnz);
        uint64_t dbl = 3ull * n + std::max(n, m) + jac_nnz + work;  // == lm_smem_doubles()
        uint64_t bytes = dbl * 8;
        smem_bytes = (uint32_t)std::min<uint64_t>(bytes, 0xFFFFFFFFu);
        uint32_t w = std::max(m, n);
        if (bytes <= 24 * 1024 && n_updates < (1u << 22)) {
            path = 0;
            // Lanes per sketch, measured on B200 (tools/tile_probe.py; M sketches/s at 4 / 8 / 16 lanes): config-4
            // topology (1.1 KB of shared state) 140 / 117 / 74; 10-point truss (2.0 KB) 93 / 121 / 83; 14-point truss
            // (2.8 KB) - / 61.5 / 62.1; 20-point truss (4.1 KB) 20 / 30 / 37.6.  Fewer lanes mean more sketches per
            // instruction (less table walking and fewer shared-memory wavefronts per sketch) but more shared memory per
            // warp, i.e. fewer resident warps; the crossover follows the per-sketch footprint.
            (void)w;
            tile = bytes <= 1300 ? 4 : (bytes <= 2600 ? 8 : (std::max(m, n) <= 96 ? 16 : 32));
        } else if (bytes <= 200 * 1024 && n_updates < (1u << 25)) {
            path = 1;
            tile = 256;
        } else {
            path = 2;
            tile = 0;
        }
        if (const char* f = std::getenv("FK_FORCE_PATH")) {
            if (std::atoi(f) == 2) { path = 2; tile = 0; }
        }
        if (const char* t = std::getenv("FK_TILE")) {
            int v = std::atoi(t);
            if (path == 0 && (v == 1 || v == 2 || v == 4 || v == 8 || v == 16 || v == 32)) tile = (uint32_t)v;
        }
        if (lanes && path == 0) tile = lanes;
    }

    lap("path selection");
    // ---- contribution lists of H = JᵀJ in L storage, and of g = Jᵀ(-r) ----------------------------------
    auto l_find = [&](uint32_t row, uint32_t col) -> int64_t {  // position of L(row, col), row >= col
        const uint32_t* b = l_rowidx.data() + l_colptr[col] + 1;
        const uint32_t* e = l_rowidx.data() + l_colptr[col + 1];
        if (row == col) return l_colptr[col];
        const uint32_t* it = std::lower_bound(b, e, row);
        return (it != e && *it == row) ? (int64_t)(it - l_rowidx.data()) : -1;
    };
    h_ptr.assign((size_t)lnnz + 1, 0);
    {
        // the L position of every (row, a, b) product, looked up once (in parallel over the rows), then
        // counted and filled in row order so that every list keeps the reference's summation order
        std::vector<uint32_t> pair_ptr((size_t)m + 1, 0);
        for (uint32_t r = 0; r < m; r++) {
            uint32_t cnt = 0;
            for (int s = 0; s < 8; s++) cnt += (slot_col[(size_t)r * 8 + s] >= 0 && !slot_dup[(size_t)r * 8 + s]) ? 1u : 0u;
            pair_ptr[r + 1] = pair_ptr[r] + cnt * (cnt + 1) / 2;
        }
        std::vector<int64_t> pair_pos(pair_ptr[m]);
        std::vector<uint32_t> pair_ab(2 * (size_t)pair_ptr[m]);
        std::atomic<bool> bad{false};
        parallel_chunks(m, 2048, symbolic_threads((uint64_t)pair_ptr[m] * 8), [&](unsigned, uint32_t rb, uint32_t re) {
            for (uint32_t r = rb; r < re; r++) {
                int32_t cs[8], ps[8];
                int cnt = 0;
                for (int s = 0; s < 8; s++) {
                    int32_t c = slot_col[(size_t)r * 8 + s];
                    if (c < 0 || slot_dup[(size_t)r * 8 + s]) continue;
                    cs[cnt] = iperm[c];
                    ps[cnt++] = slot_pos[(size_t)r * 8 + s];
                }
                size_t at = pair_ptr[r];
                for (int a = 0; a < cnt; a++)
                    for (int b = 0; b <= a; b++, at++) {
                        uint32_t hi = (uint32_t)std::max(cs[a], cs[b]), lo = (uint32_t)std::min(cs[a], cs[b]);
                        pair_pos[at] = l_find(hi, lo);
                        if (pair_pos[at] < 0) bad = true;
                        pair_ab[2 * at] = (uint32_t)ps[a];
                        pair_ab[2 * at + 1] = (uint32_t)ps[b];
                    }
            }
        });
        lap("H lookups");
        if (bad) { error = "internal: JtJ entry outside the L pattern"; return FK_ERR_INTERNAL; }
        for (size_t at = 0; at < pair_pos.size(); at++) h_ptr[pair_pos[at] + 1]++;
        for (uint32_t q = 0; q < lnnz; q++) h_ptr[q + 1] += h_ptr[q];
        h_pairs.assign(2 * (size_t)h_ptr[lnnz], 0);
        std::vector<uint32_t> fill(h_ptr.begin(), h_ptr.begin() + lnnz);
        for (size_t at = 0; at < pair_pos.size(); at++) {
            const uint32_t w = fill[pair_pos[at]]++;
            h_pairs[2 * (size_t)w] = pair_ab[2 * at];
            h_pairs[2 * (size_t)w + 1] = pair_ab[2 * at + 1];
        }
    }
    lap("H lists");
    g_ptr.assign(n + 1, 0);
    g_pairs.clear();
    for (uint32_t k = 0; k < n; k++) {
        uint32_t c = (uint32_t)perm[k];
        uint32_t jp = aug_colptr[c] - c;
        for (uint32_t q = aug_colptr[c]; q + 1 < aug_colptr[c + 1]; q++, jp++) {
            g_pairs.push_back(jp);
            g_pairs.push_back(aug_rowidx[q]);
        }
        g_ptr[k + 1] = (uint32_t)(g_pairs.size() / 2);
    }

    lap("H and g lists");
    // ---- LDLᵀ update schedule (shared-memory paths only) ------------------------------------------
    u_ptr.assign(n + 1, 0);
    u_trip.clear();
    if (path != 2) {
        u_trip.reserve(3 * (size_t)n_updates);
        for (uint32_t k = 0; k < n; k++) {
            uint32_t b0 = l_colptr[k] + 1, e0 = l_colptr[k + 1];
            for (uint32_t qb = b0; qb < e0; qb++) {       // column j = row of entry qb
                uint32_t j = l_rowidx[qb];
                for (uint32_t qa = qb; qa < e0; qa++) {   // rows i >= j
                    int64_t dst = l_find(l_rowidx[qa], j);
                    if (dst < 0) { error = "internal: fill outside the L pattern"; return FK_ERR_INTERNAL; }
                    u_trip.push_back((uint32_t)dst);
                    u_trip.push_back(qa);
                    u_trip.push_back(qb);
                }
            }
            u_ptr[k + 1] = (uint32_t)(u_trip.size() / 3);
        }
    }
    lap("update schedule");
    const int rc_tables = build_tables();
    lap("kernel tables");
    return rc_tables;
}

// Lane-padded op tables for the shared-memory kernel (see Topology::Tables).
int Topology::build_tables() {
    const uint32_t n = n_free, m = n_rows, T = path == 2 ? 1 : tile;
    const uint32_t NOP = 0xFFFFFFFFu;
    const uint32_t lnnz = (uint32_t)l_rowidx.size();
    if (path != 2 && (lnnz >= 0xFFFF || jac_nnz >= 0xFFFF || n >= 0xFFFF || m >= 0xFFFF || n_expr >= (1u << 24))) {
        error = "problem too large for the 16-bit shared-memory tables";
        return FK_ERR_TOO_LARGE;
    }
    Tables& t = tab;
    // ---- evaluation rows -------------------------------------------------------------------------
    t.eval_rounds = (m + T - 1) / T;
    t.row_hdr.assign((size_t)t.eval_rounds * T, NOP);
    t.row_slots.assign((size_t)t.eval_rounds * T * 16, NOP);
    t.uniform_kind = m ? row_kind[0] : -1;
    for (uint32_t r = 0; r < m; r++) {
        if (row_kind[r] != t.uniform_kind) t.uniform_kind = -1;
        t.row_hdr[r] = row_kind[r] | (row_expr[r] << 8);
        for (int s = 0; s < 8; s++) {
            int32_t c = slot_col[(size_t)r * 8 + s];
            if (c == -2) continue;  // unused slot
            uint32_t src = c >= 0 ? (uint32_t)c : (0x80000000u | slot_var[(size_t)r * 8 + s]);
            int32_t jp = slot_pos[(size_t)r * 8 + s];
            uint32_t pos = jp < 0 ? NOP : ((uint32_t)jp | (slot_dup[(size_t)r * 8 + s] ? 0x40000000u : 0u));
            t.row_slots[((size_t)r * 8 + s) * 2] = src;
            t.row_slots[((size_t)r * 8 + s) * 2 + 1] = pos;
        }
    }
    if (path == 2) return FK_OK;  // the global sparse path builds its own schedules (sparse_path.cu)
    const uint32_t FIRST = 1u << 16, LAST = 1u << 17;
    // ---- contribution lists, longest first, so that the lanes of a step group finish together -----
    auto pack_lists = [&](const std::vector<uint32_t>& ptr, const std::vector<uint32_t>& pairs, uint32_t count,
                          uint32_t& nsteps, std::vector<uint32_t>& flags, std::vector<uint32_t>& ops,
                          std::vector<uint32_t>& dst) {
        std::vector<uint32_t> order(count);
        for (uint32_t i = 0; i < count; i++) order[i] = i;
        std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) {
            return ptr[a + 1] - ptr[a] > ptr[b + 1] - ptr[b];
        });
        flags.clear(); ops.clear(); dst.clear();
        for (uint32_t at = 0; at < count; at += T) {
            uint32_t lanes = std::min(T, count - at), len = 1;
            for (uint32_t l = 0; l < lanes; l++) len = std::max(len, ptr[order[at + l] + 1] - ptr[order[at + l]]);
            size_t base = flags.size();
            for (uint32_t k = 0; k < len; k++) flags.push_back((k == 0 ? FIRST : 0) | (k + 1 == len ? LAST : 0));
            ops.resize((base + len) * T, NOP);
            dst.resize((base + len) * T, NOP);
            for (uint32_t l = 0; l < lanes; l++) {
                uint32_t e = order[at + l];
                for (uint32_t q = ptr[e], k = 0; q < ptr[e + 1]; q++, k++)
                    ops[(base + k) * T + l] = pairs[2 * (size_t)q] | (pairs[2 * (size_t)q + 1] << 16);
                dst[(base + len - 1) * T + l] = e;
            }
        }
        nsteps = (uint32_t)flags.size();
        flags.push_back(0);  // prefetch padding
        ops.resize(ops.size() + T, NOP);
        dst.resize(dst.size() + T, NOP);
    };
    pack_lists(h_ptr, h_pairs, lnnz, t.a_nsteps, t.a_flags, t.a_ops, t.a_dst);
    pack_lists(g_ptr, g_pairs, n, t.g_nsteps, t.g_flags, t.g_ops, t.g_dst);
    // ---- LDLt: one or more steps per column.  The forward substitution rides along: the right-hand
    // side w lives right behind L in shared memory (position wbase + i), and "w[i] -= (L D)(i,k) / d_k *
    // w[k]" has exactly the shape of a factor update with dst = w[i], a = (i,k), b = w[k]. ------------------
    const uint32_t wbase = std::max(lnnz, jac_nnz);
    if (wbase + n >= 0xFFFF) { error = "problem too large for the 16-bit shared-memory tables"; return FK_ERR_TOO_LARGE; }
    t.f_steps.clear(); t.f_ops.clear();
    for (uint32_t k = 0; k < n; k++) {
        std::vector<uint32_t> ops3;
        for (uint32_t q = u_ptr[k]; q < u_ptr[k + 1]; q++) {
            ops3.push_back(u_trip[3 * (size_t)q]); ops3.push_back(u_trip[3 * (size_t)q + 1]); ops3.push_back(u_trip[3 * (size_t)q + 2]);
        }
        for (uint32_t q = l_colptr[k] + 1; q < l_colptr[k + 1]; q++) {
            ops3.push_back(wbase + l_rowidx[q]); ops3.push_back(q); ops3.push_back(wbase + k);
        }
        uint32_t cnt = (uint32_t)(ops3.size() / 3);
        uint32_t rounds = std::max(1u, (cnt + T - 1) / T);
        size_t base = t.f_steps.size();
        for (uint32_t r = 0; r < rounds; r++)
            t.f_steps.push_back(l_colptr[k] | (r == 0 ? FIRST : 0) | (r + 1 == rounds ? LAST : 0));
        t.f_ops.resize((base + rounds) * T * 2, NOP);
        for (uint32_t q = 0; q < cnt; q++) {
            t.f_ops[(base * T + q) * 2] = ops3[3 * q] | (ops3[3 * q + 1] << 16);
            t.f_ops[(base * T + q) * 2 + 1] = ops3[3 * q + 2];
        }
    }
    t.f_nsteps = (uint32_t)t.f_steps.size();
    t.f_steps.push_back(0);
    t.f_ops.resize(t.f_ops.size() + (size_t)T * 2, NOP);
    // ---- triangular solves ---------------------------------------------------------------------------
    auto pack_cols = [&](bool backward, uint32_t& nsteps, std::vector<uint32_t>& steps, std::vector<uint32_t>& ops) {
        steps.clear(); ops.clear();
        for (uint32_t kk = 0; kk < n; kk++) {
            uint32_t k = backward ? n - 1 - kk : kk;
            std::vector<uint32_t> list;
            if (!backward) {
                for (uint32_t q = l_colptr[k] + 1; q < l_colptr[k + 1]; q++) list.push_back(l_rowidx[q] | (q << 16));
                if (list.empty()) continue;  // nothing below the diagonal: w[k] is already final
            } else {
                for (uint32_t q = r_colptr[k]; q + 1 < r_colptr[k + 1]; q++) list.push_back(r_rowidx[q] | (r_lpos[q] << 16));
            }
            uint32_t rounds = std::max<uint32_t>(1, ((uint32_t)list.size() + T - 1) / T);
            size_t base = steps.size() / 2;
            for (uint32_t r = 0; r < rounds; r++) {
                steps.push_back(l_colptr[k] | (r == 0 ? FIRST : 0) | (r + 1 == rounds ? LAST : 0));
                steps.push_back(backward ? (k | ((uint32_t)perm[k] << 16)) : k);
            }
            ops.resize((base + rounds) * T, NOP);
            for (size_t q = 0; q < list.size(); q++) ops[base * T + q] = list[q];
        }
        nsteps = (uint32_t)(steps.size() / 2);
        steps.push_back(0); steps.push_back(0);
        ops.resize(ops.size() + T, NOP);
    };
    pack_cols(false, t.s_nsteps, t.s_steps, t.s_ops);
    pack_cols(true, t.b_nsteps, t.b_steps, t.b_ops);
    build_sketch_tables();
    return FK_OK;
}

// Tables of the sketch-per-thread kernel (see Topology::SketchTables).  Summation orders are those of the tile
// kernel's lists (H and g: rows ascending from zero; LDLt: columns ascending, each target once per column;
// back substitution: rows descending), so the two kernels produce the same numbers bit for bit.
void Topology::build_sketch_tables() {
    SketchTables& k = sk;
    k = SketchTables();
    const uint32_t n = n_free, m = n_rows, lnnz = (uint32_t)l_rowidx.size();
    auto refuse = [&](const char* why) { k.ok = false; k.why = why; k.tab.clear(); };
    if (path == 2 || n == 0 || m == 0) return refuse("not a shared-memory topology");
    if (lnnz >= (1u << 22) || n >= (1u << 22) || n_vars >= (1u << 22)) return refuse("exceeds the table words");
    for (size_t q = 0; q < slot_dup.size(); q++)
        if (slot_dup[q] && slot_col[q] >= 0) return refuse("a row names a free variable twice");
    auto l_find = [&](uint32_t row, uint32_t col) -> int64_t {
        if (row == col) return l_colptr[col];
        const uint32_t* b = l_rowidx.data() + l_colptr[col] + 1;
        const uint32_t* e = l_rowidx.data() + l_colptr[col + 1];
        const uint32_t* it = std::lower_bound(b, e, row);
        return (it != e && *it == row) ? (int64_t)(it - l_rowidx.data()) : -1;
    };
    const uint32_t NONE = 0xFFFFFFFFu;
    auto pos = [](uint32_t entry) { return entry << 8; };  // byte offset of an entry inside its region
    // fixed variables and parameters some row reads
    std::vector<int32_t> fix_slot(n_vars, -1), par_slot(n_expr, -1);
    std::vector<uint32_t> fix_list, par_list;
    static const bool has_param[FK_NUM_KINDS] = {false, true, true, false, true, false, false, true, false, false, false, false, false};
    for (uint32_t r = 0; r < m; r++) {
        const int a = kind_arity(row_kind[r]);
        for (int s = 0; s < a; s++)
            if (slot_col[(size_t)r * 8 + s] < 0) {
                const uint32_t v = slot_var[(size_t)r * 8 + s];
                if (fix_slot[v] < 0) { fix_slot[v] = (int32_t)fix_list.size(); fix_list.push_back(v); }
            }
        if (has_param[row_kind[r]] && par_slot[row_expr[r]] < 0) {
            par_slot[row_expr[r]] = (int32_t)par_list.size();
            par_list.push_back(row_expr[r]);
        }
    }
    k.nfix = (uint32_t)fix_list.size(); k.npar = (uint32_t)par_list.size();
    k.xa = 0; k.xb = n; k.w = 2 * n; k.f = 3 * n; k.fx = 3 * n + lnnz; k.pr = k.fx + k.nfix; k.entries = k.pr + k.npar;
    std::vector<uint32_t>& T = k.tab;
    k.off_free = (uint32_t)T.size();
    for (uint32_t c = 0; c < n; c++) T.push_back(free_vars[c]);
    k.off_fix = (uint32_t)T.size();
    T.insert(T.end(), fix_list.begin(), fix_list.end());
    k.off_par = (uint32_t)T.size();
    T.insert(T.end(), par_list.begin(), par_list.end());
    // every record below starts on a 16-byte boundary and is padded to one (the kernel reads 4 words per load)
    auto pad4 = [&] { while (T.size() & 3u) T.push_back(0); };
    pad4();
    k.off_eval = (uint32_t)T.size();
    for (uint32_t r = 0; r < m; r++) {
        const int a = kind_arity(row_kind[r]);
        const uint32_t words = (2 + 2 * (uint32_t)a + (uint32_t)(a * (a + 1) / 2) + 3u) & ~3u;
        bool special = false;
        int32_t pc[8];
        for (int s = 0; s < a; s++) {
            const int32_t c = slot_col[(size_t)r * 8 + s];
            pc[s] = c >= 0 ? iperm[c] : -1;
            special = special || c < 0;
        }
        T.push_back(row_kind[r] | (special ? 0x100u : 0u) | (words << 16));
        T.push_back(has_param[row_kind[r]] ? pos((uint32_t)par_slot[row_expr[r]]) : 0u);
        for (int s = 0; s < a; s++) {
            const int32_t c = slot_col[(size_t)r * 8 + s];
            T.push_back(c >= 0 ? pos((uint32_t)c) : (0x80000000u | pos((uint32_t)fix_slot[slot_var[(size_t)r * 8 + s]])));
        }
        for (int s = 0; s < a; s++) T.push_back(pc[s] >= 0 ? pos((uint32_t)pc[s]) : NONE);
        for (int s = 0; s < a; s++)
            for (int b = 0; b <= s; b++) {
                if (pc[s] < 0 || pc[b] < 0) { T.push_back(NONE); continue; }
                const int64_t p = l_find((uint32_t)std::max(pc[s], pc[b]), (uint32_t)std::min(pc[s], pc[b]));
                if (p < 0) return refuse("internal: JtJ entry outside the L pattern");
                T.push_back(pos((uint32_t)p));
            }
        pad4();
    }
    T.insert(T.end(), 4, 0u);  // the kernel prefetches the header of the record after the last one
    // Column pairs: column c pairs with c + 1 when L(:,c) = {c+1} u L(:,c+1) and C(c) <= kSkPairMaxC, taken greedily in
    // column order (a wider supernode splits into consecutive pairs).  Then every target of column c+1 is a target of
    // column c, and c+1's diagonal, entries and right-hand side entry are column c's targets (0, 0), (a >= 1, 0) and its
    // first w row, so one kernel step eliminates both columns with one load and one store per target.
    // FK_SK_COLPAIR=0 emits single-column records only (A/B knob; read here, when a topology's tables are built).
    const char* env_pairs = std::getenv("FK_SK_COLPAIR");
    const bool use_pairs = !(env_pairs && std::atoi(env_pairs) == 0);
    std::vector<uint8_t> pair_first(n, 0);  // 1: column c is the first of a pair
    for (uint32_t c = 0; use_pairs && c + 1 < n; c++) {
        const uint32_t b0 = l_colptr[c] + 1, e0 = l_colptr[c + 1], C = e0 - b0;
        const uint32_t b1 = l_colptr[c + 1] + 1, e1 = l_colptr[c + 2];
        if (C < 1 || C > kSkPairMaxC || l_rowidx[b0] != c + 1 || e1 - b1 != C - 1) continue;
        if (!std::equal(l_rowidx.begin() + b0 + 1, l_rowidx.begin() + e0, l_rowidx.begin() + b1)) continue;
        pair_first[c] = 1;
        c++;
    }
    k.off_factor = (uint32_t)T.size();
    for (uint32_t c = 0; c < n; c += pair_first[c] ? 2 : 1) {
        const uint32_t b0 = l_colptr[c] + 1, e0 = l_colptr[c + 1], C = e0 - b0;
        if (C >= kSkPairFlag) return refuse("a column's count collides with the pair flag");  // (the kernel reads C as the bits below it)
        T.push_back(C | (pair_first[c] ? kSkPairFlag : 0u)); T.push_back(pos(l_colptr[c])); T.push_back(pos(c)); T.push_back(0);
        for (uint32_t q = b0; q < e0; q++) T.push_back(pos(q));
        for (uint32_t q = b0; q < e0; q++) T.push_back(pos(l_rowidx[q]));
        for (uint32_t qa = b0; qa < e0; qa++)
            for (uint32_t qb = b0; qb <= qa; qb++) {
                const int64_t dst = l_find(l_rowidx[qa], l_rowidx[qb]);
                if (dst < 0) return refuse("internal: fill outside the L pattern");
                T.push_back(pos((uint32_t)dst));
            }
        pad4();
    }
    T.insert(T.end(), 4, 0u);
    k.off_back = (uint32_t)T.size();
    for (uint32_t cc = n; cc-- > 0;) {
        const bool pair = cc > 0 && pair_first[cc - 1];
        const uint32_t c = pair ? cc - 1 : cc;  // a pair record is column c's record plus what column c+1 needs
        const uint32_t b0 = l_colptr[c] + 1, e0 = l_colptr[c + 1];
        T.push_back((e0 - b0) | (pair ? kSkPairFlag : 0u)); T.push_back(pos(l_colptr[c])); T.push_back(pos(c)); T.push_back(pos((uint32_t)perm[c]));
        for (uint32_t q = b0; q < e0; q++) T.push_back(pos(q));
        for (uint32_t q = b0; q < e0; q++) T.push_back(pos(l_rowidx[q]));
        if (pair) {
            for (uint32_t q = l_colptr[cc] + 1; q < l_colptr[cc + 1]; q++) T.push_back(pos(q));
            T.push_back(pos(l_colptr[cc])); T.push_back(pos((uint32_t)perm[cc]));
            cc--;
        }
        pad4();
    }
    T.insert(T.end(), 4, 0u);
    k.ok = true;
}

void Topology::fill_info(fk_topology_info* info) const {
    std::memset(info, 0, sizeof(*info));
    info->n_vars = n_vars; info->n_expr = n_expr; info->n_free = n_free; info->n_rows = n_rows;
    info->jac_nnz = jac_nnz;
    info->aug_nnz = jac_nnz + n_free;
    info->r_nnz = (uint32_t)r_rowidx.size();
    info->etree_height = etree_height;
    info->path = path; info->tile = tile; info->smem_bytes = smem_bytes;
    info->chol_flops = chol_flops;
    info->eval_bytes = (uint32_t)std::min<uint64_t>(eval_bytes, 0xFFFFFFFFu);
}

}  // namespace fk
