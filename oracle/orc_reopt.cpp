// ORACLE — TEST INFRASTRUCTURE ONLY.  Built on its own into oracle/liborc_reopt.so (orc_reopt_ffi.py).
// Re-optimization of an optimal Primal Simplex result (include/lpx.h, "Re-optimization"): the four tableau edits as
// plain sequential loops in the definition's order, then the oracle's own loops: primal_core (orc_simplex.cpp) for
// COST / COL and Mode B's dual_core (orc_pooled.cpp) for RHS / ROW.  Not the reference's: the reference has no
// re-optimization.
#include <algorithm>
#include <cmath>
#include <limits>
#include <memory>
#include <queue>
#include <vector>

#include "orc_solvers.hpp"

namespace orc {
namespace {
thread_local std::vector<int>* g_pivot_log = nullptr;
}
void logged_pivot(double* T, int rows, int width, int row, int col) {
    if (g_pivot_log) {
        g_pivot_log->push_back(col);
        g_pivot_log->push_back(row);
    }
    pivot(T, rows, width, row, col);
}
}  // namespace orc

// Mode B's bound-row build (extend_tableau) and its Dual Simplex loop (dual_core) have internal linkage in
// orc_pooled.cpp.  This translation unit includes that file to run both unchanged; dual_core's one call of pivot()
// goes through logged_pivot, which records the (entering, leaving) pairs dual_core itself does not keep.
#define pivot(...) logged_pivot(__VA_ARGS__)
#include "orc_pooled.cpp"
#undef pivot

namespace {

using orc::ERR_ITER_LIMIT;
enum { RHS = 1, COST = 2, ROW = 3, COL = 4 };

size_t payload_stride(int kind, int m, int n) {
    return kind == RHS ? m : kind == COST ? n : kind == ROW ? n + 2 : m + 1;
}

struct Query {
    int rows, cols;
    std::vector<double> T;
    std::vector<int> basis;
};

// The query's working tableau from base tableau Tb (mm + 1 rows, W = n + mm + 1 columns) and basis bb.
Query build(int kind, int m, int n, int sense, const int* rel, int mm, const double* Tb, const int* bb,
            const double* pay) {
    const int W = n + mm + 1, rhs = W - 1;
    auto bt = [&](int r, int k) { return Tb[(size_t)r * W + k]; };
    std::vector<int> s1(m);
    for (int i = 0, i1 = 0; i < m; i++) {
        s1[i] = n + i1;
        i1 += (rel && rel[i] == 2) ? 2 : 1;
    }
    auto is_eq = [&](int i) { return rel && rel[i] == 2; };
    Query q;
    if (kind == RHS || kind == COST) {
        q.rows = mm + 1;
        q.cols = W;
        q.T.assign(Tb, Tb + (size_t)q.rows * W);
        q.basis.assign(bb, bb + mm);
        auto at = [&](int r, int k) -> double& { return q.T[(size_t)r * W + k]; };
        if (kind == RHS) {
            for (int i = 0; i < m; i++) {
                const double d = pay[i];
                if (d == 0.0) continue;
                for (int r = 0; r <= mm; r++) {
                    at(r, rhs) += d * at(r, s1[i]);
                    if (is_eq(i)) at(r, rhs) -= d * at(r, s1[i] + 1);
                }
            }
        } else {
            for (int j = 0; j < n; j++) {
                if (pay[j] == 0.0) continue;
                const double delta = sense == 1 ? -pay[j] : pay[j];
                int r = -1;
                for (int i = 0; i < mm; i++)
                    if (q.basis[i] == j) r = i;
                if (r >= 0)
                    for (int k = 0; k < W; k++) at(mm, k) += delta * at(r, k);
                at(mm, j) -= delta;
            }
        }
        return q;
    }
    if (kind == ROW) {
        q.rows = mm + 2;
        q.cols = W + 1;
        q.T.assign((size_t)q.rows * q.cols, 0.0);
        auto at = [&](int r, int k) -> double& { return q.T[(size_t)r * q.cols + k]; };
        for (int i = 0; i <= mm; i++) {  // old rows and the z-row: the old RHS position becomes the new slack
            const int o = i < mm ? i : mm + 1;
            for (int k = 0; k < rhs; k++) at(o, k) = bt(i, k);
            at(o, rhs) = 0.0;
            at(o, W) = bt(i, rhs);
        }
        const bool ge = pay[n] == 1.0;
        for (int k = 0; k < n; k++) at(mm, k) = pay[k];
        for (int k = n; k < rhs; k++) at(mm, k) = 0.0;
        at(mm, W) = pay[n + 1];
        if (ge) {
            for (int k = 0; k < rhs; k++) at(mm, k) = -at(mm, k);
            at(mm, W) = -at(mm, W);
        }
        at(mm, rhs) = 1.0;
        for (int r = 0; r < mm; r++) {
            const int j = bb[r];
            if (j >= n || pay[j] == 0.0) continue;
            const double a = ge ? -pay[j] : pay[j];
            for (int k = 0; k < rhs; k++) at(mm, k) -= a * bt(r, k);
            at(mm, W) -= a * bt(r, rhs);
        }
        q.basis.assign(bb, bb + mm);
        q.basis.push_back(rhs);
        return q;
    }
    // COL: the new variable at column n
    q.rows = mm + 1;
    q.cols = W + 1;
    q.T.assign((size_t)q.rows * q.cols, 0.0);
    auto at = [&](int r, int k) -> double& { return q.T[(size_t)r * q.cols + k]; };
    for (int r = 0; r <= mm; r++) {
        for (int k = 0; k < n; k++) at(r, k) = bt(r, k);
        for (int k = n; k < W; k++) at(r, k + 1) = bt(r, k);
        at(r, n) = 0.0;
    }
    const double cp = sense == 1 ? -pay[m] : pay[m];
    at(mm, n) = -cp;
    for (int i = 0; i < m; i++) {
        const double a = pay[i];
        if (a == 0.0) continue;
        for (int r = 0; r <= mm; r++) {
            at(r, n) += a * bt(r, s1[i]);
            if (is_eq(i)) at(r, n) -= a * bt(r, s1[i] + 1);
        }
    }
    q.basis.resize(mm);
    for (int i = 0; i < mm; i++) q.basis[i] = bb[i] >= n ? bb[i] + 1 : bb[i];
    return q;
}

}  // namespace

extern "C" {

// `count` queries of one kind; query q reads base src[q] (src NULL: base q).  Bases: base_status[.],
// base_basis[.][m'], base_T[.][m'+1][n+m'+1].  Outputs as lpx_reoptimize_batched_dev; pivots: pivots_cap pairs per
// query (entries past the query's pivots are left alone); T_out nullable.
void orc_reopt(int kind, int count, int m, int n, int sense, const int* rel, const int* base_status,
               const int* base_basis, const double* base_T, const int* src, const double* payload, int max_iterations,
               int* status, int* n_pivots, int* pivots, int pivots_cap, int* basis, double* x, double* z,
               double* T_out) {
    int mm = 0;
    for (int i = 0; i < m; i++) mm += (rel && rel[i] == 2) ? 2 : 1;
    const size_t base_tsize = (size_t)(mm + 1) * (n + mm + 1), stride = payload_stride(kind, m, n);
    const int rows = mm + 1 + (kind == ROW), cols = n + mm + 1 + (kind == ROW || kind == COL);
    const int nx = kind == COL ? n + 1 : n, mo = rows - 1;
    for (int q = 0; q < count; q++) {
        const int s = src ? src[q] : q;
        int* bo = basis + (size_t)q * mo;
        double* xo = x + (size_t)q * nx;
        double* To = T_out ? T_out + (size_t)q * rows * cols : nullptr;
        if (base_status[s] != 0) {
            status[q] = base_status[s];
            n_pivots[q] = 0;
            std::fill(bo, bo + mo, 0);
            std::fill(xo, xo + nx, 0.0);
            z[q] = 0.0;
            if (To) std::fill(To, To + (size_t)rows * cols, 0.0);
            continue;
        }
        Query Q = build(kind, m, n, sense, rel, mm, base_T + (size_t)s * base_tsize, base_basis + (size_t)s * mm,
                        payload + (size_t)q * stride);
        int np = 0, st;
        std::vector<int> log;
        if (kind == RHS || kind == ROW) {
            orc::g_pivot_log = &log;
            st = orc::dual_core(Q.T, Q.rows, Q.cols, Q.basis, &np);
            orc::g_pivot_log = nullptr;
        } else {
            log.assign((size_t)2 * std::max(pivots_cap, 1), -1);
            st = orc::primal_core(Q.T.data(), mo, Q.cols, Q.basis.data(), max_iterations, &np, log.data(), pivots_cap);
        }
        status[q] = st == ERR_ITER_LIMIT ? ERR_ITER_LIMIT : st;
        n_pivots[q] = np;
        for (int k = 0; k < std::min(np, pivots_cap); k++) {
            pivots[((size_t)q * pivots_cap + k) * 2] = log[2 * k];
            pivots[((size_t)q * pivots_cap + k) * 2 + 1] = log[2 * k + 1];
        }
        std::copy(Q.basis.begin(), Q.basis.end(), bo);
        std::fill(xo, xo + nx, 0.0);
        for (int i = 0; i < mo; i++)
            if (Q.basis[i] < nx) xo[Q.basis[i]] = Q.T[(size_t)i * cols + cols - 1];
        z[q] = Q.T[(size_t)mo * cols + cols - 1];
        if (To) std::copy(Q.T.begin(), Q.T.end(), To);
    }
}

// Mode B's child tableau (extend_tableau, orc_pooled.cpp) of a parent tableau rows x cols: T_out (rows + 1) x
// (cols + 1), basis_out rows entries.
void orc_extend_tableau(int rows, int cols, const double* T, const int* basis, int var, int side, double val,
                        double* T_out, int* basis_out) {
    orc::PNode par, ch;
    par.rows = rows;
    par.cols = cols;
    par.T.assign(T, T + (size_t)rows * cols);
    par.basis.assign(basis, basis + rows - 1);
    orc::extend_tableau(par, var, side, val, ch);
    std::copy(ch.T.begin(), ch.T.end(), T_out);
    std::copy(ch.basis.begin(), ch.basis.end(), basis_out);
}

// Mode B's Dual Simplex loop (dual_core) in place; returns the status, pivots as (entering, leaving) pairs.
int orc_dual_core(int rows, int cols, double* T, int* basis, int* n_pivots, int* pivots, int pivots_cap) {
    std::vector<double> t(T, T + (size_t)rows * cols);
    std::vector<int> b(basis, basis + rows - 1), log;
    orc::g_pivot_log = &log;
    const int st = orc::dual_core(t, rows, cols, b, n_pivots);
    orc::g_pivot_log = nullptr;
    for (int k = 0; k < std::min(*n_pivots, pivots_cap); k++) {
        pivots[2 * k] = log[2 * k];
        pivots[2 * k + 1] = log[2 * k + 1];
    }
    std::copy(t.begin(), t.end(), T);
    std::copy(b.begin(), b.end(), basis);
    return st;
}

}  // extern "C"
