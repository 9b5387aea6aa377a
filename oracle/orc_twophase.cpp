// ORACLE — TEST INFRASTRUCTURE ONLY.  Built on its own into oracle/liborc_twophase.so (orc_twophase_ffi.py).
// Two-phase Simplex (include/lpx.h, "Two-phase Simplex") as plain sequential loops: the normalised tableau built in
// the definition's order of terms, ChooseEntering as the oracle's choose_entering scans (strict <, lowest index,
// NaN never taken) on a chosen row and column range, the oracle's choose_leaving and pivot (orc_simplex.cpp).
// Not the reference's: the reference has no two-phase method.
#include <cmath>
#include <vector>

#include "orc_solvers.hpp"

namespace {

enum { OPTIMAL = 0, UNBOUNDED = 1, INFEASIBLE = 2, ITER_LIMIT = -3 };
const double EPS = 1e-9;

// PrimalSimplex.ChooseEntering on row zr over columns 0..ncols-1
int choose_entering_row(const double* T, int width, int zr, int ncols) {
    const double* z = T + (size_t)zr * width;
    int best = -1;
    double min_val = -EPS;
    for (int j = 0; j < ncols; j++)
        if (z[j] < min_val) {
            min_val = z[j];
            best = j;
        }
    return best;
}

}  // namespace

extern "C" {

// `count` LPs of one shape: A [count][m][n], b [count][m], c [count][n], rel [m] (NULL: all LE).  Outputs, none NULL:
// status, phase1, n_pivots [count], pivots [count][pivots_cap][2] ((-1, -1) past the last), basis [count][m],
// x [count][n], z [count], T_out [count][m + 1][n + s + 1].
void orc_two_phase(int count, int m, int n, int sense, const double* A, const int* rel, const double* b,
                   const double* c, int max_iterations, int pivots_cap, int* status, int* phase1, int* n_pivots,
                   int* pivots, int* basis, double* x, double* z, double* T_out) {
    int s = 0;
    for (int i = 0; i < m; i++) s += (rel && rel[i] == 2) ? 0 : 1;
    const int ns = n + s;
    for (int q = 0; q < count; q++) {
        const double* Aq = A + (size_t)q * m * n;
        const double* bq = b + (size_t)q * m;
        const double* cq = c + (size_t)q * n;
        // normalisation and column numbering
        std::vector<int> flip(m), slk(m, -1), art(m, -1);
        int sk = n, a = 0;
        for (int i = 0; i < m; i++) {
            const int rl = rel ? rel[i] : 0;
            flip[i] = bq[i] < 0.0;
            const int rn = (flip[i] && rl != 2) ? 1 - rl : rl;
            if (rl != 2) slk[i] = sk++;
            if (rn != 0) art[i] = ns + a++;
        }
        const int W = ns + a + 1, rhs = W - 1, rows = m + 2;
        std::vector<double> T((size_t)rows * W, 0.0);
        auto at = [&](int r, int k) -> double& { return T[(size_t)r * W + k]; };
        std::vector<int> B(m);
        double S = 0.0;
        for (int i = 0; i < m; i++) {
            for (int j = 0; j < n; j++) at(i, j) = flip[i] ? -Aq[(size_t)i * n + j] : Aq[(size_t)i * n + j];
            at(i, rhs) = flip[i] ? -bq[i] : bq[i];
            if (slk[i] >= 0) at(i, slk[i]) = art[i] >= 0 ? -1.0 : 1.0;
            if (art[i] >= 0) {
                at(i, art[i]) = 1.0;
                S += at(i, rhs);
            }
            B[i] = art[i] >= 0 ? art[i] : slk[i];
        }
        for (int j = 0; j < n; j++) {
            double cj = cq[j];
            if (sense == 1) cj = -cj;
            at(m, j) = -cj;
        }
        for (int j = 0; j < W; j++) {
            if (j >= ns && j != rhs) continue;
            double w = 0.0;
            for (int i = 0; i < m; i++)
                if (art[i] >= 0) w -= at(i, j);
            at(m + 1, j) = w;
        }

        int np = 0, p1 = 0;
        int* plog = pivots + (size_t)q * pivots_cap * 2;
        for (int k = 0; k < 2 * pivots_cap; k++) plog[k] = -1;
        auto pivot_on = [&](int l, int e, int nrows) {
            orc::pivot(T.data(), nrows, W, l, e);
            B[l] = e;
            if (np < pivots_cap) {
                plog[2 * np] = e;
                plog[2 * np + 1] = l;
            }
            np++;
        };
        // 0: iteration limit, 1: no entering column, 2: no leaving row
        auto simplex = [&](int zr, int ncols, int nrows, bool ph1) {
            while (true) {
                if (np + 1 > max_iterations) return 0;
                const int e = choose_entering_row(T.data(), W, zr, ncols);
                if (e < 0) return 1;
                const int l = orc::choose_leaving(T.data(), m, W, e, 1e-9);
                if (l < 0) return 2;
                pivot_on(l, e, nrows);
                if (ph1) p1++;
            }
        };
        int st;
        const int why1 = simplex(m + 1, W - 1, rows, true);
        const double tol = 1e-9 * (1.0 + S);
        if (why1 == 0) {
            st = ITER_LIMIT;
        } else if (!(at(m + 1, rhs) >= -tol)) {
            st = INFEASIBLE;
        } else {
            for (int r = 0; r < m; r++) {
                if (B[r] < ns) continue;
                int e = -1;
                for (int j = 0; j < ns && e < 0; j++)
                    if (std::fabs(at(r, j)) > EPS) e = j;
                if (e >= 0) {
                    pivot_on(r, e, rows);
                    p1++;
                }
            }
            const int why2 = simplex(m, ns, m + 1, false);
            st = why2 == 0 ? ITER_LIMIT : (why2 == 1 ? OPTIMAL : UNBOUNDED);
        }

        status[q] = st;
        phase1[q] = p1;
        n_pivots[q] = np;
        double* xq = x + (size_t)q * n;
        for (int j = 0; j < n; j++) xq[j] = 0.0;
        for (int i = 0; i < m; i++) {
            basis[(size_t)q * m + i] = B[i];
            if (B[i] < n) xq[B[i]] = at(i, rhs);
        }
        z[q] = at(m, rhs);
        double* To = T_out + (size_t)q * (m + 1) * (ns + 1);
        for (int i = 0; i <= m; i++)
            for (int j = 0; j <= ns; j++) To[(size_t)i * (ns + 1) + j] = at(i, j < ns ? j : rhs);
    }
}

}  // extern "C"
