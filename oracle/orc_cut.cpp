// ORACLE — TEST INFRASTRUCTURE ONLY.  Built on its own into oracle/liborc_cut.so (orc_cut_ffi.py).
// The numbers of CuttingPlane.Solve (R/Models/CuttingPlane.cs:13-164) for one IP, laid out as one instance of
// lpx_cutting_plane_batched (include/lpx.h, "Gomory cutting plane").  The loop of orc_cutting.cpp restated without its
// text, on the oracle's own primal_simplex with per-iteration formatting off and a caller-set iteration limit, and
// with the status and pivots of the round that threw recorded (CutTrace does not keep them).  Its cuts are checked
// against orc_cutting.cpp's text path and the golden cases (tests/test_cutting_plane_cpu.py).
#include <cmath>
#include <vector>

#include "orc_solvers.hpp"

using namespace orc;

extern "C" int orc_cut_solve(int m, int n, int sense, const double* A, const int* rel, const double* b, const double* c,
                             int max_iterations, int* end, int* n_rounds, int* n_cuts, int* lp_status, int* lp_pivots,
                             int* frac_var, int* cut_row, double* cut_a, double* cut_b, int* basis, double* x,
                             double* z, double* tableau) {
    const int R = 50;
    const double Eps = 1e-9;
    Problem model;
    model.sense = sense;
    model.c.assign(c, c + n);
    int mm = 0;
    for (int i = 0; i < m; i++) {
        Row r;
        r.a.assign(A + (size_t)i * n, A + (size_t)(i + 1) * n);
        r.rel = rel ? rel[i] : LE;
        r.b = b[i];
        model.rows.push_back(r);
        mm += r.rel == EQ ? 2 : 1;
    }
    PrimalOptions opt;
    opt.max_iterations = max_iterations;
    opt.format_every_iteration = false;

    std::vector<int> st, piv, fv, crow;
    std::vector<std::vector<double>> ca;
    std::vector<double> cb;
    int e = CUT_INCOMPLETE;
    Outcome final_lp;
    for (int round = 0; round < R; round++) {
        Outcome lp;
        Trace t;
        try {
            lp = primal_simplex(model, Sink(), &t, opt);
        } catch (const SolveError& err) {  // CuttingPlane.cs catches it and stops
            st.push_back(err.code);
            piv.push_back((int)t.enter.size());
            e = CUT_LP_ERROR;
            break;
        }
        st.push_back(t.status);  // an UNBOUNDED round goes on: its x is read all the same
        piv.push_back((int)t.enter.size());
        int frac = -1;
        for (int j = 0; j < n; j++) {
            const double f = lp.x[j] - std::floor(lp.x[j]);
            if (f > Eps && f < 1 - Eps) {
                frac = j;
                break;
            }
        }
        if (frac == -1) {
            e = CUT_INTEGER;
            final_lp = lp;
            break;
        }
        int row = -1;  // the row BELOW the fractional variable's (CuttingPlane.cs:113)
        for (int i = 0; i < (int)lp.basis.size(); i++)
            if (lp.basis[i] == frac) {
                row = i + 1;
                break;
            }
        const double* trow = lp.T.data() + (size_t)row * lp.cols;
        Row cut;
        cut.a.assign(n, 0.0);
        cut.rel = LE;
        for (int j = 0; j < n; j++) {
            const double fj = trow[j] - std::floor(trow[j]);
            if (fj > Eps) cut.a[j] = fj;
        }
        const double rhs = trow[lp.cols - 1];
        cut.b = rhs - std::floor(rhs);
        model.rows.push_back(cut);
        fv.push_back(frac);
        crow.push_back(row);
        ca.push_back(cut.a);
        cb.push_back(cut.b);
    }

    const int rounds = (int)st.size(), cuts = (int)cb.size();
    *end = e;
    if (n_rounds) *n_rounds = rounds;
    if (n_cuts) *n_cuts = cuts;
    for (int r = 0; r < R; r++) {
        if (lp_status) lp_status[r] = r < rounds ? st[r] : 3;  // LPX_RUNNING
        if (lp_pivots) lp_pivots[r] = r < rounds ? piv[r] : 0;
        if (frac_var) frac_var[r] = r < cuts ? fv[r] : -1;
        if (cut_row) cut_row[r] = r < cuts ? crow[r] : -1;
        if (cut_b) cut_b[r] = r < cuts ? cb[r] : 0.0;
        if (cut_a)
            for (int j = 0; j < n; j++) cut_a[(size_t)r * n + j] = r < cuts ? ca[r][j] : 0.0;
    }
    const bool integral = e == CUT_INTEGER;
    if (basis)
        for (int i = 0; i < mm + R - 1; i++) basis[i] = integral && i < (int)final_lp.basis.size() ? final_lp.basis[i] : 0;
    if (x)
        for (int j = 0; j < n; j++) x[j] = integral ? final_lp.x[j] : 0.0;
    if (z) *z = integral ? final_lp.z : 0.0;
    if (tableau) {
        const size_t used = integral ? final_lp.T.size() : 0, total = (size_t)(mm + R) * (n + mm + R);
        for (size_t k = 0; k < total; k++) tableau[k] = k < used ? final_lp.T[k] : 0.0;
    }
    return 0;
}
