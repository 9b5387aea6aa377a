// ORACLE — TEST INFRASTRUCTURE ONLY.  Built on its own into oracle/liborc_twophase_sens.so (orc_twophase_sens_ffi.py),
// together with orc_twophase.cpp.
// The sensitivity report of a two-phase result (include/lpx.h, "Sensitivity analysis of a two-phase result") as plain
// sequential loops: every max / min scans in index order with a strict > / <, which is the report's tie rule (-0.0 ==
// +0.0, lowest index wins).  The report reads the full-width tableau, artificial columns included, which orc_two_phase
// does not return.  So each LP is solved by orc_two_phase with its whole pivot list, and the list is replayed with the
// oracle's pivot on the normalised tableau built in the definition's order of terms: Phase I and drive-out pivots on
// rows 0..m+1, Phase II pivots on rows 0..m, every column.  A pivot updates each row from that row and the pivot row
// alone, so rows 0..m of the replay are the solve's, bit for bit.
// Not the reference's: the reference has no two-phase method.
#include <cmath>
#include <limits>
#include <vector>

#include "orc_solvers.hpp"

extern "C" void orc_two_phase(int count, int m, int n, int sense, const double* A, const int* rel, const double* b,
                              const double* c, int max_iterations, int pivots_cap, int* status, int* phase1,
                              int* n_pivots, int* pivots, int* basis, double* x, double* z, double* T_out);

namespace {

const double EPS = 1e-9;

struct Best {
    bool have = false;
    double v = 0.0;
    void max(double c) {
        if (!have || c > v) v = c, have = true;
    }
    void min(double c) {
        if (!have || c < v) v = c, have = true;
    }
};

// One LP: its solve's status, basis and pivot list (p1 Phase I pivots, drive-out included, of np) -> rep[4m + 3n].
void report_one(int m, int n, int sense, const double* Aq, const int* rel, const double* bq, const double* cq,
                int status, const int* B, const int* plog, int p1, int np, double* rep) {
    const size_t stride = 4 * (size_t)m + 3 * (size_t)n;
    if (status != 0) {
        for (size_t e = 0; e < stride; e++) rep[e] = std::numeric_limits<double>::quiet_NaN();
        return;
    }
    const double INF = std::numeric_limits<double>::infinity();
    // normalisation and column numbering
    int s = 0;
    for (int i = 0; i < m; i++) s += (rel && rel[i] == 2) ? 0 : 1;
    const int ns = n + s;
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
    for (int i = 0; i < m; i++) {
        for (int j = 0; j < n; j++) at(i, j) = flip[i] ? -Aq[(size_t)i * n + j] : Aq[(size_t)i * n + j];
        at(i, rhs) = flip[i] ? -bq[i] : bq[i];
        if (slk[i] >= 0) at(i, slk[i]) = art[i] >= 0 ? -1.0 : 1.0;
        if (art[i] >= 0) at(i, art[i]) = 1.0;
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
    for (int k = 0; k < np; k++) orc::pivot(T.data(), k < p1 ? rows : m + 1, W, plog[2 * k + 1], plog[2 * k]);

    std::vector<int> rowof(W, -1);
    for (int r = 0; r < m; r++) rowof[B[r]] = r;
    const double* z = T.data() + (size_t)m * W;
    for (int i = 0; i < m; i++) {
        const int u = art[i] >= 0 ? art[i] : slk[i];  // the column that started as +e_i of the normalised row
        const bool f = flip[i] != 0;
        Best lo, hi;
        for (int r = 0; r < m; r++) {
            const double g = f ? -at(r, u) : at(r, u);
            if (B[r] < ns) {
                if (g > EPS) lo.max(-(at(r, rhs) / g));
                else if (g < -EPS) hi.min(-(at(r, rhs) / g));
            } else if (std::fabs(g) > EPS) {  // an artificial basic in a redundant row must stay at zero
                lo.max(-(at(r, rhs) / g));
                hi.min(-(at(r, rhs) / g));
            }
        }
        const double y = f ? -z[u] : z[u];
        rep[i] = sense == 1 ? -y : y;
        rep[m + i] = slk[i] >= 0 && rowof[slk[i]] >= 0 ? at(rowof[slk[i]], rhs) : 0.0;
        rep[2 * m + i] = lo.have ? bq[i] + lo.v : -INF;
        rep[3 * m + i] = hi.have ? bq[i] + hi.v : INF;
    }
    double* o = rep + 4 * (size_t)m;
    for (int j = 0; j < n; j++) {
        const double d = z[j];
        const int r = rowof[j];
        double l, h;
        if (r < 0) {
            l = sense == 0 ? -INF : cq[j] - d;
            h = sense == 0 ? cq[j] + d : INF;
        } else {
            Best lo, hi;
            for (int k = 0; k < ns; k++) {  // the artificial columns never take part
                if (rowof[k] >= 0) continue;
                const double al = at(r, k);
                if (al > EPS) lo.max(-(z[k] / al));
                else if (al < -EPS) hi.min(-(z[k] / al));
            }
            if (sense == 0) {
                l = lo.have ? cq[j] + lo.v : -INF;
                h = hi.have ? cq[j] + hi.v : INF;
            } else {
                l = hi.have ? cq[j] - hi.v : -INF;
                h = lo.have ? cq[j] - lo.v : INF;
            }
        }
        o[j] = d;
        o[n + j] = l;
        o[2 * (size_t)n + j] = h;
    }
}

}  // namespace

// orc_two_phase's arguments and outputs (none NULL), plus report [count][4m + 3n]: the sensitivity record of each LP,
// NaNs unless OPTIMAL.
extern "C" void orc_two_phase_sensitivity(int count, int m, int n, int sense, const double* A, const int* rel,
                                          const double* b, const double* c, int max_iterations, int pivots_cap,
                                          int* status, int* phase1, int* n_pivots, int* pivots, int* basis, double* x,
                                          double* z, double* T_out, double* report) {
    int s = 0;
    for (int i = 0; i < m; i++) s += (rel && rel[i] == 2) ? 0 : 1;
    const size_t stride = 4 * (size_t)m + 3 * (size_t)n, tsize = (size_t)(m + 1) * (n + s + 1);
    const int cap = (max_iterations > 0 ? max_iterations : 0) + m;  // drive-out pivots can go past the limit
    std::vector<int> plog((size_t)cap * 2);
    for (int q = 0; q < count; q++) {
        const double* Aq = A + (size_t)q * m * n;
        const double* bq = b + (size_t)q * m;
        const double* cq = c + (size_t)q * n;
        int* Bq = basis + (size_t)q * m;
        orc_two_phase(1, m, n, sense, Aq, rel, bq, cq, max_iterations, cap, status + q, phase1 + q, n_pivots + q,
                      plog.data(), Bq, x + (size_t)q * n, z + q, T_out + q * tsize);
        for (int k = 0; k < 2 * pivots_cap; k++) pivots[(size_t)q * pivots_cap * 2 + k] = k < 2 * cap ? plog[k] : -1;
        report_one(m, n, sense, Aq, rel, bq, cq, status[q], Bq, plog.data(), phase1[q], n_pivots[q],
                   report + q * stride);
    }
}
