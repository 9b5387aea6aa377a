// ORACLE — TEST INFRASTRUCTURE ONLY.  Built on its own into oracle/liborc_sensitivity.so (orc_sens_ffi.py).
// The sensitivity report of include/lpx.h ("Sensitivity analysis of an optimal Primal Simplex result") as plain
// sequential loops: every max / min scans in index order with a strict > / <, which is the report's tie rule
// (-0.0 == +0.0, lowest index wins).  It reads a tableau + basis, so it applies to the oracle's final tableaux and to
// tableaux downloaded from the GPU alike.  Not the reference's SensitivityAnalysis (which reads the z-row from row 0).
#include <cmath>
#include <limits>
#include <vector>


namespace {

const double EPS = 1e-9;
const double INF = std::numeric_limits<double>::infinity();

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

void one(int m, int n, int sense, const int* rel, const double* b, const double* c, int status, const int* basis,
         const double* T, double* rep) {
    const size_t stride = 4 * (size_t)m + 3 * (size_t)n;
    if (status != 0) {
        for (size_t e = 0; e < stride; e++) rep[e] = std::numeric_limits<double>::quiet_NaN();
        return;
    }
    std::vector<int> row1(m);
    int mm = 0;
    for (int i = 0; i < m; i++) {
        row1[i] = mm;
        mm += (rel && rel[i] == 2) ? 2 : 1;
    }
    const int W = n + mm + 1;
    std::vector<int> rowof(W, -1);
    for (int r = 0; r < mm; r++) rowof[basis[r]] = r;
    const double* z = T + (size_t)mm * W;
    auto at = [&](int r, int k) { return T[(size_t)r * W + k]; };

    for (int i = 0; i < m; i++) {
        const bool eq = rel && rel[i] == 2;
        const int c1 = n + row1[i], c2 = c1 + 1;
        const double u = eq ? z[c1] - z[c2] : z[c1];
        Best lo, hi;
        for (int r = 0; r < mm; r++) {
            const double g = eq ? at(r, c1) - at(r, c2) : at(r, c1);
            if (g > EPS) lo.max(-(at(r, W - 1) / g));
            else if (g < -EPS) hi.min(-(at(r, W - 1) / g));
        }
        rep[i] = sense == 1 ? -u : u;
        rep[m + i] = rowof[c1] >= 0 ? at(rowof[c1], W - 1) : 0.0;
        rep[2 * m + i] = lo.have ? b[i] + lo.v : -INF;
        rep[3 * m + i] = hi.have ? b[i] + hi.v : INF;
    }
    double* o = rep + 4 * (size_t)m;
    for (int j = 0; j < n; j++) {
        const double d = z[j];
        const int r = rowof[j];
        double l, h;
        if (r < 0) {
            l = sense == 0 ? -INF : c[j] - d;
            h = sense == 0 ? c[j] + d : INF;
        } else {
            Best lo, hi;
            for (int k = 0; k < W - 1; k++) {
                if (rowof[k] >= 0) continue;
                const double a = at(r, k);
                if (a > EPS) lo.max(-(z[k] / a));
                else if (a < -EPS) hi.min(-(z[k] / a));
            }
            if (sense == 0) {
                l = lo.have ? c[j] + lo.v : -INF;
                h = hi.have ? c[j] + hi.v : INF;
            } else {
                l = hi.have ? c[j] - hi.v : -INF;
                h = lo.have ? c[j] - lo.v : INF;
            }
        }
        o[j] = d;
        o[n + j] = l;
        o[2 * (size_t)n + j] = h;
    }
}

}  // namespace

// `count` final tableaux of one shape: b[count][m], c[count][n], status[count], basis[count][m'],
// tableau[count][m'+1][n+m'+1]; report[count][4m + 3n], NaNs unless status is OPTIMAL (0).
extern "C" void orc_sensitivity(int count, int m, int n, int sense, const int* rel, const double* b, const double* c,
                                const int* status, const int* basis, const double* tableau, double* report) {
    int mm = 0;
    for (int i = 0; i < m; i++) mm += (rel && rel[i] == 2) ? 2 : 1;
    const size_t tsize = (size_t)(mm + 1) * (n + mm + 1), stride = 4 * (size_t)m + 3 * (size_t)n;
    for (int k = 0; k < count; k++)
        one(m, n, sense, rel, b + (size_t)k * m, c + (size_t)k * n, status[k], basis + (size_t)k * mm,
            tableau + (size_t)k * tsize, report + (size_t)k * stride);
}
