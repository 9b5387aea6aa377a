// ORACLE — TEST INFRASTRUCTURE ONLY.  Built on its own into oracle/liborc_param.so (orc_param_ffi.py).
// Parametric analysis of an optimal Primal Simplex result (include/lpx.h, "Parametric analysis") as plain sequential
// loops: the direction column / row built in the definition's order of terms, every minimum a scan in index order with
// a strict < (so -0.0 == +0.0 and the lowest index wins), the oracle's choose_leaving (orc_simplex.cpp) for the
// Primal Simplex leaving row, Mode B's Dual Simplex entering scan (dual_core, orc_pooled.cpp) for the entering column,
// and the oracle's pivot.  Not the reference's: the reference has no parametric analysis.
#include <algorithm>
#include <cmath>
#include <limits>
#include <vector>

#include "orc_solvers.hpp"

namespace {

enum { RHS = 1, COST = 2 };
enum { REACHED = 0, UNBOUNDED = 1, INFEASIBLE = 2, SEG_LIMIT = 3, NO_BASE = 4 };
const double EPS = 1e-9;
const double INF = std::numeric_limits<double>::infinity();

// min{v_i} over the candidates offered in index order: strict <, NaN never taken
struct Min {
    int i = -1;
    double v = 0.0;
    void offer(double c, int k) {
        if (c != c) return;
        if (i < 0 || c < v) v = c, i = k;
    }
};

}  // namespace

extern "C" {

// `count` queries of one kind; query q reads base src[q] (src NULL: base q).  Bases: base_status[.],
// base_basis[.][m'], base_T[.][m'+1][n+m'+1].  Outputs as lpx_parametric_batched_dev, none NULL: end, n_segments,
// n_pivots [count], segments [count][seg_cap][4+2n], seg_pivots [count][seg_cap][2], basis [count][m'],
// T_out [count][rows][cols] (lpx_parametric_dims).
void orc_param(int kind, int count, int m, int n, int sense, const int* rel, const int* base_status,
               const int* base_basis, const double* base_T, const int* src, const double* payload, int seg_cap,
               int* end, int* n_segments, int* n_pivots, double* segments, int* seg_pivots, int* basis,
               double* T_out) {
    int mm = 0;
    std::vector<int> s1(m);
    for (int i = 0; i < m; i++) {
        s1[i] = n + mm;
        mm += (rel && rel[i] == 2) ? 2 : 1;
    }
    const int W = n + mm + 1, rhs = W - 1;
    const int rows = mm + 1 + (kind == COST), cols = W + (kind == RHS);
    const size_t stride = (kind == RHS ? m : n) + 1, sstride = 4 + 2 * (size_t)n, tsize = (size_t)rows * cols;
    const size_t base_tsize = (size_t)(mm + 1) * W;
    for (int q = 0; q < count; q++) {
        const int s = src ? src[q] : q;
        const double* d = payload + (size_t)q * stride;
        const double theta_max = d[stride - 1];
        double* seg = segments + (size_t)q * seg_cap * sstride;
        int* spv = seg_pivots + (size_t)q * seg_cap * 2;
        int* bo = basis + (size_t)q * mm;
        double* To = T_out + (size_t)q * tsize;
        std::fill(seg, seg + (size_t)seg_cap * sstride, 0.0);
        std::fill(spv, spv + 2 * (size_t)seg_cap, -1);
        if (base_status[s] != 0) {
            end[q] = NO_BASE;
            n_segments[q] = 0;
            n_pivots[q] = 0;
            std::fill(bo, bo + mm, 0);
            std::fill(To, To + tsize, 0.0);
            continue;
        }
        const double* Tb = base_T + (size_t)s * base_tsize;
        std::vector<int> B(base_basis + (size_t)s * mm, base_basis + (size_t)(s + 1) * mm);
        std::vector<double> T(tsize, 0.0);
        auto at = [&](int r, int k) -> double& { return T[(size_t)r * cols + k]; };
        for (int r = 0; r <= mm; r++)
            for (int k = 0; k < W; k++) at(r, k) = Tb[(size_t)r * W + k];
        if (kind == RHS) {
            for (int r = 0; r <= mm; r++) {
                double g = 0.0;
                for (int i = 0; i < m; i++) {
                    if (d[i] == 0.0) continue;
                    g += d[i] * at(r, s1[i]);
                    if (rel && rel[i] == 2) g -= d[i] * at(r, s1[i] + 1);
                }
                at(r, W) = g;
            }
        } else {
            for (int j = 0; j < n; j++) {
                if (d[j] == 0.0) continue;
                const double delta = sense == 1 ? -d[j] : d[j];
                int r = -1;
                for (int i = 0; i < mm; i++)
                    if (B[i] == j) r = i;
                if (r >= 0)
                    for (int k = 0; k < W; k++) at(mm + 1, k) += delta * at(r, k);
                at(mm + 1, j) -= delta;
            }
        }
        auto basic_row = [&](int col) {
            for (int i = 0; i < mm; i++)
                if (B[i] == col) return i;
            return -1;
        };

        double th_lo = 0.0;
        int k = 0, e_end;
        while (true) {
            Min best;
            if (kind == RHS) {
                for (int r = 0; r < mm; r++)
                    if (at(r, W) < -EPS) best.offer(-(at(r, rhs) / at(r, W)), r);
            } else {
                for (int j = 0; j < rhs; j++)
                    if (basic_row(j) < 0 && at(mm + 1, j) < -EPS) best.offer(-(at(mm, j) / at(mm + 1, j)), j);
            }
            const double cand = best.i < 0 ? INF : best.v;
            const double th_end = cand < th_lo ? th_lo : cand;
            int stop = -1, pl = -1, pe = -1;
            double th_hi = th_end;
            if (th_end >= theta_max) {
                stop = REACHED;
                th_hi = theta_max;
            } else if (k + 1 == seg_cap) {
                stop = SEG_LIMIT;
            } else if (kind == RHS) {
                const int l = best.i;
                double best_ratio = INF;
                for (int j = 0; j < rhs; j++) {  // dual_core's entering scan
                    const double a = at(l, j);
                    if (a < -1e-9) {
                        const double ratio = at(mm, j) / (-a);
                        if (ratio < best_ratio - 1e-12) {
                            best_ratio = ratio;
                            pe = j;
                        }
                    }
                }
                if (pe < 0) stop = INFEASIBLE;
                else pl = l;
            } else {
                pl = orc::choose_leaving(T.data(), mm, cols, best.i, 1e-9);
                if (pl < 0) stop = UNBOUNDED;
                else pe = best.i;
            }
            double* rec = seg + (size_t)k * sstride;
            rec[0] = th_lo;
            rec[1] = th_hi;
            rec[2] = at(mm, rhs);
            rec[3] = kind == RHS ? at(mm, W) : at(mm + 1, rhs);
            for (int j = 0; j < n; j++) {
                const int r = basic_row(j);
                rec[4 + j] = r >= 0 ? at(r, rhs) : 0.0;
                rec[4 + n + j] = (kind == RHS && r >= 0) ? at(r, W) : 0.0;
            }
            spv[2 * k] = pl;
            spv[2 * k + 1] = pe;
            k++;
            if (stop >= 0) {
                e_end = stop;
                break;
            }
            orc::pivot(T.data(), rows, cols, pl, pe);
            B[pl] = pe;
            th_lo = th_end;
        }
        end[q] = e_end;
        n_segments[q] = k;
        n_pivots[q] = k - 1;
        std::copy(B.begin(), B.end(), bo);
        std::copy(T.begin(), T.end(), To);
    }
}

}  // extern "C"
