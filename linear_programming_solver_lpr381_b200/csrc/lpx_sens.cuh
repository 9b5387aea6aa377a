// lpx_sens.cuh — device side of the sensitivity report (shadow prices, slacks, RHS ranges, reduced costs, cost
// ranges) read from the final tableau of an OPTIMAL Primal Simplex solve.  The definition is in include/lpx.h;
// oracle/orc_sensitivity.cpp restates it as sequential loops, and every value here must equal it bit for bit.
#pragma once
#include "lpx_common.cuh"

namespace lpx {

// Candidate of one min / max reduction; i == INT_MAX marks an empty side.
struct SensBest {
    double v;
    int i;
};

// The tie rule of every reduction in the report, shared by the batched and the session kernels: -0.0 and +0.0
// compare equal (IEEE ==), and among equal values the lowest row / column index wins, so the result is the one a
// sequential scan with strict < / > in index order keeps, with the winner's own value (sign of zero included).
template <bool MAX>
__device__ __forceinline__ void sens_pick(SensBest& best, const SensBest& c) {
    if (c.i == INT_MAX) return;
    if (best.i == INT_MAX || (MAX ? c.v > best.v : c.v < best.v) || (c.v == best.v && c.i < best.i)) best = c;
}

template <bool MAX>
__device__ __forceinline__ SensBest sens_warp_reduce(SensBest b) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        SensBest c;
        c.v = __shfl_xor_sync(0xffffffffu, b.v, o);
        c.i = __shfl_xor_sync(0xffffffffu, b.i, o);
        sens_pick<MAX>(b, c);
    }
    return b;
}

__device__ __forceinline__ SensBest sens_empty() {
    SensBest e;
    e.v = 0.0;
    e.i = INT_MAX;
    return e;
}

__device__ __forceinline__ double sens_nan() { return __longlong_as_double(0x7ff8000000000000LL); }
__device__ __forceinline__ double sens_inf() { return __longlong_as_double(0x7ff0000000000000LL); }

// Row map entry of original constraint i: the expanded row i1 of its slack, negative -(i1 + 1) for an EQ row
// (whose second row i2 = i1 + 1 is the negated copy).
__device__ __forceinline__ int sens_row1(int e) { return e < 0 ? -e - 1 : e; }

// One row r of the RHS-range column reduction of a constraint: direction g, RHS beta.
__device__ __forceinline__ void sens_rhs_candidate(SensBest& lo, SensBest& hi, double beta, double g, int r) {
    if (g > LPX_EPS) {
        SensBest c;
        c.v = -__ddiv_rn(beta, g);
        c.i = r;
        sens_pick<true>(lo, c);
    } else if (g < -LPX_EPS) {
        SensBest c;
        c.v = -__ddiv_rn(beta, g);
        c.i = r;
        sens_pick<false>(hi, c);
    }
}

// Two-phase report: row r holds an artificial that stayed basic in a redundant row and must stay at zero, so a
// direction with |g| > EPS bounds the RHS change on both sides at the same value.
__device__ __forceinline__ void sens_rhs_candidate_both(SensBest& lo, SensBest& hi, double beta, double g, int r) {
    if (fabs(g) > LPX_EPS) {
        SensBest c;
        c.v = -__ddiv_rn(beta, g);
        c.i = r;
        sens_pick<true>(lo, c);
        sens_pick<false>(hi, c);
    }
}

// sigma_i * v of the two-phase report: an exact sign flip when row i was negated (b_i < 0).
__device__ __forceinline__ double sens_sign(double v, bool flip) {
    return flip ? __longlong_as_double(__double_as_longlong(v) ^ (long long)0x8000000000000000ULL) : v;
}

// One non-basic column k of the cost-range row reduction of a basic variable: entry alpha of its row, reduced
// cost d of column k.
__device__ __forceinline__ void sens_cost_candidate(SensBest& lo, SensBest& hi, double d, double alpha, int k) {
    if (alpha > LPX_EPS) {
        SensBest c;
        c.v = -__ddiv_rn(d, alpha);
        c.i = k;
        sens_pick<true>(lo, c);
    } else if (alpha < -LPX_EPS) {
        SensBest c;
        c.v = -__ddiv_rn(d, alpha);
        c.i = k;
        sens_pick<false>(hi, c);
    }
}

// shadow | slack | rhs_lo | rhs_hi entries of constraint i (u = raw z-row value of its slack direction).
__device__ __forceinline__ void sens_write_constraint(double* rep, int m, int i, int sense, double u, double slack,
                                                      const SensBest& lo, const SensBest& hi, double bi) {
    rep[i] = sense == 1 ? -u : u;
    rep[m + i] = slack;
    rep[2 * m + i] = lo.i == INT_MAX ? -sens_inf() : __dadd_rn(bi, lo.v);
    rep[3 * m + i] = hi.i == INT_MAX ? sens_inf() : __dadd_rn(bi, hi.v);
}

// reduced | cost_lo | cost_hi entries of decision variable j.
__device__ __forceinline__ void sens_write_variable(double* rep, int m, int n, int j, int sense, double d, bool basic,
                                                    const SensBest& lo, const SensBest& hi, double cj) {
    double* o = rep + 4 * (size_t)m;
    double l, h;
    if (!basic) {
        l = sense == 0 ? -sens_inf() : __dsub_rn(cj, d);
        h = sense == 0 ? __dadd_rn(cj, d) : sens_inf();
    } else if (sense == 0) {
        l = lo.i == INT_MAX ? -sens_inf() : __dadd_rn(cj, lo.v);
        h = hi.i == INT_MAX ? sens_inf() : __dadd_rn(cj, hi.v);
    } else {
        l = hi.i == INT_MAX ? -sens_inf() : __dsub_rn(cj, hi.v);
        h = lo.i == INT_MAX ? sens_inf() : __dsub_rn(cj, lo.v);
    }
    o[j] = d;
    o[n + j] = l;
    o[2 * (size_t)n + j] = h;
}

// Cost range of decision variable j by one warp: a reduction along its basic row r against the z-row (row mm),
// over the non-basic columns (rowof[k] < 0) left of the RHS.  Rows are ld doubles apart.
__device__ __forceinline__ void sens_variable_warp(const double* T, size_t ld, int W, int mm, int n, int m, int j,
                                                   int sense, const int* rowof, double cj, double* rep) {
    const int lane = threadIdx.x & 31;
    const double* z = T + (size_t)mm * ld;
    const int r = rowof[j];
    SensBest lo = sens_empty(), hi = sens_empty();
    if (r >= 0) {
        const double* Tr = T + (size_t)r * ld;
        for (int k = lane; k < W - 1; k += 32)
            if (rowof[k] < 0) sens_cost_candidate(lo, hi, z[k], Tr[k], k);
        lo = sens_warp_reduce<true>(lo);
        hi = sens_warp_reduce<false>(hi);
    }
    if (lane == 0) sens_write_variable(rep, m, n, j, sense, z[j], r >= 0, lo, hi, cj);
}

}  // namespace lpx
