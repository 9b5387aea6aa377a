// lpx_cta.cuh — one CTA per tableau: the whole simplex solve (build, all pivots, extraction)
// runs inside one thread block, with the tableau resident in shared memory (SMEM_T) or in
// global memory (L2/HBM) for shapes that do not fit.
//
// Replaces, per tableau, the reference loop R/Models/PrimalSimplex.cs:57-127 (primal) and
// R/Models/DualSimplex.cs:15-114 (dual), including
//   ExpandEqualitiesToInequalities  PrimalSimplex.cs:161-177   (row map built in-kernel)
//   BuildTableau                    PrimalSimplex.cs:179-203
//   PrepareForTableau               DualSimplex.cs:117-158
//   ForceDualFeasibility            DualSimplex.cs:195-228
// Branch & Bound nodes (R/Models/Branch&Bound.cs:233-248) are expressed as "base problem +
// extra unit rows" so that a batch of nodes of different depths runs in one launch.
#pragma once
#include "lpx_common.cuh"

namespace lpx {

// Warm start from a final tableau: the problem's working tableau is built from a SOURCE tableau by one edit of
// kind `kind`, then the kind's loop runs.
//   WARM_BOUND       a pooled-tree B&B node (lpx_pooled.cu, Mode B — not the reference's tree): the parent's FINAL
//                    tableau plus one bound row on variable `var` (x_var <= val for side 0, x_var >= val for side 1,
//                    written in the parent's non-basic variables) plus one slack column; Dual Simplex pivots follow.
//                    T / basis may point into ANOTHER GPU's node pool (peer memory over NVLink); out_T / out_basis
//                    are local.
//   LPX_REOPT_*      a re-optimization query (lpx_reopt.cu; the edits are defined in include/lpx.h): the payload is
//                    CtaBatch::reopt_payload + p * reopt_stride, the model's rel / m_in are CtaBatch::rel / m_in, and
//                    a source that is not LPX_OPTIMAL (base_status) is not built: the problem gets that status.
//                    RHS / ROW run the dual loop, COST / COL the primal loop.  out_T is the working storage of the
//                    global-memory build (unused in shared memory); results go to CtaBatch::basis / tableau.
enum { WARM_BOUND = 0 };  // the other kinds are LPX_REOPT_RHS .. LPX_REOPT_COL (1 .. 4)
struct WarmNode {
    const double* T;     // source (parent's / base's) compact tableau, rows x (n_src + rows)
    const int* basis;    // its basis, rows - 1 entries
    double* out_T;       // this problem's final tableau, compact (WARM_BOUND: (rows + 1) x (n + rows + 1))
    int* out_basis;      // WARM_BOUND: rows entries
    double val;
    int rows;            // of the SOURCE tableau (constraint rows + objective row)
    int var, side, kind;
    int base_status;     // status of the source; anything but LPX_OPTIMAL is passed through unsolved
};

struct CtaBatch {
    // base problems: instance k at A + k*strideA etc.; rel (nullable = all LE) is shared
    const double* A;
    const double* b;
    const double* c;
    const int* rel;
    long long strideA, strideB, strideC;
    int m_in, n, sense;
    int m_base;  // rows of the base problem after EQ expansion
    // optional per-problem node descriptors (nullable: problem p == instance p, no extra rows)
    const int* node_inst;
    const int* node_extra_off;
    const int* node_extra_cnt;
    const int* node_mode;
    const int* ex_var;
    const int* ex_rel;
    const double* ex_rhs;
    int mode;      // 0 primal, 1 dual (used when node_mode == nullptr)
    int max_iter;
    int max_rows, max_width;  // upper bounds over the batch (shared-memory carve, output strides)
    double* scratch;          // global tableaux when !SMEM_T and tableau == nullptr
    long long scratch_stride;
    // outputs, indexed by problem p = blockIdx.x
    int* status;
    int* n_pivots;
    int* silent;
    int* pivots;  // pivots_cap pairs per problem
    int pivots_cap;
    int* basis;  // basis_stride per problem
    int basis_stride;
    double* x;  // n per problem
    double* z;
    double* tableau;  // compact rows x width per problem (nullable)
    long long tableau_stride;
    double* history;  // history_cap compact tableaux per problem (nullable)
    long long history_stride;
    int history_cap;
    int* n_history;
    unsigned long long* total_pivots;
    // Branch & Bound node epilogue (nullable): per problem, bit 0 = IsFeasible(x), bit 1 = IsIntegral(x)
    // (R/Models/Branch&Bound.cs:268-294), and the branching variable (:198-213), -1 if none
    int* node_flags;
    int* node_branch;
    const WarmNode* warm;  // nullable: problem p is built from warm[p] instead of (A, b, c) and runs its kind's loop
    const double* reopt_payload;  // LPX_REOPT_* warm records: problem p's payload at + p * reopt_stride
    long long reopt_stride;
    long long* dbg;  // LPX_CTA_PROF=1: clock64() sums per phase of the LAST problem of the batch (8 slots)
};

// Shared-memory carve shared by host (sizing) and device.
struct CtaCarve {
    size_t prow, fcol, zc, red, rsrc, rsgn, basis, ctl, T, total;
};
__host__ __device__ inline CtaCarve cta_carve(int max_rows, int max_width, bool smem_T) {
    CtaCarve c;
    size_t off = 0;
    c.prow = off;
    off += (size_t)((max_width + 2) & ~1) * 8;  // even length: the update reads it two entries at a time
    c.fcol = off;
    off += (size_t)max_rows * 8;
    c.zc = off;  // the control warp's private copy of the objective row
    off += (size_t)max_width * 8;
    c.red = off;
    off += 34 * 16;
    c.rsrc = off;
    off += (size_t)max_rows * 4;
    c.rsgn = off;
    off += (size_t)max_rows * 4;
    c.basis = off;
    off += (size_t)max_rows * 4;
    c.ctl = off;
    off += 16 * 4;
    off = (off + 15) & ~(size_t)15;
    c.T = off;
    if (smem_T) off += (size_t)max_rows * ((max_width + 1) & ~1) * 8;  // rows padded to an even length (16-byte aligned)
    c.total = off;
    return c;
}

__device__ __forceinline__ double dneg(double v) {
    return __longlong_as_double(__double_as_longlong(v) ^ (long long)0x8000000000000000ULL);
}

// Gauss-Jordan pivot on (l, e): PrimalSimplex.Pivot (PrimalSimplex.cs:245-257).
// The factor column and the normalised pivot row are staged in shared memory first, so every
// element sees factor = T[i,e] as it was BEFORE row i changed and the ROUNDED quotient T[l,j]/piv.
// Rows with factor 0 are updated too (sign-of-zero parity, SURVEY.md §8 a11).
// PAIR (shared-memory tableau, even ld): every thread updates two adjacent columns with 16-byte loads
// and stores — half the memory instructions for the same bytes; the pad column of an odd width is
// carried along and never read back.
template <int THREADS, bool PAIR = false>
__device__ __forceinline__ void cta_pivot(double* T, int ld, int rows, int width, int l, int e, double* prow,
                                          double* fcol) {
    const int tid = threadIdx.x;
    const double piv = T[(size_t)l * ld + e];
    for (int j = tid; j < width; j += THREADS) prow[j] = ddiv_by_pivot(T[(size_t)l * ld + j], piv);
    for (int i = tid; i < rows; i += THREADS) fcol[i] = T[(size_t)i * ld + e];
    if (PAIR && tid == 0 && (width & 1)) prow[width] = 0.0;
    __syncthreads();
    if (PAIR) {
        const int pairs = (width + 1) >> 1;
        const int cw2 = (pairs + 31) & ~31;
        const int G = cw2 >= THREADS ? 1 : THREADS / cw2;
        for (int q0 = 0; q0 < pairs; q0 += THREADS) {  // one trip unless the tableau is wider than 2 * THREADS
            const int g = cw2 >= THREADS ? 0 : tid / cw2;
            const int q = cw2 >= THREADS ? q0 + tid : tid - g * cw2;
            if (g < G && q < pairs) {
                const double2 pj = *reinterpret_cast<const double2*>(prow + 2 * q);
                double* t = T + (size_t)g * ld + 2 * q;
                const size_t step = (size_t)G * ld;
#pragma unroll 4
                for (int i = g; i < rows; i += G, t += step) {
                    double2 cur = *reinterpret_cast<double2*>(t);
                    const double f = fcol[i];
                    if (i == l) {
                        cur = pj;
                    } else {
                        cur.x = __dsub_rn(cur.x, __dmul_rn(f, pj.x));
                        cur.y = __dsub_rn(cur.y, __dmul_rn(f, pj.y));
                    }
                    *reinterpret_cast<double2*>(t) = cur;
                }
            }
            if (cw2 < THREADS) break;
        }
        __syncthreads();
        return;
    }
    const int cw = (width + 31) & ~31;
    if (cw >= THREADS) {
        for (int j = tid; j < width; j += THREADS) {
            const double pj = prow[j];
            double* t = T + j;
#pragma unroll 4
            for (int i = 0; i < rows; i++, t += ld) {
                const double cur = *t;
                *t = (i == l) ? pj : __dsub_rn(cur, __dmul_rn(fcol[i], pj));
            }
        }
    } else {
        const int G = THREADS / cw;
        const int g = tid / cw, j = tid - g * cw;
        if (g < G && j < width) {
            const double pj = prow[j];
            double* t = T + (size_t)g * ld + j;
            const size_t step = (size_t)G * ld;
#pragma unroll 4
            for (int i = g; i < rows; i += G, t += step) {
                const double cur = *t;
                *t = (i == l) ? pj : __dsub_rn(cur, __dmul_rn(fcol[i], pj));
            }
        }
    }
    __syncthreads();
}

// Rows i = g, g + G, .. of one pair of adjacent columns: T[i,.] -= fcol[i] * pj, row l <- pj.  The loads of four
// rows are issued before the first store — the compiler cannot hoist a shared-memory load above the previous
// row's store on its own, and a one-row-at-a-time loop pays the load latency once per row.  UNIT: the column
// `which` (0 / 1, -1: neither) of the pair enters the update as the unit vector of row l (lpx_cta_cond.cuh).
template <bool UNIT>
__device__ __forceinline__ void cta_update_pair_column(double* t, size_t step, int g, int G, int rows, int l,
                                                       const double2 pj, const double* fcol, int which) {
    auto one = [&](double2 cur, double f, int i) -> double2 {
        if (UNIT) {
            if (which == 0) cur.x = i == l ? 1.0 : 0.0;
            if (which == 1) cur.y = i == l ? 1.0 : 0.0;
        }
        if (i == l) return pj;
        cur.x = __dsub_rn(cur.x, __dmul_rn(f, pj.x));
        cur.y = __dsub_rn(cur.y, __dmul_rn(f, pj.y));
        return cur;
    };
    int i = g;
    for (; i + 3 * G < rows; i += 4 * G, t += 4 * step) {
        double2 c[4];
        double f[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            c[u] = *reinterpret_cast<const double2*>(t + u * step);
            f[u] = fcol[i + u * G];
        }
#pragma unroll
        for (int u = 0; u < 4; u++) *reinterpret_cast<double2*>(t + u * step) = one(c[u], f[u], i + u * G);
    }
    for (; i < rows; i += G, t += step)
        *reinterpret_cast<double2*>(t) = one(*reinterpret_cast<const double2*>(t), fcol[i], i);
}

// The update alone, by the UT threads utid = 0 .. UT-1 (the control warp does not take part): prow and
// fcol are staged already.  Same arithmetic and element order as cta_pivot.
template <bool PAIR>
__device__ __forceinline__ void cta_update(double* T, int ld, int rows, int width, int l, const double* prow,
                                           const double* fcol, int utid, int UT) {
    if (PAIR) {
        const int pairs = (width + 1) >> 1;
        const int cw2 = (pairs + 31) & ~31;
        const int G = cw2 >= UT ? 1 : UT / cw2;
        for (int q0 = 0; q0 < pairs; q0 += UT) {  // one trip unless the tableau is wider than 2 * UT
            const int g = cw2 >= UT ? 0 : utid / cw2;
            const int q = cw2 >= UT ? q0 + utid : utid - g * cw2;
            if (g < G && q < pairs) {
                const double2 pj = *reinterpret_cast<const double2*>(prow + 2 * q);
                cta_update_pair_column<false>(T + (size_t)g * ld + 2 * q, (size_t)G * ld, g, G, rows, l, pj, fcol, -1);
            }
            if (cw2 < UT) break;
        }
        return;
    }
    const int cw = (width + 31) & ~31;
    if (cw >= UT) {
        for (int j = utid; j < width; j += UT) {
            const double pj = prow[j];
            double* t = T + j;
#pragma unroll 4
            for (int i = 0; i < rows; i++, t += ld) {
                const double cur = *t;
                *t = (i == l) ? pj : __dsub_rn(cur, __dmul_rn(fcol[i], pj));
            }
        }
    } else {
        const int G = UT / cw;
        const int g = utid / cw, j = utid - g * cw;
        if (g < G && j < width) {
            const double pj = prow[j];
            double* t = T + (size_t)g * ld + j;
            const size_t step = (size_t)G * ld;
#pragma unroll 4
            for (int i = g; i < rows; i += G, t += step) {
                const double cur = *t;
                *t = (i == l) ? pj : __dsub_rn(cur, __dmul_rn(fcol[i], pj));
            }
        }
    }
}

// ChooseEntering by ONE warp over v[0 .. n): most negative entry below thresh, lowest index on ties, -1 if
// none; NaN never wins (PrimalSimplex.cs:205-220).  All 32 lanes return the answer.
__device__ __forceinline__ int warp_argmin_below(const double* v, int n, double thresh) {
    const int lane = threadIdx.x & 31;
    unsigned long long kl = ~0ULL;
    int il = INT_MAX;
    for (int j = lane; j < n; j += 32) {
        const double z = v[j];
        if (z < thresh) {
            const unsigned long long k = dkey(z);
            if (k < kl) {
                kl = k;
                il = j;
            }
        }
    }
    const unsigned long long K = warp_min_u64(kl);
    const int idx = __reduce_min_sync(0xffffffffu, kl == K ? il : INT_MAX);
    return K == ~0ULL ? -1 : idx;
}

// Ratios of the min-ratio test, one division per thread (a double division is a ~40-instruction
// dependent chain: never let one warp do them one after another).  NaN marks "not eligible".
// Parked in prow, which is free until the pivot itself.
template <int THREADS>
__device__ __forceinline__ void cta_stage_ratios(const double* T, int ld, int m, int e, int rhs, double* prow) {
    for (int i = threadIdx.x; i < m; i += THREADS) {
        const double a = T[(size_t)i * ld + e];
        double r = __longlong_as_double(0x7ff8000000000000LL);
        if (a > LPX_EPS) r = ddiv_by_pivot(T[(size_t)i * ld + rhs], a);
        prow[i] = r;
    }
    __syncthreads();
}

template <int THREADS>
__device__ __forceinline__ void cta_copy_out(double* dst, const double* T, int ld, int rows, int width) {
    if (ld == width) {
        const int total = rows * width;
        for (int k = threadIdx.x; k < total; k += THREADS) dst[k] = T[k];
    } else {
        for (int i = 0; i < rows; i++)
            for (int j = threadIdx.x; j < width; j += THREADS) dst[(size_t)i * width + j] = T[(size_t)i * ld + j];
    }
}

// Row map of one tableau: tableau row k <- (source row, sign), after ExpandEqualitiesToInequalities
// (PrimalSimplex.cs:161-177) or PrepareForTableau (DualSimplex.cs:117-158), plus the reference's up-front
// checks (PrimalSimplex.cs:66-77).  ctl[0] = status, ctl[1] = number of tableau rows m.
// Without '=' rows the map is the identity and is filled by all threads (a B&B node at depth 120 has
// 180 rows; one thread walking them through global memory was 4-15 % of a node solve); with '=' rows
// one thread walks the rows in order.  Ends with the caller's barrier.
template <int THREADS>
__device__ __forceinline__ void cta_row_map(const CtaBatch& B, const double* bi, int nex, int exo, int mode, int* rsrc,
                                            int* rsgn, int* ctl) {
    const int tid = threadIdx.x;
    const int nr = B.m_in + nex;
    auto fetch = [&](int r, int& rl, double& bv, int& src) {
        if (r < B.m_in) {
            rl = B.rel ? B.rel[r] : 0;
            bv = bi[r];
            src = r;
        } else {
            rl = B.ex_rel[exo + r - B.m_in];
            bv = B.ex_rhs[exo + r - B.m_in];
            src = -1 - (r - B.m_in);
        }
    };
    int has_eq = 0;
    for (int r = tid; r < nr; r += THREADS) {
        int rl, src;
        double bv;
        fetch(r, rl, bv, src);
        if (rl == 2) has_eq = 1;
    }
    if (tid == 0) ctl[4] = INT_MAX;
    if (!__syncthreads_or(has_eq)) {
        for (int r = tid; r < nr; r += THREADS) {
            int rl, src;
            double bv;
            fetch(r, rl, bv, src);
            int flip = 0;
            if (mode == 0) {
                if (rl == 1 || bv < -1e-9) atomicMin(&ctl[4], r);  // the FIRST offending row decides the message
            } else {
                if (rl == 1) {
                    flip ^= 1;
                    bv = __dmul_rn(bv, -1.0);
                }
                if (bv < -LPX_EPS) flip ^= 1;
            }
            rsrc[r] = src;
            rsgn[r] = flip;
        }
        __syncthreads();
        if (tid == 0) {
            int st = LPX_RUNNING;
            if (mode == 0 && ctl[4] != INT_MAX) {
                int rl, src;
                double bv;
                fetch(ctl[4], rl, bv, src);
                st = rl == 1 ? LPX_S_GE_ROW : LPX_S_NEG_RHS;
            }
            ctl[0] = st;
            ctl[1] = nr;
        }
        return;
    }
    if (tid == 0) {
        int st = LPX_RUNNING, k = 0;
        for (int r = 0; r < nr; r++) {
            int rl, src;
            double bv;
            fetch(r, rl, bv, src);
            if (mode == 0) {
                if (st == LPX_RUNNING) {
                    if (rl == 1) st = LPX_S_GE_ROW;
                    else if (bv < -1e-9) st = LPX_S_NEG_RHS;
                }
                rsrc[k] = src;
                rsgn[k] = 0;
                k++;
                if (rl == 2) {
                    rsrc[k] = src;
                    rsgn[k] = 1;
                    k++;
                }
            } else {
                if (rl == 2) {
                    rsrc[k] = src;
                    rsgn[k] = 0;
                    k++;
                    rsrc[k] = src;
                    rsgn[k] = 1;
                    k++;
                } else {
                    int flip = 0;
                    if (rl == 1) {
                        flip ^= 1;
                        bv = __dmul_rn(bv, -1.0);
                    }
                    if (bv < -LPX_EPS) flip ^= 1;
                    rsrc[k] = src;
                    rsgn[k] = flip;
                    k++;
                }
            }
        }
        ctl[0] = st;
        ctl[1] = k;  // == m
    }
}

// A problem the reference rejects before building a tableau (PrimalSimplex.cs:66-77) has no result: its
// output slots are zero-filled, so callers never see leftovers of an earlier solve in reused buffers.
template <int THREADS>
__device__ __forceinline__ void cta_zero_outputs(const CtaBatch& B, int p, int m, int n, int rows, int width,
                                                 int rank = 0, int nranks = 1) {
    const int tid = threadIdx.x + rank * THREADS, step = THREADS * nranks;
    if (B.basis)
        for (int i = tid; i < m; i += step) B.basis[(size_t)p * B.basis_stride + i] = 0;
    if (B.x)
        for (int j = tid; j < n; j += step) B.x[(size_t)p * n + j] = 0.0;
    if (B.z && tid == 0) B.z[p] = 0.0;
    if (B.tableau) {
        double* To = B.tableau + (size_t)p * B.tableau_stride;
        const int total = rows * width;
        for (int k = tid; k < total; k += step) To[k] = 0.0;
    }
}

// The part of SolveNode that only looks at the node's own solution (R/Models/Branch&Bound.cs:175-213), on the
// device so that the host commit merely orders records:
//   IsFeasible (:276-294)  every row sum a . x in index order (one thread per row, separate multiply and add),
//                          1e-6 slack per relation; the node's unit rows the same way; x >= -1e-6
//   IsIntegral (:268-274)  |x - Math.Round(x)| <= 1e-6 (ties to even) for every variable
//   branching variable (:198-213)  fractional part in (1e-6, 1 - 1e-6) closest to 0.5, lowest index on ties
// x = the solution in global memory (complete and visible to this block); xs = n doubles of shared scratch.
template <int THREADS>
__device__ __forceinline__ void cta_node_epilogue(const CtaBatch& B, int p, int inst, int nex, int exo, const double* x,
                                                  double* xs, ArgMin* red) {
    const int tid = threadIdx.x;
    const int n = B.n;
    const double BB = 1e-6;  // BranchAndBound.EPS
    for (int j = tid; j < n; j += THREADS) xs[j] = x[j];
    __syncthreads();
    int bad = 0;  // infeasible
    const double* Ai = B.A + (size_t)inst * B.strideA;
    const double* bi = B.b + (size_t)inst * B.strideB;
    for (int r = tid; r < B.m_in + nex; r += THREADS) {
        double sum = 0.0, bv;
        int rl;
        if (r < B.m_in) {
            const double* a = Ai + (size_t)r * n;
            for (int i = 0; i < n; i++) sum = __dadd_rn(sum, __dmul_rn(a[i], xs[i]));
            rl = B.rel ? B.rel[r] : 0;
            bv = bi[r];
        } else {
            const int var = B.ex_var[exo + r - B.m_in];
            for (int i = 0; i < n; i++) sum = __dadd_rn(sum, __dmul_rn(i == var ? 1.0 : 0.0, xs[i]));
            rl = B.ex_rel[exo + r - B.m_in];
            bv = B.ex_rhs[exo + r - B.m_in];
        }
        if (rl == 0 && sum > __dadd_rn(bv, BB)) bad = 1;
        if (rl == 1 && sum < __dsub_rn(bv, BB)) bad = 1;
        if (rl == 2 && fabs(__dsub_rn(sum, bv)) > BB) bad = 1;
    }
    int nonint = 0;
    unsigned long long kl = ~0ULL;  // key of |frac - 0.5|, then the index
    int il = INT_MAX;
    for (int i = tid; i < n; i += THREADS) {
        const double v = xs[i];
        if (v < -BB) bad = 1;
        if (fabs(__dsub_rn(v, rint(v))) > BB) nonint = 1;
        const double frac = __dsub_rn(v, floor(v));
        if (frac > BB && __dsub_rn(1.0, frac) > BB) {
            const unsigned long long k = dkey(fabs(__dsub_rn(frac, 0.5)));
            if (k < kl) {
                kl = k;
                il = i;
            }
        }
    }
    const int any_bad = __syncthreads_or(bad), any_nonint = __syncthreads_or(nonint);
    // block argmin of (distance key, index): per warp, then over the warp partials
    const int lane = tid & 31, warp = tid >> 5;
    const unsigned long long K = warp_min_u64(kl);
    const int iw = __reduce_min_sync(0xffffffffu, kl == K ? il : INT_MAX);
    if (lane == 0) {
        red[warp].v = __longlong_as_double((long long)K);
        red[warp].i = iw;
    }
    __syncthreads();
    if (warp == 0) {
        unsigned long long k2 = ~0ULL;
        int i2 = INT_MAX;
        if (lane < THREADS / 32) {
            k2 = (unsigned long long)__double_as_longlong(red[lane].v);
            i2 = red[lane].i;
        }
        const unsigned long long K2 = warp_min_u64(k2);
        const int idx = __reduce_min_sync(0xffffffffu, k2 == K2 ? i2 : INT_MAX);
        if (lane == 0) {
            B.node_flags[p] = (any_bad ? 0 : 1) | (any_nonint ? 0 : 2);
            B.node_branch[p] = K2 == ~0ULL ? -1 : idx;
        }
    }
    __syncthreads();
}

// The working tableau of a re-optimization query (include/lpx.h, "Re-optimization"): rows x width at T (leading
// dimension ld), built straight from the source tableau Ts (rows_s rows) with the edit of `kind`, in the definition's
// order of terms; sbasis receives the query's basis.  n counts the query's decision variables (COL: one more than the
// source).  rowof: n ints of shared scratch.  Ends with a block barrier.  Not inlined: the kernel's pivot loops keep
// the register allocation they have without it.
template <int THREADS>
__device__ __noinline__ void cta_reopt_build(int kind, const double* Ts, const int* bs, int rows_s, int n, int m_in,
                                             const int* rel, int sense, const double* pay, double* T, int ld, int rows,
                                             int width, int* sbasis, int* rowof) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = THREADS / 32;
    const int ms = rows_s - 1;                                // source constraint rows
    const int ns = kind == LPX_REOPT_COL ? n - 1 : n;         // source decision variables
    const int ws = ns + rows_s, rhs_s = ws - 1;               // source width and RHS column
    auto src = [&](int i, int j) { return Ts[(size_t)i * ws + j]; };
    // v + sum over constraints i ascending with d_i != 0 of d_i * T[r][s1] (EQ: - d_i * T[r][s2]), term by term
    auto slack_terms = [&](double v, int r, const double* d) {
        int i1 = 0;
        for (int i = 0; i < m_in; i++) {
            const bool eq = rel && rel[i] == 2;
            const double di = d[i];
            if (di != 0.0) {
                v = __dadd_rn(v, __dmul_rn(di, src(r, ns + i1)));
                if (eq) v = __dsub_rn(v, __dmul_rn(di, src(r, ns + i1 + 1)));
            }
            i1 += eq ? 2 : 1;
        }
        return v;
    };
    for (int i = tid; i < ms; i += THREADS) {
        const int b = bs[i];
        sbasis[i] = (kind == LPX_REOPT_COL && b >= ns) ? b + 1 : b;
    }
    if (kind == LPX_REOPT_ROW && tid == 0) sbasis[ms] = rhs_s;  // the new slack is basic in the new row
    if (kind == LPX_REOPT_COST)
        for (int j = tid; j < n; j += THREADS) rowof[j] = -1;
    __syncthreads();
    if (kind == LPX_REOPT_COST)
        for (int i = tid; i < ms; i += THREADS)
            if (sbasis[i] < n) rowof[sbasis[i]] = i;
    __syncthreads();
    const bool ge = kind == LPX_REOPT_ROW && pay[n] == 1.0;
    for (int i = warp; i < rows; i += NW) {
        double* Ti = T + (size_t)i * ld;
        for (int j = lane; j < width; j += 32) {
            double v;
            if (kind == LPX_REOPT_RHS) {
                v = j < rhs_s ? src(i, j) : slack_terms(src(i, rhs_s), i, pay);
            } else if (kind == LPX_REOPT_COST) {
                v = src(i, j);
                if (i == ms)
                    for (int q = 0; q < n; q++) {
                        const double d = pay[q];
                        if (d == 0.0) continue;
                        const double delta = sense == 1 ? dneg(d) : d;
                        if (rowof[q] >= 0) v = __dadd_rn(v, __dmul_rn(delta, src(rowof[q], j)));
                        if (j == q) v = __dsub_rn(v, delta);
                    }
            } else if (kind == LPX_REOPT_ROW) {
                if (i != ms) {  // an old row (i > ms: the objective row): the old RHS position becomes the new slack
                    const int si = i < ms ? i : ms;
                    v = j < rhs_s ? src(si, j) : (j == rhs_s ? 0.0 : src(si, rhs_s));
                } else if (j == rhs_s) {
                    v = 1.0;
                } else {  // the raw row (GE: every entry negated, zeros included), then the basic columns eliminated
                    const int k = j < rhs_s ? j : rhs_s;
                    v = k < n ? pay[k] : (k == rhs_s ? pay[n + 1] : 0.0);
                    if (ge) v = dneg(v);
                    for (int r = 0; r < ms; r++) {
                        const int b = sbasis[r];
                        if (b >= n || pay[b] == 0.0) continue;
                        v = __dsub_rn(v, __dmul_rn(ge ? dneg(pay[b]) : pay[b], src(r, k)));
                    }
                }
            } else {  // LPX_REOPT_COL: the new column sits at ns, the old columns from ns on move right by one
                if (j != ns) {
                    v = src(i, j < ns ? j : j - 1);
                } else {
                    const double cn = sense == 1 ? dneg(pay[m_in]) : pay[m_in];
                    v = slack_terms(i == ms ? dneg(cn) : 0.0, i, pay);
                }
            }
            Ti[j] = v;
        }
    }
    if (ld > width)
        for (int i = tid; i < rows; i += THREADS) T[(size_t)i * ld + width] = 0.0;  // pad column
    __syncthreads();
}

template <int THREADS, bool SMEM_T>
__global__ void __launch_bounds__(THREADS) cta_simplex_kernel(const CtaBatch B) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = THREADS / 32;
    const int p = blockIdx.x;

    const int inst = B.node_inst ? B.node_inst[p] : p;
    const int nex = B.node_extra_cnt ? B.node_extra_cnt[p] : 0;
    const int exo = B.node_extra_off ? B.node_extra_off[p] : 0;
    const bool warm = B.warm != nullptr;
    const int kind = warm ? B.warm[p].kind : WARM_BOUND;
    const int mode = warm ? (kind == LPX_REOPT_COST || kind == LPX_REOPT_COL ? 0 : 1)
                          : (B.node_mode ? B.node_mode[p] : B.mode);
    const int n = B.n;
    // a bound row or an added row gives one constraint row more than the source
    const int m = warm ? B.warm[p].rows - (kind == WARM_BOUND || kind == LPX_REOPT_ROW ? 0 : 1) : B.m_base + nex;
    const int rows = m + 1, width = n + m + 1, ld = SMEM_T ? ((width + 1) & ~1) : width;
    const int rhs = width - 1;

    const CtaCarve cv = cta_carve(B.max_rows, B.max_width, SMEM_T);
    double* prow = reinterpret_cast<double*>(smem_raw + cv.prow);
    double* fcol = reinterpret_cast<double*>(smem_raw + cv.fcol);
    ArgMin* red = reinterpret_cast<ArgMin*>(smem_raw + cv.red);
    int* rsrc = reinterpret_cast<int*>(smem_raw + cv.rsrc);
    int* rsgn = reinterpret_cast<int*>(smem_raw + cv.rsgn);
    int* sbasis = reinterpret_cast<int*>(smem_raw + cv.basis);
    int* ctl = reinterpret_cast<int*>(smem_raw + cv.ctl);
    double* T;
    if (SMEM_T) T = reinterpret_cast<double*>(smem_raw + cv.T);
    else if (warm) T = B.warm[p].out_T;  // the node's pool slot doubles as working storage (compact: ld == width)
    else T = B.tableau ? B.tableau + (size_t)p * B.tableau_stride : B.scratch + (size_t)p * B.scratch_stride;

    const double* Ai = B.A + (size_t)inst * B.strideA;
    const double* bi = B.b + (size_t)inst * B.strideB;
    const double* ci = B.c + (size_t)inst * B.strideC;

    int status = LPX_RUNNING;
    if (!warm) {
        // ---- row map + the reference's up-front checks (PrimalSimplex.cs:66-77) -------------------
        cta_row_map<THREADS>(B, bi, nex, exo, mode, rsrc, rsgn, ctl);
        __syncthreads();
        status = ctl[0];
    } else if (B.warm[p].base_status != LPX_OPTIMAL) {
        status = B.warm[p].base_status;
    }

    int n_piv = 0, n_silent = 0, n_hist = 0;
    int* plog = B.pivots ? B.pivots + (size_t)p * B.pivots_cap * 2 : nullptr;
    double* hist = B.history ? B.history + (size_t)p * B.history_stride : nullptr;
    const size_t tsize = (size_t)rows * width;

    if (status == LPX_RUNNING && warm && kind == WARM_BOUND) {
        // ---- parent's final tableau + bound row + slack column (lpx_pooled.cu; oracle/orc_pooled.cpp) -----
        const WarmNode wn = B.warm[p];
        const int mp = wn.rows - 1, wp = n + wn.rows, rhs_p = wp - 1;  // parent: constraint rows, width, RHS column
        if (tid == 0) ctl[5] = -1;
        __syncthreads();
        for (int i = tid; i < mp; i += THREADS) {
            const int bv = wn.basis[i];
            sbasis[i] = bv;
            if (bv == wn.var) ctl[5] = i;  // the row in which the branching variable is basic (exactly one)
        }
        if (tid == 0) sbasis[mp] = rhs_p;   // the new slack is basic in the new row
        __syncthreads();
        const int r = ctl[5];
        const double* Tr = wn.T + (size_t)r * wp;
        for (int i = warp; i < rows; i += NW) {
            double* Ti = T + (size_t)i * ld;
            // child row i <- parent row (i < mp: same row; i == mp: the bound row, built from parent row r;
            // i == mp + 1: the objective row)
            const double* Ts = i < mp ? wn.T + (size_t)i * wp : (i == mp ? Tr : wn.T + (size_t)mp * wp);
            for (int j = lane; j < width; j += 32) {
                double v;
                if (i != mp) {
                    v = j < rhs_p ? Ts[j] : (j == rhs_p ? 0.0 : Ts[rhs_p]);
                } else if (j < rhs_p) {
                    const double unit = j == wn.var ? 1.0 : 0.0;
                    v = wn.side == 0 ? __dsub_rn(unit, Ts[j]) : __dsub_rn(Ts[j], unit);
                } else if (j == rhs_p) {
                    v = 1.0;
                } else {
                    v = wn.side == 0 ? __dsub_rn(wn.val, Ts[rhs_p]) : __dsub_rn(Ts[rhs_p], wn.val);
                }
                Ti[j] = v;
            }
        }
        if (ld > width)
            for (int i = tid; i < rows; i += THREADS) T[(size_t)i * ld + width] = 0.0;  // pad column
        __syncthreads();
    } else if (status == LPX_RUNNING && warm) {
        // ---- a re-optimization query: the base's final tableau with one edit (lpx_reopt.cu) ---------------
        const WarmNode& wn = B.warm[p];
        cta_reopt_build<THREADS>(kind, wn.T, wn.basis, wn.rows, n, B.m_in, B.rel, B.sense,
                                 B.reopt_payload + (size_t)p * B.reopt_stride, T, ld, rows, width, sbasis,
                                 reinterpret_cast<int*>(prow));
    } else if (status == LPX_RUNNING) {
        // ---- BuildTableau -------------------------------------------------------------------
        for (int i = warp; i < rows; i += NW) {
            double* Ti = T + (size_t)i * ld;
            if (i < m) {
                const int src = rsrc[i];
                const bool flip = rsgn[i] != 0;
                const int xv = src < 0 ? B.ex_var[exo + (-1 - src)] : -1;
                const double* Ar = src >= 0 ? Ai + (size_t)src * n : nullptr;
                for (int j = lane; j < width; j += 32) {
                    double v;
                    if (j < n) {
                        v = Ar ? Ar[j] : (j == xv ? 1.0 : 0.0);
                        v = neg_if(v, flip);
                    } else if (j == rhs) {
                        v = src >= 0 ? bi[src] : B.ex_rhs[exo + (-1 - src)];
                        v = neg_if(v, flip);
                    } else {
                        v = (j == n + i) ? 1.0 : 0.0;
                    }
                    Ti[j] = v;
                }
            } else {
                for (int j = lane; j < width; j += 32) {
                    double v = 0.0;
                    if (j < n) {
                        double cj = ci[j];
                        if (B.sense == 1) cj = dneg(cj);  // Min -> Max (PrimalSimplex.cs:62-63)
                        v = dneg(cj);                     // T[m,j] = -C[j]
                    }
                    Ti[j] = v;
                }
            }
        }
        if (ld > width)
            for (int i = tid; i < rows; i += THREADS) T[(size_t)i * ld + width] = 0.0;  // pad column
        for (int i = tid; i < m; i += THREADS) sbasis[i] = n + i;
        __syncthreads();
    }
    if (status == LPX_RUNNING) {
        const double* zrow = T + (size_t)m * ld;
        double* zc = reinterpret_cast<double*>(smem_raw + cv.zc);
        long long pc[4] = {0, 0, 0, 0}, c0 = 0;
        const bool prof = B.dbg != nullptr && p == (int)gridDim.x - 1;
#define CTA_TICK(slot)                       \
    if (prof) {                              \
        const long long c1 = clock64();      \
        pc[slot] += c1 - c0;                 \
        c0 = c1;                             \
    }

        // ---- primal pivots (PrimalSimplex.cs:92-124; ForceDualFeasibility, DualSimplex.cs:195-228) -------
        // Four block barriers per pivot.  Warp 0 is the CONTROL warp: it keeps a private copy of the
        // objective row (zc, updated with the very operations the tableau's own row sees, so bit-identical)
        // and, while the other warps stream the rank-1 update through shared memory, it updates that copy
        // and picks the NEXT entering column — ChooseEntering never costs the block a phase.  After the
        // update: ratios, one division per thread | the control warp's margin scan | pivot row / factor
        // column staged | update.
        // Returns why it stopped: 0 = `limit` pivots done, 1 = no entering column, 2 = no leaving row.
        auto primal_steps = [&](double margin, int limit, bool silent) -> int {
            if (warp == 0) {
                for (int j = lane; j < width; j += 32) zc[j] = zrow[j];
                __syncwarp();
                const int e0 = warp_argmin_below(zc, width - 1, -LPX_EPS);
                if (lane == 0) ctl[3] = e0;
            }
            __syncthreads();
            int steps = 0;
            while (true) {
                if (steps >= limit) return 0;
                if (prof) c0 = clock64();
                const int e = ctl[3];
                if (e < 0) return 1;
                cta_stage_ratios<THREADS>(T, ld, m, e, rhs, prow);
                CTA_TICK(0)
                if (warp == 0) {
                    const int lv = warp_margin_scan_staged(m, margin, prow);
                    if (lane == 0) ctl[2] = lv;
                }
                __syncthreads();
                CTA_TICK(1)
                const int l = ctl[2];
                if (l < 0) return 2;
                {   // the normalised pivot row and the factor column: every element sees T[i,e] as it was before
                    // row i changed and the ROUNDED quotient T[l,j] / piv (PrimalSimplex.cs:245-257)
                    const double piv = T[(size_t)l * ld + e];
                    for (int j = tid; j < width; j += THREADS) prow[j] = ddiv_by_pivot(T[(size_t)l * ld + j], piv);
                    for (int i = tid; i < rows; i += THREADS) fcol[i] = T[(size_t)i * ld + e];
                    if (SMEM_T && tid == 0 && (width & 1)) prow[width] = 0.0;
                }
                __syncthreads();
                CTA_TICK(2)
                if (warp == 0) {
                    const double fz = fcol[m];
                    for (int j = lane; j < width; j += 32) zc[j] = __dsub_rn(zc[j], __dmul_rn(fz, prow[j]));
                    __syncwarp();
                    const int en = warp_argmin_below(zc, width - 1, -LPX_EPS);
                    if (lane == 0) {
                        ctl[3] = en;
                        sbasis[l] = e;
                        if (plog && n_piv < B.pivots_cap) {
                            plog[2 * n_piv] = e;
                            plog[2 * n_piv + 1] = l;
                        }
                    }
                } else {
                    cta_update<SMEM_T>(T, ld, rows, width, l, prow, fcol, tid - 32, THREADS - 32);
                }
                __syncthreads();
                CTA_TICK(3)
                n_piv++;
                if (silent) n_silent++;
                else if (hist && n_hist < B.history_cap) {
                    cta_copy_out<THREADS>(hist + (size_t)n_hist * tsize, T, ld, rows, width);
                    n_hist++;
                }
                steps++;
            }
        };

        // <= 100 silent pivots, ratio margin 1e-12 (a warm node starts from an optimal, hence dual feasible, tableau)
        if (mode == 1 && !warm) primal_steps(LPX_MARGIN_DUAL, 100, true);

        if (hist && n_hist < B.history_cap) {
            cta_copy_out<THREADS>(hist + (size_t)n_hist * tsize, T, ld, rows, width);
            n_hist++;
        }

        if (mode == 0) {
            // "if (iter > MaxIterations) throw" comes before the optimality test (PrimalSimplex.cs:95-96)
            const int why = primal_steps(LPX_MARGIN_PRIMAL, B.max_iter, false);
            status = why == 0 ? LPX_S_ITER_LIMIT : (why == 1 ? LPX_OPTIMAL : LPX_UNBOUNDED);
        }
        int iter = 1;
        while (mode == 1) {
            if (iter > LPX_DUAL_MAX_ITER) {
                status = LPX_S_ITER_LIMIT;
                break;
            }
            int e, l;
            // dual: leaving row = most negative RHS below -1e-9 (DualSimplex.cs:45-55)
            l = block_argmin_below_strided<THREADS>(T + rhs, (size_t)ld, m, -LPX_EPS, red);
            if (l < 0) {
                status = LPX_OPTIMAL;
                break;
            }
            // entering column: min z_j / (-a) over a < -1e-9, margin 1e-12 (DualSimplex.cs:76-91)
            {
                const double* lrow = T + (size_t)l * ld;
                for (int j = tid; j < width - 1; j += THREADS) {
                    const double a = lrow[j];
                    double r = __longlong_as_double(0x7ff8000000000000LL);
                    if (a < -LPX_EPS) r = ddiv_by_pivot(zrow[j], dneg(a));
                    prow[j] = r;
                }
                __syncthreads();
            }
            if (warp == 0) {
                const int ev = warp_margin_scan_cert(width - 1, LPX_MARGIN_DUAL, [&](int j, double& r) {
                    r = prow[j];
                    return r == r;
                });
                if (lane == 0) ctl[2] = ev;
            }
            __syncthreads();
            e = ctl[2];
            if (e < 0) {
                status = LPX_INFEASIBLE;
                break;
            }
            cta_pivot<THREADS, SMEM_T>(T, ld, rows, width, l, e, prow, fcol);
            if (tid == 0) {
                sbasis[l] = e;
                if (plog && n_piv < B.pivots_cap) {
                    plog[2 * n_piv] = e;
                    plog[2 * n_piv + 1] = l;
                }
            }
            n_piv++;
            if (hist && n_hist < B.history_cap) {
                cta_copy_out<THREADS>(hist + (size_t)n_hist * tsize, T, ld, rows, width);
                n_hist++;
            }
            iter++;
        }
#undef CTA_TICK
        if (prof && tid == 0) {
            for (int t = 0; t < 4; t++) B.dbg[t] = pc[t];
            B.dbg[4] = n_piv;
            B.dbg[5] = rows;
            B.dbg[6] = width;
        }
        __syncthreads();

        // ---- FinalizeReport's numeric part (PrimalSimplex.cs:132-138) -------------------------
        if (B.basis)
            for (int i = tid; i < m; i += THREADS) B.basis[(size_t)p * B.basis_stride + i] = sbasis[i];
        if (warm && kind == WARM_BOUND) {  // the final tableau and basis stay in the node pool for the node's own children
            for (int i = tid; i < m; i += THREADS) B.warm[p].out_basis[i] = sbasis[i];
            if (SMEM_T) cta_copy_out<THREADS>(B.warm[p].out_T, T, ld, rows, width);
        }
        if (B.x) {
            double* xo = B.x + (size_t)p * n;
            for (int j = tid; j < n; j += THREADS) xo[j] = 0.0;
            __syncthreads();
            for (int i = tid; i < m; i += THREADS)  // distinct rows, distinct basic variables
                if (sbasis[i] < n) xo[sbasis[i]] = T[(size_t)i * ld + rhs];
        }
        if (B.z && tid == 0) B.z[p] = T[(size_t)m * ld + rhs];
        if (B.tableau && (SMEM_T || T != B.tableau + (size_t)p * B.tableau_stride))
            cta_copy_out<THREADS>(B.tableau + (size_t)p * B.tableau_stride, T, ld, rows, width);
        if (B.node_flags && B.x && (mode == 0 || warm)) {  // prow (width > n doubles) is free now
            __syncthreads();
            cta_node_epilogue<THREADS>(B, p, inst, nex, exo, B.x + (size_t)p * n, prow, red);
        }
    } else {
        cta_zero_outputs<THREADS>(B, p, m, n, rows, width);
    }

    if (tid == 0) {
        B.status[p] = status;
        if (B.n_pivots) B.n_pivots[p] = n_piv;
        if (B.silent) B.silent[p] = n_silent;
        if (B.n_history) B.n_history[p] = n_hist;
        if (B.total_pivots && n_piv) atomicAdd(B.total_pivots, (unsigned long long)n_piv);
    }
}

// Host-side launcher (lpx_cta.cu): picks SMEM_T from the carve size, sets the shared-memory
// attribute, launches `count` CTAs on `stream`.  scratch must be provided when the tableau does
// not fit in shared memory and B.tableau is null.
int cta_launch(const CtaBatch& B, int count, int kernel_pref, int threads_pref, cudaStream_t stream, bool* used_smem);
bool cta_fits_smem(int max_rows, int max_width);
// condensed-tableau node kernel (lpx_cta_cond.cuh)
bool cta_condensed_fits(int max_rows, int n);
int cta_condensed_ctas_per_sm(int rows, int n);  // by shared memory
int cta_condensed_launch(const CtaBatch& B, int count, cudaStream_t stream);
int cta_cluster_size_for(int max_rows, int max_width);

}  // namespace lpx
