// lpx_stream_param.cuh — parametric analysis of an optimal streaming session (lpx_session_parametric).  The working
// tableau (the base's plus the direction column g at index W, or the direction row h at row m' + 1) is built in HBM
// straight from the base's current buffer; then one CTA decides up to K breakpoints on the tableau as the last pass
// left it, and the unchanged blocked pass (stream_update_block_kernel / stream_update_block_tma_kernel) applies their
// pivots in one HBM pass.  The rule of lpx_stream_block.cuh,
//       v <- (row == l_s) ? p_s[col] : v - f_s[row] * p_s[col]          for the pending pivots s in order,
// brings every value a decision reads up to date, so K decisions and one pass give the bits of K single passes, and
// the whole analysis the bits of oracle/orc_param.cpp (the definition is in include/lpx.h, "Parametric analysis").
//
// Included by lpx_stream.cu after lpx_stream_reopt.cuh (StreamParams / StreamCtl, block_min_int, LPX_BLOCK_KMAX,
// ReoptTerm).
#include "lpx_sens.cuh"

namespace lpx {

// The look-ahead's vectors.  Each lives in dynamic shared memory when it fits next to the ones placed before it,
// otherwise in global memory (L2): z and h together with the compact columns do not fit one CTA at C3's shape.
//   PV_Z     z-row, ld
//   PV_HG    COST: h, ld;  RHS: compact g (column W), colstride
//   PV_RHS   compact RHS (column W - 1; row m' is z0, and for COST row m' + 1 is dz), colstride
//   PV_COL   the entering column brought up to date, colstride
//   PV_RATIO RHS: entering-column ratios, ld;  COST: leaving-row ratios, colstride
enum { PV_Z = 0, PV_HG, PV_RHS, PV_COL, PV_RATIO, PV_N };

// The analysis' progress, handed from look-ahead to look-ahead.  end is the device status word: -1 while the
// analysis runs; once it holds an LPX_PARAM_* every later look-ahead (and so its pass) is a no-op.
struct ParamState {
    double th_lo;  // theta_lo of the segment being decided
    int k;         // segments recorded
    int end;
};

struct ParamLa {
    double* gvec[PV_N];  // global-memory home of each vector
    int soff[PV_N];      // its offset in dynamic shared memory (doubles), -1: global memory
    int* isb;            // COST: 1 for a basic column, 0 otherwise (W entries), kept up to date by the look-ahead
    ParamState* st;
    double* seg;  // seg_cap records of 4 + 2n doubles, zeroed before the first look-ahead (nullable)
    int* spv;     // seg_cap (leaving row, entering column) pairs, -1 before the first look-ahead (nullable)
    int seg_cap, n;
    double theta_max;
};

// The working tableau from the base tableau Tb (mb + 1 rows, leading dimension ldb, width W = Q.width): the base's
// entries, pad columns zero, and for COST h in row mb + 1 from a zero row with the COST query's terms in the
// definition's order (h[k] += a * Tb[idx][k] when idx >= 0, then h[aux] -= a).  RHS: column W is left at zero for
// stream_param_g_kernel.  grid = (column strips of 256, row groups).
__global__ void __launch_bounds__(256) stream_param_build_kernel(StreamParams Q, const double* __restrict__ Tb, int ldb,
                                                                 int mb, int cost, const ReoptTerm* __restrict__ t,
                                                                 int nt) {
    const int j = blockIdx.x * 256 + threadIdx.x;
    if (j >= Q.ld) return;
    const int W = Q.width;
    for (int i = blockIdx.y; i < Q.rows; i += gridDim.y) {
        double v = 0.0;
        if (!cost) {
            if (j < W) v = Tb[(size_t)i * ldb + j];
        } else if (j < W) {
            if (i <= mb) {
                v = Tb[(size_t)i * ldb + j];
            } else {
                for (int q = 0; q < nt; q++) {
                    if (t[q].idx >= 0) v = __dadd_rn(v, __dmul_rn(t[q].a, Tb[(size_t)t[q].idx * ldb + j]));
                    if (j == t[q].aux) v = __dsub_rn(v, t[q].a);
                }
            }
        }
        Q.T[(size_t)i * Q.ld + j] = v;
    }
}

// RHS: g in column W of the working tableau, one thread per row r: from +0.0, the RHS query's terms in the
// definition's order (g_r (+ or -)= a * Tb[r][idx]).  The entries of a batch of terms are loaded together, then added
// in order.  (Written by the build kernel, the column's one thread per row group would walk its rows one after the
// other: 50 ms for a dense direction at C3's shape.)
#define LPX_PARAM_G_THREADS 64
__global__ void __launch_bounds__(LPX_PARAM_G_THREADS) stream_param_g_kernel(StreamParams Q, const double* __restrict__ Tb,
                                                                             int ldb, const ReoptTerm* __restrict__ t,
                                                                             int nt) {
    const int i = blockIdx.x * LPX_PARAM_G_THREADS + threadIdx.x;
    if (i >= Q.rows) return;
    const double* Ti = Tb + (size_t)i * ldb;
    double v = 0.0;
    for (int q0 = 0; q0 < nt; q0 += 8) {
        double x[8];
#pragma unroll
        for (int u = 0; u < 8; u++) x[u] = q0 + u < nt ? Ti[t[q0 + u].idx] : 0.0;
#pragma unroll
        for (int u = 0; u < 8; u++)
            if (q0 + u < nt) {
                const double d = __dmul_rn(t[q0 + u].a, x[u]);
                v = t[q0 + u].aux ? __dsub_rn(v, d) : __dadd_rn(v, d);
            }
    }
    Q.T[(size_t)i * Q.ld + Q.width] = v;
}

// One CTA, 1024 threads: up to P.kblock breakpoints on the tableau as the last pass left it.  For each:
//   theta_cand with the sensitivity report's tie rule (RHS: min -(beta_r / g_r) over constraint rows with g_r < -EPS;
//   COST: min -(z_k / h_k) over non-basic k < W - 1 with h_k < -EPS); theta_end = max(theta_cand, theta_lo); REACHED
//   at theta_max, SEG_LIMIT at the last record, else the pivot search (RHS: that row leaves, the entering column by
//   the Dual Simplex rule with the 1e-12 replay over columns < W - 1, none: INFEASIBLE; COST: that column enters, the
//   leaving row by the Primal Simplex rule with the 1e-9 replay over rows < m', none: UNBOUNDED); the segment record
//   and its pivot pair from the values before the pivot; then the pivot is handed to the pass (Fbuf / Pbuf / Lbuf,
//   block_cnt, P.basis) and the compact vectors advance with the rule above.
template <bool COST>
__global__ void __launch_bounds__(1024) stream_param_lookahead_kernel(StreamParams P, ParamLa A) {
    extern __shared__ double sm_pl[];
    __shared__ SensBest sred[32];
    __shared__ int ired[34];
    __shared__ int s_L[LPX_BLOCK_KMAX];
    __shared__ double s_pe[LPX_BLOCK_KMAX];  // p_s[e]   for the column being brought up to date
    __shared__ double s_fl[LPX_BLOCK_KMAX];  // f_s[l]   for the row being brought up to date
    constexpr int TH = 1024;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ld = P.ld, cs = P.colstride, m = P.m, rows = P.rows, nc = P.width - 1, n = A.n;
    double* vec[PV_N];
#pragma unroll
    for (int v = 0; v < PV_N; v++) vec[v] = A.soff[v] >= 0 ? sm_pl + A.soff[v] : A.gvec[v];
    double* z = vec[PV_Z];
    double* hg = vec[PV_HG];
    double* rhs = vec[PV_RHS];
    double* col = vec[PV_COL];
    double* ratio = vec[PV_RATIO];
    StreamCtl* ctl = P.ctl;
    ParamState* S = A.st;
    const int end0 = S->end;
    const int done = ctl->pivots;
    double th_lo = S->th_lo;
    int k = S->k;
    __syncthreads();  // every thread has read the state before thread 0 rewrites it
    if (tid == 0) ctl->block_cnt = 0;
    if (end0 >= 0) return;

    const double* Tz = P.T + (size_t)m * ld;
    for (int j = tid; j < ld; j += TH) {
        z[j] = Tz[j];
        if (COST) hg[j] = Tz[ld + j];
    }
    for (int i = tid; i < rows; i += TH) {
        rhs[i] = P.T[(size_t)i * ld + nc];
        if (!COST) hg[i] = P.T[(size_t)i * ld + nc + 1];
    }
    __syncthreads();

    int cnt = 0, end = -1;
    while (cnt < P.kblock) {
        // ---- theta_cand: NaN never chosen, -0.0 == +0.0, the lowest index wins ties ---------------------------
        SensBest b = sens_empty();
        if (!COST) {
            for (int r = tid; r < m; r += TH) {
                const double g = hg[r];
                if (g < -LPX_EPS) {
                    SensBest c;
                    c.v = -__ddiv_rn(rhs[r], g);
                    c.i = r;
                    if (c.v == c.v) sens_pick<false>(b, c);
                }
            }
        } else {
            for (int j = tid; j < nc; j += TH) {
                const double h = hg[j];
                if (h < -LPX_EPS && !A.isb[j]) {
                    SensBest c;
                    c.v = -__ddiv_rn(z[j], h);
                    c.i = j;
                    if (c.v == c.v) sens_pick<false>(b, c);
                }
            }
        }
        b = sens_warp_reduce<false>(b);
        if (lane == 0) sred[warp] = b;
        __syncthreads();
        const SensBest all = sens_warp_reduce<false>(sred[lane]);
        __syncthreads();  // sred is free again
        const double cand = all.i == INT_MAX ? sens_inf() : all.v;
        const double th_end = cand < th_lo ? th_lo : cand;
        int stop = -1, pl = -1, pe = -1;
        double th_hi = th_end;
        if (th_end >= A.theta_max) {
            stop = LPX_PARAM_REACHED;
            th_hi = A.theta_max;
        } else if (k + 1 == A.seg_cap) {
            stop = LPX_PARAM_SEG_LIMIT;
        } else if (!COST) {
            // ---- row all.i leaves: bring it up to date into Pbuf[cnt], ratios z_j / -a_j over a_j < -EPS ----------
            const int l = all.i;
            if (tid < cnt) s_fl[tid] = P.Fbuf[(size_t)tid * cs + l];
            __syncthreads();
            double* prow = P.Pbuf + (size_t)cnt * ld;
            const double* Tl = P.T + (size_t)l * ld;
            for (int base = 0; base < ld; base += 8 * TH) {
                double r8[8];
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const int j = base + u * TH + tid;
                    r8[u] = j < ld ? Tl[j] : 0.0;
                }
                for (int s = 0; s < cnt; s++) {
                    const double fs = s_fl[s];
                    const bool same = l == s_L[s];
                    double ps[8];
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        const int j = base + u * TH + tid;
                        ps[u] = j < ld ? P.Pbuf[(size_t)s * ld + j] : 0.0;
                    }
#pragma unroll
                    for (int u = 0; u < 8; u++) r8[u] = same ? ps[u] : __dsub_rn(r8[u], __dmul_rn(fs, ps[u]));
                }
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const int j = base + u * TH + tid;
                    if (j < ld) {
                        const double a = r8[u];
                        prow[j] = a;
                        if (j < nc) {
                            double r = __longlong_as_double(0x7ff8000000000000LL);  // NaN: never eligible
                            if (a < -LPX_EPS) r = ddiv_by_pivot(z[j], dneg_s(a));
                            ratio[j] = r;
                        }
                    }
                }
            }
            __syncthreads();
            // the sequential "ratio < best - 1e-12" rule in first-hit rounds; thread t owns columns [t R, t R + R),
            // held in registers when they fit (as in stream_dual_lookahead_kernel)
            const int R = (nc + TH - 1) / TH;
            const int lo = tid * R, hi = min(nc, lo + R);
            const bool in_regs = R <= LPX_DUAL_SCAN_REGS;
            double rv[LPX_DUAL_SCAN_REGS];
#pragma unroll
            for (int u = 0; u < LPX_DUAL_SCAN_REGS; u++)
                rv[u] = (in_regs && lo + u < hi) ? ratio[lo + u] : __longlong_as_double(0x7ff8000000000000LL);
            double best = __longlong_as_double(0x7ff0000000000000LL);
            int e = -1, start = 0;
            while (true) {
                const double thr = __dsub_rn(best, LPX_MARGIN_DUAL);
                int c = INT_MAX;
                if (in_regs) {
#pragma unroll
                    for (int u = LPX_DUAL_SCAN_REGS - 1; u >= 0; u--)
                        if (lo + u >= start && rv[u] < thr) c = lo + u;
                } else {
                    for (int j = max(lo, start); j < hi; j++)
                        if (ratio[j] < thr) {
                            c = j;
                            break;
                        }
                }
                c = block_min_int<TH>(c, ired);
                if (c == INT_MAX) break;
                best = ratio[c];
                e = c;
                start = c + 1;
            }
            if (e < 0) {
                stop = LPX_PARAM_INFEASIBLE;
            } else {
                pl = l;
                pe = e;
            }
        } else {
            // ---- column all.i enters: bring it up to date (col, Fbuf[cnt]), ratios beta_i / a_i over a_i > EPS ------
            const int e = all.i;
            if (tid < cnt) s_pe[tid] = P.Pbuf[(size_t)tid * ld + e];
            __syncthreads();
            double* fout = P.Fbuf + (size_t)cnt * cs;
            for (int base = 0; base < rows; base += 8 * TH) {
                double c8[8];
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const int i = base + u * TH + tid;
                    c8[u] = i < rows ? P.T[(size_t)i * ld + e] : 0.0;
                }
                for (int s = 0; s < cnt; s++) {
                    const double ps = s_pe[s];
                    const int ls = s_L[s];
                    double f[8];
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        const int i = base + u * TH + tid;
                        f[u] = i < rows ? P.Fbuf[(size_t)s * cs + i] : 0.0;
                    }
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        const int i = base + u * TH + tid;
                        c8[u] = (i == ls) ? ps : __dsub_rn(c8[u], __dmul_rn(f[u], ps));
                    }
                }
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const int i = base + u * TH + tid;
                    if (i < rows) {
                        const double a = c8[u];
                        col[i] = a;
                        fout[i] = a;
                        if (i < m) {
                            double r = __longlong_as_double(0x7ff8000000000000LL);  // NaN: never eligible
                            if (a > LPX_EPS) r = ddiv_by_pos(rhs[i], a);
                            ratio[i] = r;
                        }
                    }
                }
            }
            __syncthreads();
            // the sequential "ratio < best - 1e-9" rule in first-hit rounds over interleaved rows (as in
            // stream_lookahead_kernel)
            double best = __longlong_as_double(0x7ff0000000000000LL);
            int row = -1, start = 0;
            while (true) {
                const double thr = __dsub_rn(best, LPX_MARGIN_PRIMAL);
                int c = INT_MAX;
                int i = tid;
                if (start > tid) i = tid + ((start - tid + TH - 1) / TH) * TH;
                for (; i < m; i += TH)
                    if (ratio[i] < thr) {
                        c = i;
                        break;
                    }
                c = block_min_int<TH>(c, ired);
                if (c == INT_MAX) break;
                best = ratio[c];
                row = c;
                start = c + 1;
            }
            if (row < 0) {
                stop = LPX_PARAM_UNBOUNDED;
            } else {
                pl = row;
                pe = e;
            }
        }

        // ---- segment k: theta_lo | theta_hi | z0 | dz | x0[n] | dx[n], read before the pivot; x0 / dx of the basic
        // decision variables only (the record is zero otherwise) ------------------------------------------------------
        if (A.seg) {
            double* rec = A.seg + (size_t)k * (4 + 2 * (size_t)n);
            if (tid == 0) {
                rec[0] = th_lo;
                rec[1] = th_hi;
                rec[2] = rhs[m];
                rec[3] = COST ? rhs[m + 1] : hg[m];
            }
            for (int r = tid; r < m; r += TH) {
                const int j = P.basis[r];
                if (j < n) {
                    rec[4 + j] = rhs[r];
                    if (!COST) rec[4 + n + j] = hg[r];
                }
            }
        }
        if (A.spv && tid == 0) {
            A.spv[2 * k] = pl;
            A.spv[2 * k + 1] = pe;
        }
        k++;
        if (stop >= 0) {
            end = stop;
            break;
        }
        __syncthreads();  // the record has read rhs / g / basis before they advance

        const int l = pl, e = pe;
        if (!COST) {
            // ---- column e brought up to date: this pivot's factor column; row l divided by its pivot element ----
            if (tid < cnt) s_pe[tid] = P.Pbuf[(size_t)tid * ld + e];
            __syncthreads();
            double* fout = P.Fbuf + (size_t)cnt * cs;
            for (int base = 0; base < rows; base += 8 * TH) {
                double c8[8];
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const int i = base + u * TH + tid;
                    c8[u] = i < rows ? P.T[(size_t)i * ld + e] : 0.0;
                }
                for (int s = 0; s < cnt; s++) {
                    const double ps = s_pe[s];
                    const int ls = s_L[s];
                    double f[8];
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        const int i = base + u * TH + tid;
                        f[u] = i < rows ? P.Fbuf[(size_t)s * cs + i] : 0.0;
                    }
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        const int i = base + u * TH + tid;
                        c8[u] = (i == ls) ? ps : __dsub_rn(c8[u], __dmul_rn(f[u], ps));
                    }
                }
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const int i = base + u * TH + tid;
                    if (i < rows) {
                        col[i] = c8[u];
                        fout[i] = c8[u];
                    }
                }
            }
            __syncthreads();
            const double piv = col[l], fz = col[m];
            double* prow = P.Pbuf + (size_t)cnt * ld;
            for (int j = tid; j < ld; j += TH) {
                const double pj = ddiv_by_pivot(prow[j], piv);
                prow[j] = pj;
                if (j < nc) z[j] = __dsub_rn(z[j], __dmul_rn(fz, pj));
            }
            // the compact RHS and g of row l equal row l's entries brought up to date (same operations, same order)
            const double prhs = ddiv_by_pivot(rhs[l], piv), pg = ddiv_by_pivot(hg[l], piv);
            __syncthreads();  // every thread has read rhs[l] and g[l]
            for (int i = tid; i < rows; i += TH) {
                const double f = col[i];
                rhs[i] = (i == l) ? prhs : __dsub_rn(rhs[i], __dmul_rn(f, prhs));
                hg[i] = (i == l) ? pg : __dsub_rn(hg[i], __dmul_rn(f, pg));
            }
        } else {
            // ---- row l brought up to date and divided by its pivot element; z and h advanced -------------------
            const double piv = col[l], fz = col[m], fh = col[m + 1];
            if (tid < cnt) s_fl[tid] = P.Fbuf[(size_t)tid * cs + l];
            __syncthreads();
            double* pout = P.Pbuf + (size_t)cnt * ld;
            const double* Tl = P.T + (size_t)l * ld;
            for (int base = 0; base < ld; base += 8 * TH) {
                double r8[8];
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const int j = base + u * TH + tid;
                    r8[u] = j < ld ? Tl[j] : 0.0;
                }
                for (int s = 0; s < cnt; s++) {
                    const double fs = s_fl[s];
                    const bool same = l == s_L[s];
                    double ps[8];
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        const int j = base + u * TH + tid;
                        ps[u] = j < ld ? P.Pbuf[(size_t)s * ld + j] : 0.0;
                    }
#pragma unroll
                    for (int u = 0; u < 8; u++) r8[u] = same ? ps[u] : __dsub_rn(r8[u], __dmul_rn(fs, ps[u]));
                }
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const int j = base + u * TH + tid;
                    if (j < ld) {
                        const double pj = ddiv_by_pos(r8[u], piv);
                        pout[j] = pj;
                        if (j < nc) {
                            z[j] = __dsub_rn(z[j], __dmul_rn(fz, pj));
                            hg[j] = __dsub_rn(hg[j], __dmul_rn(fh, pj));
                        }
                    }
                }
            }
            const double prhs = ddiv_by_pos(rhs[l], piv);
            __syncthreads();  // every thread has read rhs[l]
            for (int i = tid; i < rows; i += TH) rhs[i] = (i == l) ? prhs : __dsub_rn(rhs[i], __dmul_rn(col[i], prhs));
        }
        if (tid == 0) {
            s_L[cnt] = l;
            P.Lbuf[cnt] = l;
            if (COST) {
                A.isb[P.basis[l]] = 0;
                A.isb[e] = 1;
            }
            P.basis[l] = e;
        }
        cnt++;
        th_lo = th_end;
        __syncthreads();
    }
    if (tid == 0) {
        ctl->block_cnt = cnt;
        ctl->pivots = done + cnt;
        S->th_lo = th_lo;
        S->k = k;
        S->end = end;
    }
}

}  // namespace lpx
