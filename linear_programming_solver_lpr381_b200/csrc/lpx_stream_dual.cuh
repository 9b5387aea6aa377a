// lpx_stream_dual.cuh — blocked look-ahead for the streaming Dual Simplex (cold Dual Simplex sessions and the RHS / ROW
// re-optimization queries).  The rule of lpx_stream_block.cuh,
//       v <- (row == l_s) ? p_s[col] : v - f_s[row] * p_s[col]          for the pending pivots s in order,
// brings every value a Dual Simplex decision reads up to date from the tableau as the last pass left it, so one CTA
// decides up to K pivots with the rules of stream_dual_select_kernel and the unchanged blocked pass
// (stream_update_block_kernel / stream_update_block_tma_kernel) applies them: bit-identical to K per-pivot passes.
//
// Included by lpx_stream.cu after lpx_stream_block.cuh (StreamParams / StreamCtl, block_min_int, LPX_BLOCK_KMAX).

namespace lpx {

#define LPX_DUAL_SCAN_REGS 16  // ratios a thread holds in registers for the entering-column scan (W - 1 <= 16 K columns)

// Dynamic shared memory of stream_dual_lookahead_kernel: z[ld] | rhs[cs] | col[cs].  The width-long ratio vector goes
// to P.ratio (sized max(colstride, ld) in dual sessions) and the pivot row is built in Pbuf[s]: both stay in L2.
static inline size_t dual_lookahead_smem(const StreamParams& P) {
    return ((size_t)P.ld + 2 * (size_t)P.colstride) * 8;
}

// One CTA, 1024 threads.  For each decided pivot s (at most min(budget, P.kblock)):
//   iteration limit (done + s >= P.max_iter: ITER_LIMIT); leaving row l = first minimum of the compact RHS below -1e-9
//   over rows < m (none: OPTIMAL); row l brought up to date into Pbuf[s] and the ratios z_j / (-a_lj) over
//   a_lj < -1e-9, j < W - 1, replayed with "ratio < best - 1e-12" (none: INFEASIBLE); column e brought up to date into
//   Fbuf[s]; row l divided by its pivot element in place; compact RHS and z advanced with the same rule.
// budget = 0: probe only (resolve OPTIMAL / INFEASIBLE / ITER_LIMIT for the tableau as it stands, no pivot).
// A terminal status met inside a block leaves the pivots decided before it for the pass, then stands.
__global__ void __launch_bounds__(1024) stream_dual_lookahead_kernel(StreamParams P, int budget) {
    extern __shared__ double sm_dl[];
    __shared__ ArgMin red[34];
    __shared__ int ired[34];
    __shared__ int s_L[LPX_BLOCK_KMAX];
    __shared__ double s_pe[LPX_BLOCK_KMAX];  // p_s[e]   for the column being brought up to date
    __shared__ double s_fl[LPX_BLOCK_KMAX];  // f_s[l]   for the row being brought up to date
    constexpr int TH = 1024;
    const int tid = threadIdx.x;
    const int ld = P.ld, cs = P.colstride, m = P.m, rows = P.rows, nc = P.width - 1;
    double* z = sm_dl;
    double* rhs = z + ld;
    double* col = rhs + cs;
    StreamCtl* ctl = P.ctl;
    const int status0 = ctl->status;
    const int done = ctl->pivots;
    if (tid == 0) ctl->block_cnt = 0;
    if (status0 != LPX_RUNNING) return;

    const double* Tz = P.T + (size_t)m * ld;
    for (int j = tid; j < ld; j += TH) z[j] = Tz[j];
    for (int i = tid; i < rows; i += TH) rhs[i] = P.rhsbuf[i];
    __syncthreads();

    const bool probe = budget <= 0;
    const int steps = probe ? 1 : min(budget, P.kblock);
    int cnt = 0, st = LPX_RUNNING;
    for (int k = 0; k < steps; k++) {
        if (done + cnt >= P.max_iter) {  // "if (iter > 10000)" comes before the leaving-row test
            st = LPX_S_ITER_LIMIT;
            break;
        }
        // ---- leaving row on the up-to-date compact RHS ------------------------------------------------
        const int l = block_argmin_below<TH>(rhs, m, -LPX_EPS, red);
        if (l < 0) {
            st = LPX_OPTIMAL;
            break;
        }
        // ---- row l: gather, apply the pivots decided so far (into Pbuf[cnt]), form the ratios --------------
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
                        P.ratio[j] = r;
                    }
                }
            }
        }
        __syncthreads();
        // ---- entering column: the sequential "ratio < best - 1e-12" rule, first-hit rounds ------------------
        // Thread t owns the R consecutive columns from t * R.  Up to LPX_DUAL_SCAN_REGS of them are loaded once, all
        // loads in flight together, and every round scans registers: a round that walks them in global memory pays
        // one dependent L2 round trip per column.
        const int R = (nc + TH - 1) / TH;
        const int lo = tid * R, hi = min(nc, lo + R);
        const bool in_regs = R <= LPX_DUAL_SCAN_REGS;
        double rv[LPX_DUAL_SCAN_REGS];
#pragma unroll
        for (int u = 0; u < LPX_DUAL_SCAN_REGS; u++)
            rv[u] = (in_regs && lo + u < hi) ? P.ratio[lo + u] : __longlong_as_double(0x7ff8000000000000LL);
        double best = __longlong_as_double(0x7ff0000000000000LL);
        int e = -1, start = 0;
        while (true) {
            const double thr = __dsub_rn(best, LPX_MARGIN_DUAL);
            int cand = INT_MAX;
            if (in_regs) {
#pragma unroll
                for (int u = LPX_DUAL_SCAN_REGS - 1; u >= 0; u--)
                    if (lo + u >= start && rv[u] < thr) cand = lo + u;
            } else {
                for (int j = max(lo, start); j < hi; j++)
                    if (P.ratio[j] < thr) {
                        cand = j;
                        break;
                    }
            }
            cand = block_min_int<TH>(cand, ired);
            if (cand == INT_MAX) break;
            best = P.ratio[cand];
            e = cand;
            start = cand + 1;
        }
        if (e < 0) {
            st = LPX_INFEASIBLE;
            break;
        }
        if (probe) break;
        // ---- column e: gather, apply the pivots decided so far; it is this pivot's factor column --------------
        if (tid < cnt) s_pe[tid] = P.Pbuf[(size_t)tid * ld + e];
        __syncthreads();
        double* fout = P.Fbuf + (size_t)cnt * cs;
        for (int base = 0; base < rows; base += 8 * TH) {
            double c[8];
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int i = base + u * TH + tid;
                c[u] = i < rows ? P.T[(size_t)i * ld + e] : 0.0;
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
                    c[u] = (i == ls) ? ps : __dsub_rn(c[u], __dmul_rn(f[u], ps));
                }
            }
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int i = base + u * TH + tid;
                if (i < rows) {
                    col[i] = c[u];
                    fout[i] = c[u];
                }
            }
        }
        __syncthreads();
        // ---- row l divided by the pivot element (true division, as pivot() does), z advanced ----------------
        const double piv = col[l], fz = col[m];
        for (int j = tid; j < ld; j += TH) {
            const double pj = ddiv_by_pivot(prow[j], piv);
            prow[j] = pj;
            if (j < nc) z[j] = __dsub_rn(z[j], __dmul_rn(fz, pj));
        }
        // the compact RHS of row l equals row l's RHS entry brought up to date (same operations, same order)
        const double prhs = ddiv_by_pivot(rhs[l], piv);
        __syncthreads();  // every thread has read rhs[l]; z is complete for the next pivot's ratios
        for (int i = tid; i < rows; i += TH) rhs[i] = (i == l) ? prhs : __dsub_rn(rhs[i], __dmul_rn(col[i], prhs));
        if (tid == 0) {
            s_L[cnt] = l;
            P.Lbuf[cnt] = l;
            P.basis[l] = e;
            if (done + cnt < P.pivlog_cap) {
                P.pivlog[2 * (done + cnt)] = e;
                P.pivlog[2 * (done + cnt) + 1] = l;
            }
        }
        cnt++;
        __syncthreads();
    }
    for (int i = tid; i < rows; i += TH) P.rhsbuf[i] = rhs[i];
    if (tid == 0) {
        ctl->block_cnt = cnt;
        ctl->pivots = done + cnt;
        if (st != LPX_RUNNING) ctl->status = st;
    }
}

}  // namespace lpx
