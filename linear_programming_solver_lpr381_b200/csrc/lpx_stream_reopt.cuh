// lpx_stream_reopt.cuh — re-optimization of an optimal streaming session (lpx_session_reoptimize): the query's
// tableau is built in HBM straight from the base session's, then RHS / ROW queries run the streaming Dual Simplex
// below and COST / COL queries the session's Primal Simplex protocol.  The edits are defined in include/lpx.h
// ("Re-optimization"); oracle/orc_reopt.cpp restates them as sequential loops.
//
// Included by lpx_stream.cu after StreamParams / StreamCtl and the per-pivot kernels.

namespace lpx {

// One term of an edit, in the definition's order (the host keeps only the terms whose payload coefficient is
// non-zero):
//   RHS / COL  v (+ or -)= a * Tb[r][idx]   on every row r; aux = 1 subtracts (the s2 term of an EQ row)
//   COST       z[k] += a * Tb[idx][k] when idx >= 0 (the basic row of column aux), then z[aux] -= a
//   ROW        row[k] -= a * Tb[idx][k]     (idx: a basis row whose decision variable has a non-zero coefficient)
struct ReoptTerm {
    double a;
    int idx;
    int aux;
};

// The query's padded tableau Q.T (Q.rows x Q.ld, pad columns zero) from the base tableau Tb (mb + 1 rows, width wb,
// leading dimension ldb, nb decision variables).  grid = (column strips of 256, row groups).  pay: the query's
// payload on the device (ROW reads its raw row there); zstart: the new column's z-row start -c'_new (COL); ge: the
// added row is '>=' (ROW).  FP64 with separate multiply / add / subtract, term by term in the definition's order.
__global__ void __launch_bounds__(256) stream_reopt_build_kernel(StreamParams Q, const double* __restrict__ Tb, int ldb,
                                                                 int wb, int mb, int nb, int kind,
                                                                 const ReoptTerm* __restrict__ t, int nt,
                                                                 const double* __restrict__ pay, double zstart, int ge) {
    const int j = blockIdx.x * 256 + threadIdx.x;
    if (j >= Q.ld) return;
    const int rhs_s = wb - 1;
    auto src = [&](int r, int k) { return Tb[(size_t)r * ldb + k]; };
    for (int i = blockIdx.y; i < Q.rows; i += gridDim.y) {
        double v = 0.0;
        if (j < Q.width) {
            if (kind == LPX_REOPT_RHS) {
                v = src(i, j);
                if (j == rhs_s)
                    for (int q = 0; q < nt; q++) {
                        const double d = __dmul_rn(t[q].a, src(i, t[q].idx));
                        v = t[q].aux ? __dsub_rn(v, d) : __dadd_rn(v, d);
                    }
            } else if (kind == LPX_REOPT_COST) {
                v = src(i, j);
                if (i == mb)
                    for (int q = 0; q < nt; q++) {
                        if (t[q].idx >= 0) v = __dadd_rn(v, __dmul_rn(t[q].a, src(t[q].idx, j)));
                        if (j == t[q].aux) v = __dsub_rn(v, t[q].a);
                    }
            } else if (kind == LPX_REOPT_ROW) {
                if (i != mb) {  // an old row (i > mb: the z-row): the old RHS position becomes the new slack column
                    const int si = i < mb ? i : mb;
                    v = j < rhs_s ? src(si, j) : (j == rhs_s ? 0.0 : src(si, rhs_s));
                } else if (j == rhs_s) {
                    v = 1.0;
                } else {  // the raw row (GE: every entry negated, zeros included), then the basic columns eliminated
                    const int k = j < rhs_s ? j : rhs_s;
                    v = k < nb ? pay[k] : (k == rhs_s ? pay[nb + 1] : 0.0);
                    if (ge) v = dneg_s(v);
                    for (int q = 0; q < nt; q++) v = __dsub_rn(v, __dmul_rn(t[q].a, src(t[q].idx, k)));
                }
            } else {  // LPX_REOPT_COL: the new column sits at nb, the old columns from nb on move right by one
                if (j != nb) {
                    v = src(i, j < nb ? j : j - 1);
                } else {
                    v = i == mb ? zstart : 0.0;
                    for (int q = 0; q < nt; q++) {
                        const double d = __dmul_rn(t[q].a, src(i, t[q].idx));
                        v = t[q].aux ? __dsub_rn(v, d) : __dadd_rn(v, d);
                    }
                }
            }
        }
        Q.T[(size_t)i * Q.ld + j] = v;
    }
}

// One Dual Simplex pivot of a streaming session, decided by one CTA; stream_update_kernel<4> applies it (npartial 0,
// no entering capture: the next entering column depends on the next leaving row, which the pass decides).  The rules
// are dual_core's (oracle/orc_pooled.cpp), the loop of the batched re-optimization kernel:
//   iteration limit first (P.max_iter = 10000), then the leaving row l = most negative compact rhsbuf[i] < -1e-9
//   (first index on ties; none: OPTIMAL), then the entering column: ratios z_j / (-a_lj) over a_lj < -1e-9, j < W - 1,
//   scanned with "ratio < best - 1e-12" in column order (none: INFEASIBLE).
// Row l and the z-row are contiguous in HBM; the ratios go to P.ratio (sized by the width in dual sessions).  Then
// column e is gathered into colbuf[k & 1] for the pass and row l is normalised by its (negative) pivot element.
// probe_only: resolve the status of the tableau as it stands, no pivot (lpx_session_sync).
__global__ void __launch_bounds__(1024) stream_dual_select_kernel(StreamParams P, int probe_only) {
    __shared__ ArgMin red[34];
    __shared__ int ired[34];
    StreamCtl* ctl = P.ctl;
    const int tid = threadIdx.x;
    if (tid == 0) ctl->active = 0;
    if (ctl->status != LPX_RUNNING) return;
    const int k = ctl->pivots;
    if (k >= P.max_iter) {  // "if (iter > 10000) return ITER_LIMIT" comes before the leaving-row test
        if (tid == 0) ctl->status = LPX_S_ITER_LIMIT;
        return;
    }
    const int m = P.m;
    const int l = block_argmin_below<1024>(P.rhsbuf, m, -LPX_EPS, red);
    if (l < 0) {
        if (tid == 0) ctl->status = LPX_OPTIMAL;
        return;
    }
    double* Tl = P.T + (size_t)l * P.ld;
    const double* Tz = P.T + (size_t)m * P.ld;
    const int nc = P.width - 1;
    for (int j = tid; j < nc; j += 1024) {
        const double a = Tl[j];
        double r = __longlong_as_double(0x7ff8000000000000LL);  // NaN: never eligible
        if (a < -LPX_EPS) r = ddiv_by_pivot(Tz[j], dneg_s(a));
        P.ratio[j] = r;
    }
    __syncthreads();
    // the sequential rule "take j if ratio < best - 1e-12", reproduced exactly as in stream_select_kernel: repeatedly
    // find the FIRST column after the last accepted one that beats the running best
    const int R = (nc + 1023) / 1024;
    const int lo = tid * R, hi = min(nc, lo + R);
    double best = __longlong_as_double(0x7ff0000000000000LL);
    int e = -1, start = 0;
    while (true) {
        const double thr = __dsub_rn(best, LPX_MARGIN_DUAL);
        int cand = INT_MAX;
        for (int j = max(lo, start); j < hi; j++)
            if (P.ratio[j] < thr) {
                cand = j;
                break;
            }
        cand = block_min_int<1024>(cand, ired);
        if (cand == INT_MAX) break;
        best = P.ratio[cand];
        e = cand;
        start = cand + 1;
    }
    if (e < 0) {
        if (tid == 0) ctl->status = LPX_INFEASIBLE;
        return;
    }
    if (probe_only) return;

    // column e before the pivot (the pass's factors; row l's entry is the pivot element) ...
    double* col = P.colbuf + (size_t)(k & 1) * P.colstride;
    for (int i = tid; i < P.rows; i += 1024) col[i] = P.T[(size_t)i * P.ld + e];
    const double piv = Tl[e];
    __syncthreads();
    // ... then row l divided by the pivot element (true division, as pivot() does)
    for (int j = tid; j < P.ld; j += 1024) {
        const double pj = ddiv_by_pivot(Tl[j], piv);
        P.prow[j] = pj;
        Tl[j] = pj;
        if (j == nc) P.rhsbuf[l] = pj;
    }
    if (tid == 0) {
        P.basis[l] = e;
        if (k < P.pivlog_cap) {
            P.pivlog[2 * k] = e;
            P.pivlog[2 * k + 1] = l;
        }
        ctl->leave = l;
        ctl->capture = -1;
        ctl->k = k;
        ctl->pivots = k + 1;
        ctl->enter = -1;
        ctl->active = 1;
    }
}

}  // namespace lpx
