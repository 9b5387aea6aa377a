// lpx_stream_twophase.cuh — the two-phase Simplex (include/lpx.h, "Two-phase Simplex") on one LP whose tableau lives
// in HBM (lpx_two_phase_session_open).  The build kernel writes the normalised tableau with its slack and artificial
// columns and the Phase I row m + 1; then one CTA decides up to K pivots of Phase I, the drive-out and Phase II on the
// tableau as the last pass left it, and the unchanged blocked pass (stream_update_block_kernel /
// stream_update_block_tma_kernel) applies them in one HBM pass.  The rule of lpx_stream_block.cuh,
//       v <- (row == l_s) ? p_s[col] : v - f_s[row] * p_s[col]          for the pending pivots s in order,
// brings every value a decision reads up to date, so K decisions and one pass give the bits of K single passes, and
// the whole solve the bits of oracle/orc_twophase.cpp and lpx_two_phase_solve_batched.
//
// The pass updates every row of the session.  In Phase II that includes row m + 1, which the definition leaves alone
// from the end of Phase I on; nothing reads that row again and no output contains it.
//
// Included by lpx_stream.cu after lpx_stream_param.cuh (StreamParams / StreamCtl, block_min_int, LPX_BLOCK_KMAX).

namespace lpx {

// The look-ahead's vectors: dynamic shared memory where they fit, global memory otherwise (vec_place).
//   TV_Z     the active objective row (Phase I: row m + 1; from the passed feasibility test on: row m), ld
//   TV_RHS   compact RHS, colstride
//   TV_COL   the entering column brought up to date, colstride
//   TV_RATIO leaving-row ratios, colstride
enum { TV_Z = 0, TV_RHS, TV_COL, TV_RATIO, TV_N };

// The solve's progress, handed from look-ahead to look-ahead (next to StreamCtl, which holds the status and the pivot
// count).
struct TwoPhaseState {
    int phase;   // 1: Phase I; 2: from the passed feasibility test on (the drive-out, then Phase II)
    int cursor;  // phase 2: the next row the drive-out examines (m: the drive-out is over)
    int p1;      // Phase I pivots, drive-out pivots included
    int pad;
    double S;    // the normalised b summed over the artificial rows in row order from +0
};

struct TwoPhaseLa {
    double* gvec[TV_N];  // global-memory home of each vector
    int soff[TV_N];      // its offset in dynamic shared memory (doubles), -1: global memory
    TwoPhaseState* st;
    int ns;              // n + s: the structural and slack columns
};

// Row i's normalisation and columns: flip (b_i < 0), slack column (-1 for EQ), artificial column (-1 for none).
struct TwoPhaseRows {
    const int* flip;
    const int* slk;
    const int* art;
    const int* arows;  // the artificial rows in row order
    int a;
};

// Entry (i, j) of constraint row i < m as the definition writes it.
__device__ __forceinline__ double two_phase_entry(const double* __restrict__ A, const double* __restrict__ b,
                                                  const TwoPhaseRows& R, int n, int rhs, int i, int j) {
    const bool f = R.flip[i] != 0;
    if (j < n) {
        const double v = A[(size_t)i * n + j];
        return f ? dneg_s(v) : v;
    }
    if (j == rhs) return f ? dneg_s(b[i]) : b[i];
    if (j == R.slk[i]) return R.art[i] >= 0 ? -1.0 : 1.0;  // a row with both a slack and an artificial is GE
    if (j == R.art[i]) return 1.0;
    return 0.0;
}

// The initial tableau: rows 0..m-1 the normalised constraints, row m the objective row, row m + 1 the Phase I row
// (w_j = ((+0 - T[i1][j]) - T[i2][j]) - ... over the artificial rows in row order, one thread per column; +0 on the
// artificial columns), pad columns zero; and the initial basis.  grid = (column strips of 256, row groups).
__global__ void __launch_bounds__(256) stream_two_phase_build_kernel(StreamParams P, const double* __restrict__ A,
                                                                     const double* __restrict__ b,
                                                                     const double* __restrict__ c, TwoPhaseRows R,
                                                                     int sense, int ns) {
    const int j = blockIdx.x * 256 + threadIdx.x;
    const int m = P.m, n = P.n, W = P.width, rhs = W - 1;
    if (blockIdx.x == 0)
        for (int i = blockIdx.y * 256 + threadIdx.x; i < m; i += gridDim.y * 256)
            P.basis[i] = R.art[i] >= 0 ? R.art[i] : R.slk[i];
    if (j >= P.ld) return;
    for (int i = blockIdx.y; i < P.rows; i += gridDim.y) {
        double v = 0.0;
        if (j < W) {
            if (i < m) {
                v = two_phase_entry(A, b, R, n, rhs, i, j);
            } else if (i == m) {
                if (j < n) v = dneg_s(sense == 1 ? dneg_s(c[j]) : c[j]);  // T[m][j] = -C[j], Min -> Max
            } else if (j < ns || j == rhs) {
                // the artificial rows' entries of a batch are loaded together, then subtracted in row order
                for (int q0 = 0; q0 < R.a; q0 += 8) {
                    double x[8];
#pragma unroll
                    for (int u = 0; u < 8; u++) x[u] = q0 + u < R.a ? two_phase_entry(A, b, R, n, rhs, R.arows[q0 + u], j) : 0.0;
#pragma unroll
                    for (int u = 0; u < 8; u++)
                        if (q0 + u < R.a) v = __dsub_rn(v, x[u]);
                }
            }
        }
        P.T[(size_t)i * P.ld + j] = v;
    }
}

// One CTA, 1024 threads: up to min(budget, P.kblock) pivots on the tableau as the last pass left it.
//   Phase I    ITER_LIMIT when the pivot count has reached P.max_iter; ChooseEntering on row m + 1 over columns
//              < W - 1; the leaving row by the 1e-9 first-hit replay over rows < m.  No column or no row: the
//              feasibility test !(w >= -1e-9 (1 + S)) on the up-to-date RHS of row m + 1 (INFEASIBLE), else phase 2
//              and row m, brought up to date, becomes the active objective row.
//   Drive-out  rows r ascending from the cursor whose basic variable is >= n + s: row r brought up to date, the lowest
//              j < n + s with |T[r][j]| > 1e-9; none: the row is redundant, no pivot; else the pivot (r, j), whose
//              element can be negative (ddiv_by_pivot).  Counted as Phase I pivots and against the budget, not checked
//              against the limit.
//   Phase II   as Phase I on row m over columns < n + s: OPTIMAL / UNBOUNDED.
// budget = 0: probe only.  It resolves every terminal status reachable without a pivot, and may advance the phase and
// the drive-out cursor past redundant rows, since those make no pivot.  A terminal status met inside a block leaves
// the pivots decided before it for the pass, then stands.
__global__ void __launch_bounds__(1024) stream_two_phase_lookahead_kernel(StreamParams P, TwoPhaseLa A, int budget) {
    extern __shared__ double sm_tp[];
    __shared__ ArgMin red[34];
    __shared__ int ired[34];
    __shared__ int s_L[LPX_BLOCK_KMAX];
    __shared__ double s_pe[LPX_BLOCK_KMAX];  // p_s[e]   for the column being brought up to date
    __shared__ double s_fl[LPX_BLOCK_KMAX];  // f_s[l]   for the row being brought up to date
    constexpr int TH = 1024;
    const int tid = threadIdx.x;
    const int ld = P.ld, cs = P.colstride, m = P.m, rows = P.rows, nc = P.width - 1, ns = A.ns;
    double* vec[TV_N];
#pragma unroll
    for (int v = 0; v < TV_N; v++) vec[v] = A.soff[v] >= 0 ? sm_tp + A.soff[v] : A.gvec[v];
    double* z = vec[TV_Z];
    double* rhs = vec[TV_RHS];
    double* col = vec[TV_COL];
    double* ratio = vec[TV_RATIO];
    StreamCtl* ctl = P.ctl;
    TwoPhaseState* S = A.st;
    const int status0 = ctl->status;
    const int done = ctl->pivots;
    int phase = S->phase, cursor = S->cursor, p1 = S->p1;
    const double tol = __dmul_rn(1e-9, __dadd_rn(1.0, S->S));
    __syncthreads();  // every thread has read the state before thread 0 rewrites it
    if (tid == 0) ctl->block_cnt = 0;
    if (status0 != LPX_RUNNING) return;

    const double* Tz = P.T + (size_t)(phase == 1 ? m + 1 : m) * ld;
    for (int j = tid; j < ld; j += TH) z[j] = Tz[j];
    for (int i = tid; i < rows; i += TH) rhs[i] = P.rhsbuf[i];
    __syncthreads();

    const bool probe = budget <= 0;
    const int steps = probe ? 0 : min(budget, P.kblock);
    int cnt = 0, st = LPX_RUNNING;

    // Row r brought up to date into out[0..ld).  norm: divided by piv (ddiv_by_pivot: bit-identical to ddiv_by_pos for
    // a positive element) and z advanced by fz times it over columns < W - 1.
    auto row_pass = [&](int r, double* out, bool norm, double piv, double fz) {
        if (tid < cnt) s_fl[tid] = P.Fbuf[(size_t)tid * cs + r];
        __syncthreads();
        const double* Tr = P.T + (size_t)r * ld;
        for (int base = 0; base < ld; base += 8 * TH) {
            double r8[8];
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int j = base + u * TH + tid;
                r8[u] = j < ld ? Tr[j] : 0.0;
            }
            for (int s = 0; s < cnt; s++) {
                const double fs = s_fl[s];
                const bool same = r == s_L[s];
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
                    if (norm) {
                        const double pj = ddiv_by_pivot(r8[u], piv);
                        out[j] = pj;
                        if (j < nc) z[j] = __dsub_rn(z[j], __dmul_rn(fz, pj));
                    } else {
                        out[j] = r8[u];
                    }
                }
            }
        }
        __syncthreads();
    };
    // Column e brought up to date into col and Fbuf[cnt] (this pivot's factor column); ratios: the leaving-row ratios
    // over rows < m.
    auto col_pass = [&](int e, bool ratios) {
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
                    if (ratios && i < m) {
                        double r = __longlong_as_double(0x7ff8000000000000LL);  // NaN: never eligible
                        if (a > LPX_EPS) r = ddiv_by_pos(rhs[i], a);
                        ratio[i] = r;
                    }
                }
            }
        }
        __syncthreads();
    };
    // The compact RHS advanced by the pivot (l, e) whose row is already in Pbuf[cnt], and the bookkeeping.
    auto finish_pivot = [&](int l, int e, double piv) {
        const double prhs = ddiv_by_pivot(rhs[l], piv);
        __syncthreads();  // every thread has read rhs[l]
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
    };

    while (probe || cnt < steps) {
        if (phase == 2 && cursor < m) {
            // ---- drive-out: the next row from the cursor whose basic variable is an artificial ------------------
            int r = INT_MAX;
            for (int i = cursor + tid; i < m; i += TH)
                if (P.basis[i] >= ns) {
                    r = i;
                    break;
                }
            r = block_min_int<TH>(r, ired);
            if (r == INT_MAX) {
                cursor = m;
                continue;
            }
            double* prow = P.Pbuf + (size_t)cnt * ld;
            row_pass(r, prow, false, 1.0, 0.0);
            int e = INT_MAX;
            for (int j = tid; j < ns; j += TH)
                if (fabs(prow[j]) > LPX_EPS) {
                    e = j;
                    break;
                }
            e = block_min_int<TH>(e, ired);
            if (e == INT_MAX) {  // redundant: the artificial stays basic
                cursor = r + 1;
                continue;
            }
            cursor = r;
            if (probe) break;
            col_pass(e, false);
            const double piv = col[r], fz = col[m];
            for (int j = tid; j < ld; j += TH) {
                const double pj = ddiv_by_pivot(prow[j], piv);
                prow[j] = pj;
                if (j < nc) z[j] = __dsub_rn(z[j], __dmul_rn(fz, pj));
            }
            finish_pivot(r, e, piv);
            p1++;
            cursor = r + 1;
            continue;
        }
        // ---- Phase I on row m + 1 over columns < W - 1, Phase II on row m over columns < n + s -------------------
        if (done + cnt >= P.max_iter) {  // "iter > MaxIterations" before the column is chosen
            st = LPX_S_ITER_LIMIT;
            break;
        }
        const int e = block_argmin_below<TH>(z, phase == 1 ? nc : ns, -LPX_EPS, red);
        int l = -1;
        if (e >= 0) {
            col_pass(e, true);
            double best = __longlong_as_double(0x7ff0000000000000LL);
            int start = 0;
            while (true) {
                const double thr = __dsub_rn(best, LPX_MARGIN_PRIMAL);
                int cand = INT_MAX;
                int i = tid;
                if (start > tid) i = tid + ((start - tid + TH - 1) / TH) * TH;
                for (; i < m; i += TH)
                    if (ratio[i] < thr) {
                        cand = i;
                        break;
                    }
                cand = block_min_int<TH>(cand, ired);
                if (cand == INT_MAX) break;
                best = ratio[cand];
                l = cand;
                start = cand + 1;
            }
        }
        if (e < 0 || l < 0) {
            if (phase == 2) {
                st = e < 0 ? LPX_OPTIMAL : LPX_UNBOUNDED;
                break;
            }
            // ---- end of Phase I: the feasibility test, then row m becomes the active objective row ---------------
            if (!(rhs[m + 1] >= -tol)) {
                st = LPX_INFEASIBLE;
                break;
            }
            phase = 2;
            cursor = 0;
            row_pass(m, z, false, 1.0, 0.0);
            continue;
        }
        if (probe) break;
        const double piv = col[l], fz = col[phase == 1 ? m + 1 : m];
        row_pass(l, P.Pbuf + (size_t)cnt * ld, true, piv, fz);
        finish_pivot(l, e, piv);
        if (phase == 1) p1++;
    }
    for (int i = tid; i < rows; i += TH) P.rhsbuf[i] = rhs[i];
    if (tid == 0) {
        ctl->block_cnt = cnt;
        ctl->pivots = done + cnt;
        if (st != LPX_RUNNING) ctl->status = st;
        S->phase = phase;
        S->cursor = cursor;
        S->p1 = p1;
    }
}

}  // namespace lpx
