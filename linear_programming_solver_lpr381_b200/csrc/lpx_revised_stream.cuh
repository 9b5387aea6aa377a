// lpx_revised_stream.cuh — Revised Primal Simplex on the whole GPU (lpx_revised_solve past the one-CTA
// kernel of lpx_revised.cu).  Same algorithm, same operation order, same bits (RevisedPrimalSimplex.cs:17-145):
//
//   refresh  [B | I] (m x ld, ld = 2m padded to 16 doubles) is built from the columns Bidx of A | I and
//            inverted by Gauss-Jordan with the blocked look-ahead protocol of the streaming tableau
//            (lpx_stream_block.cuh): one Gauss-Jordan step IS a tableau pivot (true division of the pivot
//            row, unfused a - f * p on every other row) whose entering column is known in advance (step k
//            eliminates column k).  rev_lookahead_kernel decides up to K steps from the matrix as the last
//            pass left it, and ONE unchanged blocked pass applies them.  The reference's row swap is a
//            logical permutation: logical row i lives in physical row perm[i], so the swap costs nothing
//            and every element still sees exactly the reference's operations (the elimination of a row by
//            its own entry in the pivot column does not depend on where the row is stored).
//   price    pi = c_B B^-1, r_N = c_N - pi N, entering = most negative r_N below -1e-9 (lowest LIST
//            position on ties: per-CTA partials, then one CTA), d = B^-1 a_e, the ratios, the certified
//            margin scan (1e-12) and the list update.
//
// Every dot product is summed by one thread per output in index order, never by a tree.  Iterations are
// enqueued in chunks; every kernel returns once the status word is no longer RUNNING, and the host
// synchronises once per chunk.
//
// Included by lpx_stream.cu (uses StreamParams / StreamCtl, the blocked pass kernels and their sizing).
#pragma once

namespace lpx {

#define LPX_REV_LA_THREADS 512
#ifndef LPX_REV_DEFAULT_K
#define LPX_REV_DEFAULT_K 8  // Gauss-Jordan steps per pass when opt.stream_block is 0
#endif

struct RevCtl {
    StreamCtl s;  // s.status: the status word; s.pivots: Gauss-Jordan steps of the current inversion
    int iters;    // iterations performed
    int pos;      // entering position in the nonbasic list (this iteration)
    int enter;    // entering column (this iteration)
    int pad;
    double theta;  // chosen ratio (this iteration)
};

struct RevParams {
    int m, n, ntot, sense, max_iter, ld;
    const double* A;  // m x n
    const double* b;
    const double* c;
    double* Af;     // m x ntot: A | I
    double* cf;     // ntot: c (negated for MAX, Standardize :153-154), 0 for the slacks
    double* aug;    // m x ld: [B | I] during the inversion
    int* perm;      // m: logical row -> physical row of aug
    double* Binv;   // m x m, row-major (logical rows)
    double* BinvT;  // m x m, its transpose (coalesced reads for the one-thread-per-row sums)
    double* xB;
    double* cB;
    double* pi;
    double* d;
    double* ratio;
    double* rN;     // n
    int* Bidx;      // m
    int* Nidx;      // n
    ArgMin* part;   // per-CTA entering candidates
    RevCtl* ctl;
    int* pivots;    // 2 per iteration (entering column, leaving row), pivots_cap of them
    double* theta;
    int pivots_cap;
    double* history;  // history_cap records of rev_history_stride(m, n) doubles
    int history_cap;
};

#define LPX_REV_TH 128  // threads of the one-output-per-thread kernels

__device__ __forceinline__ bool rev_running(const RevParams& R) { return R.ctl->s.status == LPX_RUNNING; }

// A | I, c, the slack basis, the identity list; the control block.
__global__ void __launch_bounds__(256) rev_setup_kernel(RevParams R) {
    const size_t stride = (size_t)gridDim.x * blockDim.x, t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t ntot = (size_t)R.ntot, total = (size_t)R.m * ntot;
    for (size_t k = t0; k < total; k += stride) {
        const size_t i = k / ntot, j = k - i * ntot;
        R.Af[k] = j < (size_t)R.n ? R.A[i * R.n + j] : (j == R.n + i ? 1.0 : 0.0);
    }
    for (size_t j = t0; j < ntot; j += stride) {
        double v = 0.0;
        if (j < (size_t)R.n) v = R.sense == 0 ? dneg_s(R.c[j]) : R.c[j];
        R.cf[j] = v;
    }
    for (size_t i = t0; i < (size_t)R.m; i += stride) R.Bidx[i] = R.n + (int)i;
    for (size_t j = t0; j < (size_t)R.n; j += stride) R.Nidx[j] = (int)j;
    if (t0 == 0) {
        RevCtl& c = *R.ctl;
        c.s.status = LPX_RUNNING;
        c.s.pivots = c.s.block_cnt = 0;
        c.iters = c.pos = 0;
        c.enter = -1;
        c.theta = 0.0;
    }
}

// [B | I]: column j < m of B is column Bidx[j] of A | I; pad columns are zero.  Resets the permutation.
__global__ void __launch_bounds__(256) rev_build_kernel(RevParams R) {
    if (!rev_running(R)) return;
    const int m = R.m;
    const size_t ld = (size_t)R.ld, total = (size_t)m * ld;
    const size_t stride = (size_t)gridDim.x * blockDim.x, t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (size_t k = t0; k < total; k += stride) {
        const size_t i = k / ld, j = k - i * ld;
        double v = 0.0;
        if (j < (size_t)m) v = R.Af[i * R.ntot + R.Bidx[j]];
        else if (j == m + i) v = 1.0;
        R.aug[k] = v;
    }
    for (size_t i = t0; i < (size_t)m; i += stride) R.perm[i] = (int)i;
    if (t0 == 0) {
        R.ctl->s.pivots = 0;
        R.ctl->s.block_cnt = 0;
    }
}

// Look-ahead of the blocked inversion: decides up to P.kblock Gauss-Jordan steps (columns done .. done+K-1)
// on aug as the last pass left it, brings each pivot column and pivot row up to date through the block's
// pending steps with the protocol's rule  v <- (row == l_s) ? p_s[col] : v - f_s[row] * p_s[col],
// and writes Fbuf / Pbuf / Lbuf for the pass.  One CTA; dynamic shared memory: column (colstride doubles)
// then the permutation (m ints).
__global__ void __launch_bounds__(LPX_REV_LA_THREADS) rev_lookahead_kernel(StreamParams P, int* perm_g) {
    extern __shared__ double sm_rv[];
    __shared__ unsigned long long s_key[32];
    __shared__ int s_idx[32];
    __shared__ int s_L[LPX_BLOCK_KMAX];
    __shared__ double s_pe[LPX_BLOCK_KMAX];
    __shared__ double s_fl[LPX_BLOCK_KMAX];
    constexpr int TH = LPX_REV_LA_THREADS, KM = LPX_BLOCK_KMAX;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int m = P.m, ld = P.ld, cs = P.colstride;
    double* colv = sm_rv;
    int* perm = reinterpret_cast<int*>(colv + cs);
    StreamCtl* ctl = P.ctl;
    const int status0 = ctl->status;
    const int done = ctl->pivots;
    if (tid == 0) ctl->block_cnt = 0;
    if (status0 != LPX_RUNNING) return;
    for (int i = tid; i < m; i += TH) perm[i] = perm_g[i];
    __syncthreads();

    const int steps = min(P.kblock, m - done);
    int cnt = 0, st = LPX_RUNNING;
    for (int k = 0; k < steps; k++) {
        const int col = done + cnt;
        // ---- column col, every physical row, brought up to date ----------------------------------------
        if (tid < cnt) s_pe[tid] = P.Pbuf[(size_t)tid * ld + col];
        __syncthreads();
        // all factor entries of a thread are loaded before the dependent multiply / subtract chain
        for (int base = 0; base < m; base += 2 * TH) {
            double c2[2], f[2][KM];
#pragma unroll
            for (int u = 0; u < 2; u++) {
                const int i = base + u * TH + tid;
                c2[u] = i < m ? P.T[(size_t)i * ld + col] : 0.0;
            }
#pragma unroll
            for (int s = 0; s < KM; s++)
#pragma unroll
                for (int u = 0; u < 2; u++) {
                    const int i = base + u * TH + tid;
                    f[u][s] = (s < cnt && i < m) ? P.Fbuf[(size_t)s * cs + i] : 0.0;
                }
#pragma unroll
            for (int s = 0; s < KM; s++)
                if (s < cnt) {
                    const double ps = s_pe[s];
                    const int ls = s_L[s];
#pragma unroll
                    for (int u = 0; u < 2; u++) {
                        const int i = base + u * TH + tid;
                        c2[u] = (i == ls) ? ps : __dsub_rn(c2[u], __dmul_rn(f[u][s], ps));
                    }
                }
#pragma unroll
            for (int u = 0; u < 2; u++) {
                const int i = base + u * TH + tid;
                if (i < m) colv[i] = c2[u];
            }
        }
        __syncthreads();
        // ---- pivot row: the FIRST largest |entry| over logical rows col .. m-1 (strict '>', Invert :428);
        // a NaN on the diagonal sticks, NaNs below it never win
        unsigned long long kl = ~0ULL;
        int il = INT_MAX;
        for (int r = col + tid; r < m; r += TH) {
            const double v = fabs(colv[perm[r]]);
            if (v == v) {
                const unsigned long long key = ~dkey(v);  // max |v|  ==  min of the complemented key
                if (key < kl) {
                    kl = key;
                    il = r;
                }
            }
        }
        const unsigned long long K1 = warp_min_u64(kl);
        const int i1 = __reduce_min_sync(0xffffffffu, kl == K1 ? il : INT_MAX);
        if (lane == 0) {
            s_key[warp] = K1;
            s_idx[warp] = i1;
        }
        __syncthreads();
        const unsigned long long k2 = lane < TH / 32 ? s_key[lane] : ~0ULL;
        const int i2 = lane < TH / 32 ? s_idx[lane] : INT_MAX;
        const unsigned long long K2 = warp_min_u64(k2);
        int prow = __reduce_min_sync(0xffffffffu, k2 == K2 ? i2 : INT_MAX);
        const double diag = colv[perm[col]];
        if (!(diag == diag) || prow == INT_MAX) prow = col;
        const int l = perm[prow];  // physical row of the pivot
        const double piv = colv[l];
        if (fabs(piv) < LPX_EPS) {  // "Singular basis encountered." (:433)
            st = LPX_S_SINGULAR;
            break;
        }
        __syncthreads();  // everybody has read perm, s_key and s_idx
        if (tid == 0) {
            perm[prow] = perm[col];
            perm[col] = l;
            s_L[cnt] = l;
            P.Lbuf[cnt] = l;
        }
        if (tid < cnt) s_fl[tid] = P.Fbuf[(size_t)tid * cs + l];
        __syncthreads();
        // ---- pivot row l: bring up to date, true division by the pivot ---------------------------------
        // ddiv_by_pivot is bit-identical to the division for every divisor but NaN (it returns a signed zero
        // for a zero numerator); a NaN pivot (one that stuck on the diagonal) divides for real.
        const bool nan_piv = !(piv == piv);
        double* pout = P.Pbuf + (size_t)cnt * ld;
        const double* Tl = P.T + (size_t)l * ld;
        for (int base = 0; base < ld; base += 2 * TH) {
            double r2[2], pp[2][KM];
#pragma unroll
            for (int u = 0; u < 2; u++) {
                const int j = base + u * TH + tid;
                r2[u] = j < ld ? Tl[j] : 0.0;
            }
#pragma unroll
            for (int s = 0; s < KM; s++)
#pragma unroll
                for (int u = 0; u < 2; u++) {
                    const int j = base + u * TH + tid;
                    pp[u][s] = (s < cnt && j < ld) ? P.Pbuf[(size_t)s * ld + j] : 0.0;
                }
#pragma unroll
            for (int s = 0; s < KM; s++)
                if (s < cnt) {
                    const double fs = s_fl[s];
                    const bool same = l == s_L[s];
#pragma unroll
                    for (int u = 0; u < 2; u++) r2[u] = same ? pp[u][s] : __dsub_rn(r2[u], __dmul_rn(fs, pp[u][s]));
                }
#pragma unroll
            for (int u = 0; u < 2; u++) {
                const int j = base + u * TH + tid;
                if (j < ld) pout[j] = nan_piv ? __ddiv_rn(r2[u], piv) : ddiv_by_pivot(r2[u], piv);
            }
        }
        double* fout = P.Fbuf + (size_t)cnt * cs;
        for (int i = tid; i < m; i += TH) fout[i] = colv[i];
        cnt++;
        __syncthreads();  // colv, s_pe and s_fl are rewritten by the next step
    }
    __syncthreads();
    for (int i = tid; i < m; i += TH) perm_g[i] = perm[i];
    if (tid == 0) {
        ctl->block_cnt = st == LPX_RUNNING ? cnt : 0;
        ctl->pivots = done + cnt;
        if (st != LPX_RUNNING) ctl->status = st;
    }
}

static size_t rev_lookahead_smem(int m) { return (size_t)((m + 15) & ~15) * 8 + (size_t)m * 4; }

// Binv (logical row i = physical row perm[i], columns m .. 2m-1 of aug) and its transpose, through 32 x 32 tiles.
__global__ void __launch_bounds__(256) rev_extract_kernel(RevParams R) {
    __shared__ double tile[32][33];
    if (!rev_running(R)) return;
    const int m = R.m;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int i0 = blockIdx.y * 32, j0 = blockIdx.x * 32;
    for (int q = ty; q < 32; q += 8) {
        const int i = i0 + q, j = j0 + tx;
        if (i < m && j < m) {
            const double v = R.aug[(size_t)R.perm[i] * R.ld + m + j];
            R.Binv[(size_t)i * m + j] = v;
            tile[q][tx] = v;
        }
    }
    __syncthreads();
    for (int q = ty; q < 32; q += 8) {
        const int j = j0 + q, i = i0 + tx;
        if (i < m && j < m) R.BinvT[(size_t)j * m + i] = tile[tx][q];
    }
}

// x_B = B^-1 b (row i summed left to right), c_B.
__global__ void __launch_bounds__(LPX_REV_TH) rev_xb_kernel(RevParams R) {
    if (!rev_running(R)) return;
    const int m = R.m, i = blockIdx.x * LPX_REV_TH + threadIdx.x;
    if (i >= m) return;
    double s = 0.0;
    for (int j = 0; j < m; j++) s = __dadd_rn(s, __dmul_rn(R.BinvT[(size_t)j * m + i], R.b[j]));
    R.xB[i] = s;
    R.cB[i] = R.cf[R.Bidx[i]];
}

// History record ctl->iters (BuildIterationBlock :62, :134), the layout of lpx_revised.cu's kernel; z = c_B . x_B.
__global__ void __launch_bounds__(256) rev_record_kernel(RevParams R) {
    if (!rev_running(R)) return;
    const int k = R.ctl->iters;
    if (k >= R.history_cap) return;
    const int m = R.m, n = R.n;
    const bool pr = k > 0;  // record 0 (the initial basis) has no pricing
    const size_t hs = (size_t)m * m + m + 1 + n + m + 1 + m + n + 1;
    double* h = R.history + (size_t)k * hs;
    const size_t t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
    for (size_t q = t0; q < (size_t)m * m; q += stride) h[q] = R.Binv[q];
    double* p = h + (size_t)m * m;
    for (size_t i = t0; i < (size_t)m; i += stride) p[i] = R.xB[i];
    p += m;
    if (t0 == 0) {
        double s = 0.0;
        for (int i = 0; i < m; i++) s = __dadd_rn(s, __dmul_rn(R.cB[i], R.xB[i]));
        p[0] = s;
    }
    p += 1;
    for (size_t j = t0; j < (size_t)n; j += stride) p[j] = pr ? R.rN[j] : 0.0;
    p += n;
    for (size_t i = t0; i < (size_t)m; i += stride) p[i] = pr ? R.d[i] : 0.0;
    p += m;
    if (t0 == 0) p[0] = pr ? R.ctl->theta : 0.0;
    p += 1;
    for (size_t i = t0; i < (size_t)m; i += stride) p[i] = (double)R.Bidx[i];
    p += m;
    for (size_t j = t0; j < (size_t)n; j += stride) p[j] = (double)R.Nidx[j];
    p += n;
    if (t0 == 0) p[0] = pr ? (double)R.ctl->enter : -1.0;
}

// pi = c_B^T B^-1 (column j summed top to bottom).  First kernel of an iteration: the iteration limit
// ("throw" after MaxIterations full iterations, :144) is tested here, before anything changes.
__global__ void __launch_bounds__(LPX_REV_TH) rev_pi_kernel(RevParams R) {
    if (!rev_running(R)) return;
    if (R.ctl->iters >= R.max_iter) {  // every CTA sees the same count and returns
        if (blockIdx.x == 0 && threadIdx.x == 0) R.ctl->s.status = LPX_S_ITER_LIMIT;
        return;
    }
    const int m = R.m, j = blockIdx.x * LPX_REV_TH + threadIdx.x;
    if (j >= m) return;
    double s = 0.0;
    for (int i = 0; i < m; i++) s = __dadd_rn(s, __dmul_rn(R.cB[i], R.Binv[(size_t)i * m + j]));
    R.pi[j] = s;
}

// r_N[k] = c[Nidx[k]] - pi . A_{Nidx[k]}, and this CTA's most negative entry below -1e-9 (lowest position).
__global__ void __launch_bounds__(LPX_REV_TH) rev_rn_kernel(RevParams R) {
    __shared__ ArgMin red[34];
    if (!rev_running(R)) return;
    const int m = R.m, n = R.n, base = blockIdx.x * LPX_REV_TH, k = base + threadIdx.x;
    double v = 0.0;
    if (k < n) {
        const int col = R.Nidx[k];
        double s = 0.0;
        for (int i = 0; i < m; i++) s = __dadd_rn(s, __dmul_rn(R.pi[i], R.Af[(size_t)i * R.ntot + col]));
        v = __dsub_rn(R.cf[col], s);
        R.rN[k] = v;
    }
    const int cnt = min(LPX_REV_TH, n - base);
    const int w = block_argmin_core<LPX_REV_TH>(cnt, -LPX_EPS, red, [&](int) { return v; });
    if (threadIdx.x == 0) {
        ArgMin a;
        a.v = w < 0 ? __longlong_as_double(0x7ff0000000000000LL) : R.rN[base + w];
        a.i = w < 0 ? INT_MAX : base + w;
        R.part[blockIdx.x] = a;
    }
}

// Entering position: the CTA partials in one CTA (smaller value, then lower position); none: OPTIMAL.
__global__ void __launch_bounds__(1024) rev_enter_kernel(RevParams R, int nparts) {
    __shared__ ArgMin red[32];
    if (!rev_running(R)) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    ArgMin a;
    a.v = __longlong_as_double(0x7ff0000000000000LL);
    a.i = INT_MAX;
    for (int q = threadIdx.x; q < nparts; q += 1024) a = argmin_pick(a, R.part[q]);
    a = warp_argmin(a);
    if (lane == 0) red[warp] = a;
    __syncthreads();
    if (warp == 0) {
        a = red[lane];
        a = warp_argmin(a);
        if (lane == 0) {
            if (a.i == INT_MAX) {
                R.ctl->s.status = LPX_OPTIMAL;
            } else {
                R.ctl->pos = a.i;
                R.ctl->enter = R.Nidx[a.i];
            }
        }
    }
}

// d = B^-1 a_entering (row i summed left to right); theta_i = x_B[i] / d_i over d_i > 1e-9, else NaN.
__global__ void __launch_bounds__(LPX_REV_TH) rev_dir_kernel(RevParams R) {
    if (!rev_running(R)) return;
    const int m = R.m, i = blockIdx.x * LPX_REV_TH + threadIdx.x;
    if (i >= m) return;
    const int e = R.ctl->enter;
    double s = 0.0;
    for (int j = 0; j < m; j++) s = __dadd_rn(s, __dmul_rn(R.BinvT[(size_t)j * m + i], R.Af[(size_t)j * R.ntot + e]));
    R.d[i] = s;
    R.ratio[i] = s > LPX_EPS ? __ddiv_rn(R.xB[i], s) : __longlong_as_double(0x7ff8000000000000LL);
}

// Leaving row (the sequential margin scan, margin 1e-12, :104); none: UNBOUNDED.  Then Bidx[row] = entering,
// Nidx.RemoveAt(pos) + Add(leaving) as an in-place shift, the pivot record and the iteration count.
__global__ void __launch_bounds__(1024) rev_leave_kernel(RevParams R) {
    __shared__ int s_row;
    if (!rev_running(R)) return;
    const int tid = threadIdx.x, m = R.m, n = R.n;
    if (tid < 32) {
        const int l = warp_margin_scan_cert(m, LPX_MARGIN_DUAL, [&](int i, double& r) {
            r = R.ratio[i];
            return r == r;
        });
        if (tid == 0) s_row = l;
    }
    __syncthreads();
    const int row = s_row;
    RevCtl* ctl = R.ctl;
    if (row < 0) {
        if (tid == 0) ctl->s.status = LPX_UNBOUNDED;
        return;
    }
    const int pos = ctl->pos, entering = ctl->enter, it = ctl->iters;
    const int leaving = R.Bidx[row];
    __syncthreads();  // everybody has read Bidx[row] and the control block
    if (tid == 0) {
        const double th = R.ratio[row];
        R.Bidx[row] = entering;
        ctl->theta = th;
        if (R.pivots && it < R.pivots_cap) {
            R.pivots[2 * it] = entering;
            R.pivots[2 * it + 1] = row;
            R.theta[it] = th;
        }
        ctl->iters = it + 1;
    }
    // ascending 1024-wide windows: a window reads one entry past its end, which the next window writes later
    for (int base = pos; base < n; base += 1024) {
        const int k = base + tid;
        int v = 0;
        if (k < n) v = k + 1 < n ? R.Nidx[k + 1] : leaving;
        __syncthreads();
        if (k < n) R.Nidx[k] = v;
        __syncthreads();
    }
}

// ---- host driver ------------------------------------------------------------------------------------------

struct RevStream {
    RevParams R;
    StreamParams P;  // the inversion as a "tableau" of m rows for the look-ahead and the pass kernels
    int variant = 0, rpc = 0;
    dim3 grid_pass;
    int grid_fill = 0;  // CTAs of the grid-stride kernels
};

static void rev_enqueue_refresh(const RevStream& S, cudaStream_t st) {
    const RevParams& R = S.R;
    rev_build_kernel<<<S.grid_fill, 256, 0, st>>>(R);
    count_launch();
    const int K = S.P.kblock, nb = (R.m + K - 1) / K;
    const BlockPassFn pass = block_pass_fn(S.variant, K);
    const size_t pass_smem = block_pass_smem(S.variant, K, S.rpc);
    for (int q = 0; q < nb; q++) {
        rev_lookahead_kernel<<<1, LPX_REV_LA_THREADS, rev_lookahead_smem(R.m), st>>>(S.P, R.perm);
        pass<<<S.grid_pass, 256, pass_smem, st>>>(S.P, S.rpc);
        count_launch(2);
    }
    const int tiles = (R.m + 31) / 32;
    rev_extract_kernel<<<dim3(tiles, tiles), 256, 0, st>>>(R);
    rev_xb_kernel<<<(R.m + LPX_REV_TH - 1) / LPX_REV_TH, LPX_REV_TH, 0, st>>>(R);
    count_launch(2);
    if (R.history) {
        rev_record_kernel<<<S.grid_fill, 256, 0, st>>>(R);
        count_launch();
    }
}

static void rev_enqueue_iteration(const RevStream& S, cudaStream_t st) {
    const RevParams& R = S.R;
    const int gm = (R.m + LPX_REV_TH - 1) / LPX_REV_TH, gn = (R.n + LPX_REV_TH - 1) / LPX_REV_TH;
    rev_pi_kernel<<<gm, LPX_REV_TH, 0, st>>>(R);
    rev_rn_kernel<<<gn, LPX_REV_TH, 0, st>>>(R);
    rev_enter_kernel<<<1, 1024, 0, st>>>(R, gn);
    rev_dir_kernel<<<gm, LPX_REV_TH, 0, st>>>(R);
    rev_leave_kernel<<<1, 1024, 0, st>>>(R);
    count_launch(5);
    rev_enqueue_refresh(S, st);
}

int revised_stream_solve(int m, int n, int sense, const double* A, const double* b, const double* c,
                         const lpx_options& o, int* status, int* n_iters, int* pivots, double* theta, int pivots_cap,
                         int* basis, int* nonbasic, double* xB, double* Binv, double* x, double* history,
                         int history_cap) {
    if (rev_lookahead_smem(m) + 8192 > (size_t)max_smem_optin()) {
        set_error("lpx_revised_solve: m too large for the inversion look-ahead's shared memory");
        return LPX_E_CAPACITY;
    }
    const int K = o.stream_block > 0 ? std::min(o.stream_block, LPX_BLOCK_KMAX) : LPX_REV_DEFAULT_K;
    const int ntot = n + m, ld = (2 * m + 15) & ~15, cs = (m + 15) & ~15;
    const int gn = (n + LPX_REV_TH - 1) / LPX_REV_TH;
    const size_t hs = (size_t)m * m + m + 1 + n + m + 1 + m + n + 1;
    // one allocation for the vectors (each piece starts on a 128-byte boundary), one for the integers
    size_t nd = 0;
    auto take = [&](size_t count) {
        const size_t at = nd;
        nd += (count + 15) & ~(size_t)15;
        return at;
    };
    const size_t o_binvt = take((size_t)m * m), o_cf = take(ntot), o_xb = take(m), o_cb = take(m), o_pi = take(m),
                 o_d = take(m), o_ratio = take(m), o_rn = take(n), o_f = take((size_t)LPX_BLOCK_KMAX * cs),
                 o_p = take((size_t)LPX_BLOCK_KMAX * ld), o_part = take((size_t)gn * 2),
                 o_ctl = take((sizeof(RevCtl) + 7) / 8);
    double* dA = ws_dev_as<double>(WS_A, (size_t)m * n);
    double* db = ws_dev_as<double>(WS_B, m);
    double* dc = ws_dev_as<double>(WS_C, n);
    double* dAf = ws_dev_as<double>(WS_TABLEAU, (size_t)m * ntot);
    double* daug = ws_dev_as<double>(WS_SCRATCH, (size_t)m * ld);
    double* dBinv = ws_dev_as<double>(WS_MISC0, (size_t)m * m);
    double* dvec = ws_dev_as<double>(WS_MISC2, nd);
    int* dint = ws_dev_as<int>(WS_BASIS, (size_t)3 * m + n + LPX_BLOCK_KMAX);
    int* dpiv = ws_dev_as<int>(WS_PIVOTS, (size_t)std::max(pivots_cap, 1) * 2);
    double* dtheta = ws_dev_as<double>(WS_MISC1, (size_t)std::max(pivots_cap, 1));
    if (!dA || !db || !dc || !dAf || !daug || !dBinv || !dvec || !dint || !dpiv || !dtheta) {
        cudaGetLastError();
        set_error("lpx_revised_solve: no device memory for the work buffers of m = " + std::to_string(m) + ", n = " +
                  std::to_string(n) + " ([B | I] alone is " + std::to_string((size_t)m * ld * 8) + " bytes)");
        return LPX_E_CAPACITY;
    }
    double* dH = nullptr;
    if (history_cap) {
        dH = ws_dev_as<double>(WS_HISTORY, hs * (size_t)history_cap);
        if (!dH) {
            cudaGetLastError();
            set_error("lpx_revised_solve: no device memory for the history (" + std::to_string(history_cap) +
                      " records of " + std::to_string(hs * 8) + " bytes)");
            return LPX_E_CAPACITY;
        }
    }
    cudaStream_t st = rt().stream;
    LPX_CUDA(cudaMemcpyAsync(dA, A, (size_t)m * n * 8, cudaMemcpyHostToDevice, st));
    LPX_CUDA(cudaMemcpyAsync(db, b, (size_t)m * 8, cudaMemcpyHostToDevice, st));
    LPX_CUDA(cudaMemcpyAsync(dc, c, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    // Fbuf / Pbuf are read in whole 8-row tiles and full rows by the pass: pads must hold finite values
    LPX_CUDA(cudaMemsetAsync(dvec + o_f, 0, (size_t)LPX_BLOCK_KMAX * (cs + ld) * 8, st));

    RevStream S;
    RevParams& R = S.R;
    std::memset(&R, 0, sizeof R);
    R.m = m;
    R.n = n;
    R.ntot = ntot;
    R.sense = sense;
    R.max_iter = o.max_iterations;
    R.ld = ld;
    R.A = dA;
    R.b = db;
    R.c = dc;
    R.Af = dAf;
    R.cf = dvec + o_cf;
    R.aug = daug;
    R.Binv = dBinv;
    R.BinvT = dvec + o_binvt;
    R.xB = dvec + o_xb;
    R.cB = dvec + o_cb;
    R.pi = dvec + o_pi;
    R.d = dvec + o_d;
    R.ratio = dvec + o_ratio;
    R.rN = dvec + o_rn;
    R.Bidx = dint;
    R.Nidx = dint + m;
    R.perm = dint + m + n;
    R.part = reinterpret_cast<ArgMin*>(dvec + o_part);
    R.ctl = reinterpret_cast<RevCtl*>(dvec + o_ctl);
    R.pivots = pivots_cap ? dpiv : nullptr;
    R.theta = dtheta;
    R.pivots_cap = pivots_cap;
    R.history = dH;
    R.history_cap = history_cap;

    StreamParams& P = S.P;
    std::memset(&P, 0, sizeof P);
    P.T = daug;
    P.ld = ld;
    P.rows = m;
    P.m = m;
    P.n = m;
    P.width = 2 * m + 1;
    P.colstride = cs;
    P.ctl = &R.ctl->s;
    P.Fbuf = dvec + o_f;
    P.Pbuf = dvec + o_p;
    P.Lbuf = dint + 2 * m + n;
    P.kblock = K;
    S.variant = o.stream_pass_variant;
    size_block_pass(P, S.variant, &S.rpc, &S.grid_pass);
    LPX_CUDA(cudaFuncSetAttribute(rev_lookahead_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)rev_lookahead_smem(m)));
    S.grid_fill = sm_count() * 4;

    rev_setup_kernel<<<S.grid_fill, 256, 0, st>>>(R);
    count_launch();
    rev_enqueue_refresh(S, st);
    LPX_CUDA(cudaGetLastError());
    // chunks of iterations between host synchronisations, doubling up to ~1024 launches per chunk: the launches of
    // a chunk after the status has left RUNNING return at once, so a solve ends with fewer than that many no-ops
    const int per_iter = 8 + 2 * ((m + K - 1) / K);
    const int chunk_max = std::max(1, 1024 / per_iter);
    int chunk = 1;
    RevCtl h;
    while (true) {
        LPX_CUDA(cudaMemcpyAsync(&h, R.ctl, sizeof h, cudaMemcpyDeviceToHost, st));
        LPX_CUDA(cudaStreamSynchronize(st));
        if (h.s.status != LPX_RUNNING) break;
        // iteration max_iter + 1 only raises the limit
        const int todo = (int)std::min<long long>(chunk, std::max<long long>(1, (long long)o.max_iterations - h.iters + 1));
        for (int q = 0; q < todo; q++) rev_enqueue_iteration(S, st);
        LPX_CUDA(cudaGetLastError());
        chunk = std::min(2 * chunk, chunk_max);
    }
    *status = h.s.status;
    if (n_iters) *n_iters = h.iters;
    if (h.s.status == LPX_S_SINGULAR) {
        // Invert threw inside iteration n_iters: the records of the iterations before it are returned
        if (history && history_cap && h.iters > 0) {
            const int nh = std::min(h.iters, history_cap);
            LPX_CUDA(cudaMemcpyAsync(history, dH, hs * nh * 8, cudaMemcpyDeviceToHost, st));
            LPX_CUDA(cudaStreamSynchronize(st));
        }
        return LPX_OK;
    }
    std::vector<int> hb(m);
    std::vector<double> hx(m);
    const int np = std::min(h.iters, pivots_cap);
    if (np > 0) {
        LPX_CUDA(cudaMemcpyAsync(pivots, dpiv, (size_t)np * 8, cudaMemcpyDeviceToHost, st));
        if (theta) LPX_CUDA(cudaMemcpyAsync(theta, dtheta, (size_t)np * 8, cudaMemcpyDeviceToHost, st));
    }
    LPX_CUDA(cudaMemcpyAsync(hb.data(), R.Bidx, (size_t)m * 4, cudaMemcpyDeviceToHost, st));
    LPX_CUDA(cudaMemcpyAsync(hx.data(), R.xB, (size_t)m * 8, cudaMemcpyDeviceToHost, st));
    if (nonbasic) LPX_CUDA(cudaMemcpyAsync(nonbasic, R.Nidx, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    if (Binv) LPX_CUDA(cudaMemcpyAsync(Binv, dBinv, (size_t)m * m * 8, cudaMemcpyDeviceToHost, st));
    if (history && history_cap) {
        const int nh = std::min(h.iters + 1, history_cap);
        LPX_CUDA(cudaMemcpyAsync(history, dH, hs * nh * 8, cudaMemcpyDeviceToHost, st));
    }
    LPX_CUDA(cudaStreamSynchronize(st));
    if (basis) std::memcpy(basis, hb.data(), (size_t)m * 4);
    if (xB) std::memcpy(xB, hx.data(), (size_t)m * 8);
    if (x) {
        std::fill(x, x + n, 0.0);
        for (int i = 0; i < m; i++)
            if (hb[i] < n) x[hb[i]] = hx[i];
    }
    return LPX_OK;
}

}  // namespace lpx
