// lpx_revised.cu — Revised Primal Simplex (price-out), one CTA per LP.
//
// Replaces R/Models/RevisedPrimalSimplex.cs:17-145.  The reference recomputes the basis inverse from
// scratch every iteration by Gauss-Jordan with partial pivoting (:121, :409-456) and forms every
// product as a left-to-right sum (:331-394), so the GPU program keeps exactly that operation order:
//   * Invert: the m x 2m augmented matrix [B | I] lives in global memory (L2 resident); per column the
//     pivot search is a block arg-max with the FIRST largest |entry| (the strict '>' of :428), then a
//     row swap, a true division of the pivot row, and an unfused multiply-subtract of every other row —
//     the same rank-1 update as a tableau pivot, all elements in parallel;
//   * every dot product (pi = c_B B^-1, r_N, d = B^-1 a_e, x_B = B^-1 b, z) is summed by ONE thread
//     in index order — different outputs in parallel, never a tree reduction;
//   * entering = most negative reduced cost below -1e-9, lowest position in the nonbasic LIST;
//     leaving = the sequential margin scan with margin 1e-12 (:104), certified shortcut as elsewhere.
// Standardize (:148-186) negates C for a MAX objective; the nonbasic list is kept in the reference's
// order (RemoveAt(enteringPos), Add(leaving)).
#include <cstring>

#include "lpx_cta.cuh"
#include "lpx_runtime.hpp"
#include "lpx_stream.hpp"

namespace lpx {

// AUTO's crossover: the largest m that stays on the one-CTA kernel.  Measured on one B200 (1000 W,
// profiles/r08_revised_stream.json, DESIGN.md §4.11): at m = 64 the two paths are within 4 % per iteration (square
// 0.304 vs 0.316 ms, wide 0.322 vs 0.315 ms); at m = 96 the whole GPU is 2.0-3.2x faster.
#define LPX_REV_CTA_MAX_M 64

struct RevBatch {
    const double* A;  // m x n
    const double* b;
    const double* c;
    int m, n, sense, max_iter;
    // global scratch
    double* Af;    // m x (n + m)
    double* aug;   // m x 2m
    double* Binv;  // m x m (output too)
    // outputs
    int* status;   // [0] status, [1] iterations
    int* pivots;   // 2 per iteration: entering column, leaving row
    double* theta; // per iteration
    int pivots_cap;
    int* basis;     // m
    int* nonbasic;  // n
    double* xB;     // m
    double* x;      // n
    double* history;  // history_cap records of rev_history_stride(m, n) doubles
    int history_cap;
};

__host__ __device__ inline size_t rev_history_stride(int m, int n) {
    return (size_t)m * m + m + 1 + n + m + 1 + m + n + 1;
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS) revised_simplex_kernel(const RevBatch B) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int m = B.m, n = B.n, ntot = n + m, w2 = 2 * m;
    double* cf = reinterpret_cast<double*>(smem_raw);  // ntot
    double* bv = cf + ntot;     // m
    double* xB = bv + m;        // m
    double* cB = xB + m;        // m
    double* piT = cB + m;       // m
    double* dv = piT + m;       // m
    double* ratio = dv + m;     // m
    double* fcol = ratio + m;   // m
    double* rN = fcol + m;      // n
    int* Bidx = reinterpret_cast<int*>(rN + n);  // m
    int* Nidx = Bidx + m;                        // n
    __shared__ ArgMin red[34];
    __shared__ int s_ctl[4];
    __shared__ double s_z, s_theta;
    double* Af = B.Af;
    double* aug = B.aug;
    double* Binv = B.Binv;

    // ---- A | I, c (negated for MAX: Standardize :153-154), b; slack basis -------------------------
    for (int k = tid; k < m * ntot; k += THREADS) {
        const int i = k / ntot, j = k - i * ntot;
        Af[k] = j < n ? B.A[(size_t)i * n + j] : (j == n + i ? 1.0 : 0.0);
    }
    for (int j = tid; j < ntot; j += THREADS) {
        double v = 0.0;
        if (j < n) v = B.sense == 0 ? dneg(B.c[j]) : B.c[j];
        cf[j] = v;
    }
    for (int i = tid; i < m; i += THREADS) {
        bv[i] = B.b[i];
        Bidx[i] = n + i;
    }
    for (int j = tid; j < n; j += THREADS) Nidx[j] = j;
    if (tid == 0) s_ctl[0] = LPX_RUNNING;
    __syncthreads();

    // Invert(GetSubmatrix(A, Bidx)) -> Binv; then x_B = B^-1 b, c_B, z.  Returns false on a singular basis.
    auto refresh_basis = [&]() -> bool {
        for (int k = tid; k < m * w2; k += THREADS) {
            const int i = k / w2, j = k - i * w2;
            aug[k] = j < m ? Af[(size_t)i * ntot + Bidx[j]] : (j == m + i ? 1.0 : 0.0);
        }
        __syncthreads();
        for (int col = 0; col < m; col++) {
            // pivot row: first largest |aug[r][col]|, r >= col; a NaN at r == col sticks, NaNs below never win
            unsigned long long kl = ~0ULL;
            int il = INT_MAX;
            for (int r = col + tid; r < m; r += THREADS) {
                const double v = fabs(aug[(size_t)r * w2 + col]);
                if (v == v) {
                    const unsigned long long k = ~dkey(v);  // max |v|  ==  min of the complemented key
                    if (k < kl) {
                        kl = k;
                        il = r;
                    }
                }
            }
            const unsigned long long K = warp_min_u64(kl);
            const int iw = __reduce_min_sync(0xffffffffu, kl == K ? il : INT_MAX);
            if (lane == 0) {
                red[warp].v = __longlong_as_double((long long)K);
                red[warp].i = iw;
            }
            __syncthreads();
            unsigned long long k2 = ~0ULL;
            int i2 = INT_MAX;
            if (lane < THREADS / 32) {
                k2 = (unsigned long long)__double_as_longlong(red[lane].v);
                i2 = red[lane].i;
            }
            const unsigned long long K2 = warp_min_u64(k2);
            int prow = __reduce_min_sync(0xffffffffu, k2 == K2 ? i2 : INT_MAX);
            const double diag = aug[(size_t)col * w2 + col];
            if (!(diag == diag) || prow == INT_MAX) prow = col;
            const double pabs = fabs(aug[(size_t)prow * w2 + col]);
            __syncthreads();  // red is free; everybody has read the column
            if (pabs < LPX_EPS) return false;  // "Singular basis encountered." (:433)
            if (prow != col) {
                for (int j = tid; j < w2; j += THREADS) {
                    const double t0 = aug[(size_t)col * w2 + j];
                    aug[(size_t)col * w2 + j] = aug[(size_t)prow * w2 + j];
                    aug[(size_t)prow * w2 + j] = t0;
                }
                __syncthreads();
            }
            const double piv = aug[(size_t)col * w2 + col];
            for (int r = tid; r < m; r += THREADS) fcol[r] = aug[(size_t)r * w2 + col];
            __syncthreads();
            for (int j = tid; j < w2; j += THREADS) aug[(size_t)col * w2 + j] = __ddiv_rn(aug[(size_t)col * w2 + j], piv);
            __syncthreads();
            for (int k = tid; k < m * w2; k += THREADS) {
                const int r = k / w2, j = k - r * w2;
                if (r != col) aug[k] = __dsub_rn(aug[k], __dmul_rn(fcol[r], aug[(size_t)col * w2 + j]));
            }
            __syncthreads();
        }
        for (int k = tid; k < m * m; k += THREADS) {
            const int i = k / m, j = k - i * m;
            Binv[k] = aug[(size_t)i * w2 + m + j];
        }
        __syncthreads();
        for (int i = tid; i < m; i += THREADS) {
            double s = 0.0;
            for (int j = 0; j < m; j++) s = __dadd_rn(s, __dmul_rn(Binv[(size_t)i * m + j], bv[j]));
            xB[i] = s;
            cB[i] = cf[Bidx[i]];
        }
        __syncthreads();
        if (tid == 0) {
            double s = 0.0;
            for (int i = 0; i < m; i++) s = __dadd_rn(s, __dmul_rn(cB[i], xB[i]));
            s_z = s;
        }
        __syncthreads();
        return true;
    };
    const size_t hs = rev_history_stride(m, n);
    auto record = [&](int k, int entering, bool with_pricing) {
        if (!B.history || k >= B.history_cap) return;
        double* h = B.history + (size_t)k * hs;
        for (int q = tid; q < m * m; q += THREADS) h[q] = Binv[q];
        double* p = h + (size_t)m * m;
        for (int i = tid; i < m; i += THREADS) p[i] = xB[i];
        p += m;
        if (tid == 0) p[0] = s_z;
        p += 1;
        for (int j = tid; j < n; j += THREADS) p[j] = with_pricing ? rN[j] : 0.0;
        p += n;
        for (int i = tid; i < m; i += THREADS) p[i] = with_pricing ? dv[i] : 0.0;
        p += m;
        if (tid == 0) p[0] = with_pricing ? s_theta : 0.0;
        p += 1;
        for (int i = tid; i < m; i += THREADS) p[i] = (double)Bidx[i];
        p += m;
        for (int j = tid; j < n; j += THREADS) p[j] = (double)Nidx[j];
        p += n;
        if (tid == 0) p[0] = (double)entering;
    };

    int status = LPX_RUNNING, iters = 0;
    if (!refresh_basis()) status = LPX_S_SINGULAR;
    if (status == LPX_RUNNING) {
        record(0, -1, false);
        while (true) {
            if (iters >= B.max_iter) {
                status = LPX_S_ITER_LIMIT;  // thrown after MaxIterations full iterations (:144)
                break;
            }
            // price out: pi = c_B^T B^-1, r_N = c_N - pi N
            for (int j = tid; j < m; j += THREADS) {
                double s = 0.0;
                for (int i = 0; i < m; i++) s = __dadd_rn(s, __dmul_rn(cB[i], Binv[(size_t)i * m + j]));
                piT[j] = s;
            }
            __syncthreads();
            for (int k = tid; k < n; k += THREADS) {
                const int col = Nidx[k];
                double s = 0.0;
                for (int i = 0; i < m; i++) s = __dadd_rn(s, __dmul_rn(piT[i], Af[(size_t)i * ntot + col]));
                rN[k] = __dsub_rn(cf[col], s);
            }
            __syncthreads();
            const int pos = block_argmin_below<THREADS>(rN, n, -LPX_EPS, red);
            if (pos < 0) {
                status = LPX_OPTIMAL;
                break;
            }
            const int entering = Nidx[pos];
            // d = B^-1 a_entering; theta_i = x_B[i] / d_i over d_i > 1e-9
            for (int i = tid; i < m; i += THREADS) {
                double s = 0.0;
                for (int j = 0; j < m; j++) s = __dadd_rn(s, __dmul_rn(Binv[(size_t)i * m + j], Af[(size_t)j * ntot + entering]));
                dv[i] = s;
                ratio[i] = s > LPX_EPS ? __ddiv_rn(xB[i], s) : __longlong_as_double(0x7ff8000000000000LL);
            }
            __syncthreads();
            if (warp == 0) {
                const int l = warp_margin_scan_cert(m, LPX_MARGIN_DUAL, [&](int i, double& r) {
                    r = ratio[i];
                    return r == r;
                });
                if (lane == 0) {
                    s_ctl[2] = l;
                    if (l >= 0) s_theta = ratio[l];
                }
            }
            __syncthreads();
            const int row = s_ctl[2];
            if (row < 0) {
                status = LPX_UNBOUNDED;
                break;
            }
            if (tid == 0) {
                const int leaving = Bidx[row];
                Bidx[row] = entering;
                for (int k = pos; k + 1 < n; k++) Nidx[k] = Nidx[k + 1];  // RemoveAt(enteringPos); Add(leaving)
                Nidx[n - 1] = leaving;
                if (B.pivots && iters < B.pivots_cap) {
                    B.pivots[2 * iters] = entering;
                    B.pivots[2 * iters + 1] = row;
                    if (B.theta) B.theta[iters] = s_theta;
                }
            }
            __syncthreads();
            iters++;
            if (!refresh_basis()) {
                status = LPX_S_SINGULAR;
                break;
            }
            record(iters, entering, true);
        }
    }
    __syncthreads();
    if (status != LPX_S_SINGULAR) {
        for (int i = tid; i < m; i += THREADS) {
            if (B.basis) B.basis[i] = Bidx[i];
            if (B.xB) B.xB[i] = xB[i];
        }
        for (int j = tid; j < n; j += THREADS) {
            if (B.nonbasic) B.nonbasic[j] = Nidx[j];
            if (B.x) B.x[j] = 0.0;
        }
        __syncthreads();
        if (B.x)
            for (int i = tid; i < m; i += THREADS)
                if (Bidx[i] < n) B.x[Bidx[i]] = xB[i];
    }
    if (tid == 0) {
        B.status[0] = status;
        B.status[1] = iters;
    }
}

}  // namespace lpx

using namespace lpx;

extern "C" {

size_t lpx_revised_history_stride(int m, int n) { return rev_history_stride(m, n); }

int lpx_revised_solve(int m, int n, int sense, const double* A, const int* rel, const double* b, const double* c,
                      const lpx_options* opt, int* status, int* n_iters, int* pivots, double* theta, int pivots_cap,
                      int* basis, int* nonbasic, double* xB, double* Binv, double* x, double* history,
                      int history_cap) {
    if (m < 1 || n < 1 || !A || !b || !c || !status || (sense != 0 && sense != 1)) {
        set_error("lpx_revised_solve: bad arguments");
        return LPX_E_BAD_ARGS;
    }
    int rc = ensure_device();
    if (rc != LPX_OK) return rc;
    Runtime& r = rt();
    std::lock_guard<std::recursive_mutex> lk(r.mu);
    if (n_iters) *n_iters = 0;
    // the reference's up-front check (:19-21): only <= rows with b >= -1e-9
    for (int i = 0; i < m; i++)
        if ((rel && rel[i] != 0) || !(b[i] >= -1e-9)) {
            *status = LPX_S_REV_UNSUPPORTED;
            return LPX_OK;
        }
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    if (pivots_cap < 0 || !pivots) pivots_cap = 0;
    if (!history) history_cap = 0;
    const size_t smem = ((size_t)(n + m) + 7 * (size_t)m + n) * 8 + ((size_t)m + n) * 4 + 16;
    const bool fits = smem <= (size_t)max_smem_optin();
    // STREAM forces the whole-GPU path, CTA_GLOBAL this kernel; anything else is AUTO: this kernel while its
    // work vectors fit and m is at most LPX_REV_CTA_MAX_M (measured crossover, above)
    const bool stream = o.kernel == LPX_KERNEL_STREAM || (o.kernel != LPX_KERNEL_CTA_GLOBAL && (!fits || m > LPX_REV_CTA_MAX_M));
    if (stream)
        return revised_stream_solve(m, n, sense, A, b, c, o, status, n_iters, pivots, theta, pivots_cap, basis, nonbasic,
                                    xB, Binv, x, history, history_cap);
    if (!fits) {
        set_error("lpx_revised_solve: m + n too large for the shared-memory work vectors");
        return LPX_E_CAPACITY;
    }
    const size_t hs = rev_history_stride(m, n);
    double* dA = ws_dev_as<double>(WS_A, (size_t)m * n);
    double* db = ws_dev_as<double>(WS_B, m);
    double* dc = ws_dev_as<double>(WS_C, n);
    double* dAf = ws_dev_as<double>(WS_TABLEAU, (size_t)m * (n + m));
    double* daug = ws_dev_as<double>(WS_SCRATCH, (size_t)m * 2 * m);
    double* dBinv = ws_dev_as<double>(WS_MISC0, (size_t)m * m + 16);
    int* dstat = ws_dev_as<int>(WS_STATUS, 4);
    int* dpiv = ws_dev_as<int>(WS_PIVOTS, (size_t)std::max(pivots_cap, 1) * 2);
    double* dtheta = ws_dev_as<double>(WS_MISC1, (size_t)std::max(pivots_cap, 1));
    int* dbasis = ws_dev_as<int>(WS_BASIS, (size_t)m + n);
    double* dx = ws_dev_as<double>(WS_X, (size_t)n + m);
    double* dH = history_cap ? ws_dev_as<double>(WS_HISTORY, hs * history_cap) : nullptr;
    if (!dA || !db || !dc || !dAf || !daug || !dBinv || !dstat || !dpiv || !dtheta || !dbasis || !dx || (history_cap && !dH))
        return LPX_E_CUDA;
    cudaStream_t s = r.stream;
    LPX_CUDA(cudaMemcpyAsync(dA, A, (size_t)m * n * 8, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemcpyAsync(db, b, (size_t)m * 8, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemcpyAsync(dc, c, (size_t)n * 8, cudaMemcpyHostToDevice, s));
    RevBatch B;
    std::memset(&B, 0, sizeof B);
    B.A = dA;
    B.b = db;
    B.c = dc;
    B.m = m;
    B.n = n;
    B.sense = sense;
    B.max_iter = o.max_iterations;
    B.Af = dAf;
    B.aug = daug;
    B.Binv = dBinv;
    B.status = dstat;
    B.pivots = pivots_cap ? dpiv : nullptr;
    B.theta = pivots_cap ? dtheta : nullptr;
    B.pivots_cap = pivots_cap;
    B.basis = dbasis;
    B.nonbasic = dbasis + m;
    B.xB = dx + n;
    B.x = dx;
    B.history = dH;
    B.history_cap = history_cap;
    auto kfn = revised_simplex_kernel<256>;
    LPX_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kfn<<<1, 256, smem, s>>>(B);
    LPX_CUDA(cudaGetLastError());
    count_launch();
    int hstat[2] = {0, 0};
    LPX_CUDA(cudaMemcpyAsync(hstat, dstat, sizeof hstat, cudaMemcpyDeviceToHost, s));
    LPX_CUDA(cudaStreamSynchronize(s));
    *status = hstat[0];
    if (n_iters) *n_iters = hstat[1];
    if (hstat[0] == LPX_S_SINGULAR) {
        // Invert threw inside iteration n_iters (or on the initial basis when n_iters == 0): the blocks of
        // the iterations before it had already been printed, so their records are returned
        if (history && history_cap && hstat[1] > 0) {
            const int nh = std::min(hstat[1], history_cap);
            LPX_CUDA(cudaMemcpyAsync(history, dH, hs * nh * 8, cudaMemcpyDeviceToHost, s));
            LPX_CUDA(cudaStreamSynchronize(s));
        }
    } else {
        const int np = std::min(hstat[1], pivots_cap);
        if (np > 0) {
            LPX_CUDA(cudaMemcpyAsync(pivots, dpiv, (size_t)np * 8, cudaMemcpyDeviceToHost, s));
            if (theta) LPX_CUDA(cudaMemcpyAsync(theta, dtheta, (size_t)np * 8, cudaMemcpyDeviceToHost, s));
        }
        if (basis) LPX_CUDA(cudaMemcpyAsync(basis, dbasis, (size_t)m * 4, cudaMemcpyDeviceToHost, s));
        if (nonbasic) LPX_CUDA(cudaMemcpyAsync(nonbasic, dbasis + m, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
        if (xB) LPX_CUDA(cudaMemcpyAsync(xB, dx + n, (size_t)m * 8, cudaMemcpyDeviceToHost, s));
        if (x) LPX_CUDA(cudaMemcpyAsync(x, dx, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
        if (Binv) LPX_CUDA(cudaMemcpyAsync(Binv, dBinv, (size_t)m * m * 8, cudaMemcpyDeviceToHost, s));
        if (history && history_cap) {
            const int nh = std::min(hstat[1] + 1, history_cap);
            LPX_CUDA(cudaMemcpyAsync(history, dH, hs * nh * 8, cudaMemcpyDeviceToHost, s));
        }
        LPX_CUDA(cudaStreamSynchronize(s));
    }
    return LPX_OK;
}

}  // extern "C"
