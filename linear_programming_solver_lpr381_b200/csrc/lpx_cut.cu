// lpx_cut.cu — CuttingPlane.Solve (R/Models/CuttingPlane.cs:13-164) on the GPU, one CTA per IP: all 50 rounds of
// "Primal Simplex on the grown model, then one Gomory cut" run inside one launch, with nothing crossing PCIe between
// rounds.  Every round builds its tableau cold, as PrimalSimplex.Solve would for the model with the cuts so far, and
// pivots with the rules of cta_simplex_kernel's primal loop (lpx_cta.cuh), so the bits are the host loop's.
// The definition of the outputs is in include/lpx.h ("Gomory cutting plane"); oracle/orc_cutting.cpp restates the
// reference statement by statement.
//
// The primal loop is written here from the helpers cta_simplex_kernel uses (cta_stage_ratios,
// warp_margin_scan_staged, warp_argmin_below, cta_update) rather than shared with it: that kernel's loop also keeps the
// pivot log, the iteration history, the silent dual phase and the profiling ticks, and sharing it would make it branch
// on which caller it serves.
#include <cstring>
#include <vector>

#include "lpx_cta.cuh"
#include "lpx_runtime.hpp"

namespace lpx {

struct CutBatch {
    // the base IPs and the final-LP outputs: A, b, c, rel, strides, m_in, n, sense, m_base (= m'), max_iter,
    // max_rows / max_width (m' + 50, n + m' + 50), basis (stride m' + 49), x, z, tableau (stride
    // max_rows * max_width), total_pivots
    CtaBatch B;
    int* end;
    int* n_rounds;
    int* n_cuts;
    int* lp_status;  // [count][50], nullable
    int* lp_pivots;  // [count][50], nullable
    int* frac_var;   // [count][50], nullable
    int* cut_row;    // [count][50], nullable
    double* cut_a;   // the cut store, never null: [count][50][n]
    double* cut_b;   // [count][50]
    double* work;    // global-memory tableaux (!SMEM_T), stride B.tableau_stride
};

template <int THREADS, bool SMEM_T>
__global__ void __launch_bounds__(THREADS) cut_plane_kernel(const CutBatch K) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const CtaBatch& B = K.B;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = THREADS / 32;
    constexpr int R = LPX_CUT_MAX_ROUNDS;
    const int p = blockIdx.x;
    const int n = B.n, mm = B.m_base;

    const CtaCarve cv = cta_carve(B.max_rows, B.max_width, SMEM_T);
    double* prow = reinterpret_cast<double*>(smem_raw + cv.prow);
    double* fcol = reinterpret_cast<double*>(smem_raw + cv.fcol);
    double* zc = reinterpret_cast<double*>(smem_raw + cv.zc);
    int* rsrc = reinterpret_cast<int*>(smem_raw + cv.rsrc);
    int* rsgn = reinterpret_cast<int*>(smem_raw + cv.rsgn);
    int* sbasis = reinterpret_cast<int*>(smem_raw + cv.basis);
    int* ctl = reinterpret_cast<int*>(smem_raw + cv.ctl);
    double* T = SMEM_T ? reinterpret_cast<double*>(smem_raw + cv.T) : K.work + (size_t)p * B.tableau_stride;

    const double* Ai = B.A + (size_t)p * B.strideA;
    const double* bi = B.b + (size_t)p * B.strideB;
    const double* ci = B.c + (size_t)p * B.strideC;
    double* ca = K.cut_a + (size_t)p * R * n;
    double* cb = K.cut_b + (size_t)p * R;
    int* lst = K.lp_status ? K.lp_status + (size_t)p * R : nullptr;
    int* lpv = K.lp_pivots ? K.lp_pivots + (size_t)p * R : nullptr;

    // The base rows are the same in every round and a cut row is '<=' with b >= 0, so the GE / negative-RHS checks
    // (PrimalSimplex.cs:66-77) can only throw in round 1, and the row map (EQ expansion) is built once.
    cta_row_map<THREADS>(B, bi, 0, 0, 0, rsrc, rsgn, ctl);
    __syncthreads();
    const int st0 = ctl[0];

    int end = LPX_CUT_INCOMPLETE, rounds = 0;
    unsigned long long total = 0;
    int m = mm, rows = m + 1, width = n + m + 1, ld = width, rhs = width - 1;
    double* xs = prow;  // x of the round's LP: prow is free once its pivots are done
    if (st0 != LPX_RUNNING) {
        if (tid == 0) {
            if (lst) lst[0] = st0;
            if (lpv) lpv[0] = 0;
        }
        end = LPX_CUT_LP_ERROR;
        rounds = 1;
    }
    for (int r = 0; r < R && st0 == LPX_RUNNING; r++) {
        // ---- BuildTableau of the base model plus r cuts: base rows, cut rows, z-row last --------------------------
        m = mm + r;
        rows = m + 1;
        width = n + m + 1;
        ld = SMEM_T ? ((width + 1) & ~1) : width;
        rhs = width - 1;
        for (int i = warp; i < rows; i += NW) {
            double* Ti = T + (size_t)i * ld;
            if (i < mm) {
                const int src = rsrc[i];
                const bool flip = rsgn[i] != 0;
                const double* Ar = Ai + (size_t)src * n;
                for (int j = lane; j < width; j += 32) {
                    double v;
                    if (j < n) v = neg_if(Ar[j], flip);
                    else if (j == rhs) v = neg_if(bi[src], flip);
                    else v = (j == n + i) ? 1.0 : 0.0;
                    Ti[j] = v;
                }
            } else if (i < m) {
                const int k = i - mm;
                for (int j = lane; j < width; j += 32) {
                    double v;
                    if (j < n) v = ca[(size_t)k * n + j];
                    else if (j == rhs) v = cb[k];
                    else v = (j == n + i) ? 1.0 : 0.0;
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

        // ---- Primal Simplex (PrimalSimplex.cs:92-124), the rules of cta_simplex_kernel's primal loop: the control warp
        // keeps a private copy of the z-row and picks the next entering column while the other warps update ---------
        const double* zrow = T + (size_t)m * ld;
        if (warp == 0) {
            for (int j = lane; j < width; j += 32) zc[j] = zrow[j];
            __syncwarp();
            const int e0 = warp_argmin_below(zc, width - 1, -LPX_EPS);
            if (lane == 0) ctl[3] = e0;
        }
        __syncthreads();
        int steps = 0, why;
        while (true) {
            // "if (iter > MaxIterations) throw" comes before the optimality test (PrimalSimplex.cs:95-96)
            if (steps >= B.max_iter) {
                why = 0;
                break;
            }
            const int e = ctl[3];
            if (e < 0) {
                why = 1;
                break;
            }
            cta_stage_ratios<THREADS>(T, ld, m, e, rhs, prow);
            if (warp == 0) {
                const int lv = warp_margin_scan_staged(m, LPX_MARGIN_PRIMAL, prow);
                if (lane == 0) ctl[2] = lv;
            }
            __syncthreads();
            const int l = ctl[2];
            if (l < 0) {
                why = 2;
                break;
            }
            {
                const double piv = T[(size_t)l * ld + e];
                for (int j = tid; j < width; j += THREADS) prow[j] = ddiv_by_pivot(T[(size_t)l * ld + j], piv);
                for (int i = tid; i < rows; i += THREADS) fcol[i] = T[(size_t)i * ld + e];
                if (SMEM_T && tid == 0 && (width & 1)) prow[width] = 0.0;
            }
            __syncthreads();
            if (warp == 0) {
                const double fz = fcol[m];
                for (int j = lane; j < width; j += 32) zc[j] = __dsub_rn(zc[j], __dmul_rn(fz, prow[j]));
                __syncwarp();
                const int en = warp_argmin_below(zc, width - 1, -LPX_EPS);
                if (lane == 0) {
                    ctl[3] = en;
                    sbasis[l] = e;
                }
            } else {
                cta_update<SMEM_T>(T, ld, rows, width, l, prow, fcol, tid - 32, THREADS - 32);
            }
            __syncthreads();
            steps++;
        }
        const int st = why == 0 ? LPX_S_ITER_LIMIT : (why == 1 ? LPX_OPTIMAL : LPX_UNBOUNDED);
        if (tid == 0) {
            if (lst) lst[r] = st;
            if (lpv) lpv[r] = steps;
        }
        total += (unsigned long long)steps;
        rounds = r + 1;
        if (st == LPX_S_ITER_LIMIT) {  // PrimalSimplex threw: CuttingPlane.cs catches it and stops
            end = LPX_CUT_LP_ERROR;
            break;
        }

        // ---- x (an UNBOUNDED round's too), the first fractional x_j and its basis position (CuttingPlane.cs:77-117)
        for (int j = tid; j < n; j += THREADS) xs[j] = 0.0;
        if (tid == 0) ctl[6] = INT_MAX;
        __syncthreads();
        for (int i = tid; i < m; i += THREADS)  // distinct rows, distinct basic variables
            if (sbasis[i] < n) xs[sbasis[i]] = T[(size_t)i * ld + rhs];
        __syncthreads();
        for (int j = tid; j < n; j += THREADS) {
            const double v = xs[j];
            const double f = __dsub_rn(v, floor(v));
            if (f > LPX_EPS && f < 1.0 - LPX_EPS) atomicMin(&ctl[6], j);
        }
        __syncthreads();
        const int fv = ctl[6];
        if (fv == INT_MAX) {
            end = LPX_CUT_INTEGER;
            break;
        }
        // a fractional value is non-zero, hence basic in exactly one row; the cut is read one row BELOW it
        // ("+1 because row 0 is objective", CuttingPlane.cs:113), the z-row when that row is the last constraint row
        for (int i = tid; i < m; i += THREADS)
            if (sbasis[i] == fv) ctl[7] = i + 1;
        __syncthreads();
        const int row = ctl[7];

        // ---- GenerateGomoryCut (CuttingPlane.cs:142-163) into the cut store, read back by the next round's build --
        const double* trow = T + (size_t)row * ld;
        for (int j = tid; j < n; j += THREADS) {
            const double a = trow[j];
            const double f = __dsub_rn(a, floor(a));
            ca[(size_t)r * n + j] = f > LPX_EPS ? f : 0.0;
        }
        if (tid == 0) {
            const double v = trow[rhs];
            cb[r] = __dsub_rn(v, floor(v));
            if (K.frac_var) K.frac_var[(size_t)p * R + r] = fv;
            if (K.cut_row) K.cut_row[(size_t)p * R + r] = row;
        }
        __syncthreads();
    }
    __syncthreads();

    // ---- outputs: unused per-round / per-cut entries, then the final LP (INTEGER only) or zeros ------------------
    const int cuts = end == LPX_CUT_INCOMPLETE ? rounds : rounds - 1;
    for (int r = rounds + tid; r < R; r += THREADS) {
        if (lst) lst[r] = LPX_RUNNING;
        if (lpv) lpv[r] = 0;
    }
    for (int k = cuts + tid; k < R; k += THREADS) {
        if (K.frac_var) K.frac_var[(size_t)p * R + k] = -1;
        if (K.cut_row) K.cut_row[(size_t)p * R + k] = -1;
        cb[k] = 0.0;
    }
    for (size_t k = (size_t)cuts * n + tid; k < (size_t)R * n; k += THREADS) ca[k] = 0.0;

    const bool integral = end == LPX_CUT_INTEGER;
    if (B.basis) {
        int* bo = B.basis + (size_t)p * B.basis_stride;
        for (int i = tid; i < B.basis_stride; i += THREADS) bo[i] = integral && i < m ? sbasis[i] : 0;
    }
    if (B.x)
        for (int j = tid; j < n; j += THREADS) B.x[(size_t)p * n + j] = integral ? xs[j] : 0.0;
    if (B.z && tid == 0) B.z[p] = integral ? T[(size_t)m * ld + rhs] : 0.0;
    if (B.tableau) {
        double* To = B.tableau + (size_t)p * B.tableau_stride;
        const size_t used = integral ? (size_t)rows * width : 0;
        if (integral && (SMEM_T || T != To)) cta_copy_out<THREADS>(To, T, ld, rows, width);
        for (size_t k = used + tid; k < (size_t)B.tableau_stride; k += THREADS) To[k] = 0.0;
    }
    if (tid == 0) {
        K.end[p] = end;
        if (K.n_rounds) K.n_rounds[p] = rounds;
        if (K.n_cuts) K.n_cuts[p] = cuts;
        if (B.total_pivots && total) atomicAdd(B.total_pivots, total);
    }
}

static int expanded_rows(int m, const int* rel) {
    int mm = 0;
    for (int i = 0; i < m; i++) mm += (rel && rel[i] == 2) ? 2 : 1;
    return mm;
}

static int check_args(int count, int m, int n, int sense, const int* host_rel, const lpx_options& o) {
    if (count < 1 || m < 1 || n < 1 || (sense != 0 && sense != 1)) {
        set_error("cutting plane: bad arguments: need count >= 1, m >= 1, n >= 1, sense in {0,1}");
        return LPX_E_BAD_ARGS;
    }
    if (host_rel)
        for (int i = 0; i < m; i++)
            if (host_rel[i] < 0 || host_rel[i] > 2) {
                set_error("bad arguments: rel[i] must be 0 (LE), 1 (GE) or 2 (EQ)");
                return LPX_E_BAD_ARGS;
            }
    if (o.kernel != LPX_KERNEL_AUTO && o.kernel != LPX_KERNEL_CTA_SMEM && o.kernel != LPX_KERNEL_CTA_GLOBAL) {
        set_error("cutting plane runs on the per-CTA kernels: opt.kernel must be AUTO, CTA_SMEM or CTA_GLOBAL");
        return LPX_E_BAD_ARGS;
    }
    return LPX_OK;
}

template <int THREADS, bool SMEM_T>
static int launch_cut_variant(const CutBatch& K, int count, size_t smem, cudaStream_t stream) {
    auto kfn = cut_plane_kernel<THREADS, SMEM_T>;
    LPX_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kfn<<<count, THREADS, smem, stream>>>(K);
    LPX_CUDA(cudaGetLastError());
    count_launch();
    return LPX_OK;
}

// Everything on the device already; mm (rows after EQ expansion) known on the host.  cut_a / cut_b / tableau may be
// null: library scratch stands in for the cut store and for the working tableaux of the global-memory build.
static int cut_launch(int count, int m, int n, int sense, int mm, const double* A, const int* rel, const double* b,
                      const double* c, const lpx_options& o, int* end, int* n_rounds, int* n_cuts, int* lp_status,
                      int* lp_pivots, int* frac_var, int* cut_row, double* cut_a, double* cut_b, int* basis, double* x,
                      double* z, double* tableau, unsigned long long* total_pivots, cudaStream_t stream) {
    const int R = LPX_CUT_MAX_ROUNDS;
    const int max_rows = mm + R, max_cols = n + mm + R;
    const bool fits = cta_fits_smem(max_rows, max_cols);
    if (o.kernel == LPX_KERNEL_CTA_SMEM && !fits) {
        set_error("cutting plane: the 50-round tableau does not fit in shared memory (LPX_KERNEL_CTA_SMEM forced)");
        return LPX_E_CAPACITY;
    }
    const bool smem_T = fits && o.kernel != LPX_KERNEL_CTA_GLOBAL;
    const size_t smem = cta_carve(max_rows, max_cols, smem_T).total;
    if (smem > (size_t)max_smem_optin()) {
        set_error("cutting plane: problem too wide for the per-CTA kernels (work vectors exceed shared memory)");
        return LPX_E_CAPACITY;
    }
    const size_t cnt = (size_t)count, tstride = (size_t)max_rows * max_cols;
    if (!cut_a || !cut_b) {
        double* store = ws_dev_as<double>(WS_CUT_STORE, cnt * R * ((size_t)n + 1));
        if (!store) return LPX_E_CUDA;
        if (!cut_a) cut_a = store;
        if (!cut_b) cut_b = store + cnt * R * n;
    }
    double* work = nullptr;
    if (!smem_T) {
        work = tableau ? tableau : ws_dev_as<double>(WS_SCRATCH, cnt * tstride);
        if (!work) return LPX_E_CUDA;
    }

    CutBatch K;
    std::memset(&K, 0, sizeof K);
    CtaBatch& B = K.B;
    B.A = A;
    B.b = b;
    B.c = c;
    B.rel = rel;
    B.strideA = (long long)m * n;
    B.strideB = m;
    B.strideC = n;
    B.m_in = m;
    B.n = n;
    B.sense = sense;
    B.m_base = mm;
    B.max_iter = o.max_iterations;
    B.max_rows = max_rows;
    B.max_width = max_cols;
    B.basis = basis;
    B.basis_stride = mm + R - 1;
    B.x = x;
    B.z = z;
    B.tableau = tableau;
    B.tableau_stride = (long long)tstride;
    B.total_pivots = total_pivots;
    K.end = end;
    K.n_rounds = n_rounds;
    K.n_cuts = n_cuts;
    K.lp_status = lp_status;
    K.lp_pivots = lp_pivots;
    K.frac_var = frac_var;
    K.cut_row = cut_row;
    K.cut_a = cut_a;
    K.cut_b = cut_b;
    K.work = work;

    int threads = o.threads;
    if (threads != 128 && threads != 256 && threads != 512)  // as cta_launch chooses (lpx_cta.cu)
        threads = (!smem_T || (size_t)max_rows * max_cols >= 8192) ? 512 : 256;
    if (smem_T) {
        if (threads == 128) return launch_cut_variant<128, true>(K, count, smem, stream);
        if (threads == 256) return launch_cut_variant<256, true>(K, count, smem, stream);
        return launch_cut_variant<512, true>(K, count, smem, stream);
    }
    if (threads == 128) return launch_cut_variant<128, false>(K, count, smem, stream);
    if (threads == 256) return launch_cut_variant<256, false>(K, count, smem, stream);
    return launch_cut_variant<512, false>(K, count, smem, stream);
}

}  // namespace lpx

using namespace lpx;

extern "C" {

int lpx_cutting_plane_dims(int m, int n, const int* rel, int* max_rows, int* max_cols) {
    lpx_options o;
    lpx_default_options(&o);
    int rc = check_args(1, m, n, 0, rel, o);
    if (rc != LPX_OK) return rc;
    const int mm = expanded_rows(m, rel);
    if (max_rows) *max_rows = mm + LPX_CUT_MAX_ROUNDS;
    if (max_cols) *max_cols = n + mm + LPX_CUT_MAX_ROUNDS;
    return LPX_OK;
}

int lpx_cutting_plane_batched_dev(int count, int m, int n, int sense, const double* A, const int* rel, const double* b,
                                  const double* c, const lpx_options* opt, int* end, int* n_rounds, int* n_cuts,
                                  int* lp_status, int* lp_pivots, int* frac_var, int* cut_row, double* cut_a,
                                  double* cut_b, int* basis, double* x, double* z, double* tableau,
                                  unsigned long long* total_pivots, void* stream) {
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    int rc = check_args(count, m, n, sense, nullptr, o);
    if (rc != LPX_OK) return rc;
    if (!A || !b || !c || !end) {
        set_error("lpx_cutting_plane_batched_dev: A, b, c and end must not be NULL");
        return LPX_E_BAD_ARGS;
    }
    if ((rc = ensure_device()) != LPX_OK) return rc;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    cudaStream_t s = (cudaStream_t)stream;
    // rel is a device pointer; the tableau shape needs it on the host
    int mm = m;
    if (rel) {
        std::vector<int> hrel(m);
        LPX_CUDA(cudaMemcpyAsync(hrel.data(), rel, (size_t)m * 4, cudaMemcpyDeviceToHost, s));
        LPX_CUDA(cudaStreamSynchronize(s));
        if ((rc = check_args(count, m, n, sense, hrel.data(), o)) != LPX_OK) return rc;
        mm = expanded_rows(m, hrel.data());
    }
    return cut_launch(count, m, n, sense, mm, A, rel, b, c, o, end, n_rounds, n_cuts, lp_status, lp_pivots, frac_var,
                      cut_row, cut_a, cut_b, basis, x, z, tableau, total_pivots, s);
}

int lpx_cutting_plane_batched(int count, int m, int n, int sense, const double* A, const int* rel, const double* b,
                              const double* c, const lpx_options* opt, int* end, int* n_rounds, int* n_cuts,
                              int* lp_status, int* lp_pivots, int* frac_var, int* cut_row, double* cut_a, double* cut_b,
                              int* basis, double* x, double* z, double* tableau, long long* total_pivots) {
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    int rc = check_args(count, m, n, sense, rel, o);
    if (rc != LPX_OK) return rc;
    if (!A || !b || !c || !end) {
        set_error("lpx_cutting_plane_batched: A, b, c and end must not be NULL");
        return LPX_E_BAD_ARGS;
    }
    if ((rc = ensure_device()) != LPX_OK) return rc;
    Runtime& r = rt();
    std::lock_guard<std::recursive_mutex> lk(r.mu);
    cudaStream_t s = r.stream;
    const int R = LPX_CUT_MAX_ROUNDS;
    const int mm = expanded_rows(m, rel);
    const size_t cnt = (size_t)count, per = cnt * R, bstride = (size_t)mm + R - 1;
    const size_t tstride = (size_t)(mm + R) * (n + mm + R);

    double* dA = ws_dev_as<double>(WS_A, cnt * m * n);
    double* db = ws_dev_as<double>(WS_B, cnt * m);
    double* dc = ws_dev_as<double>(WS_C, cnt * n);
    int* drel = ws_dev_as<int>(WS_REL, m);
    // ints: end, n_rounds, n_cuts | lp_status, lp_pivots, frac_var, cut_row | basis
    int* di = ws_dev_as<int>(WS_CUT_INT, 3 * cnt + 4 * per + cnt * bstride);
    // doubles: cut_a | cut_b | x | z
    double* dd = ws_dev_as<double>(WS_CUT_DBL, per * n + per + cnt * n + cnt);
    double* dT = tableau ? ws_dev_as<double>(WS_TABLEAU, cnt * tstride) : nullptr;
    unsigned long long* dtot = ws_dev_as<unsigned long long>(WS_TOTAL, 1);
    if (!dA || !db || !dc || !drel || !di || !dd || (tableau && !dT) || !dtot) return LPX_E_CUDA;
    int *dend = di, *dnr = di + cnt, *dnc = di + 2 * cnt, *dls = di + 3 * cnt, *dlp = dls + per, *dfv = dlp + per,
        *dcr = dfv + per, *dbasis = dcr + per;
    double *dca = dd, *dcb = dd + per * n, *dx = dcb + per, *dz = dx + cnt * n;

    LPX_CUDA(cudaMemcpyAsync(dA, A, cnt * m * n * 8, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemcpyAsync(db, b, cnt * m * 8, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemcpyAsync(dc, c, cnt * n * 8, cudaMemcpyHostToDevice, s));
    if (rel) LPX_CUDA(cudaMemcpyAsync(drel, rel, (size_t)m * 4, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemsetAsync(dtot, 0, 8, s));
    rc = cut_launch(count, m, n, sense, mm, dA, rel ? drel : nullptr, db, dc, o, dend, dnr, dnc,
                    lp_status ? dls : nullptr, lp_pivots ? dlp : nullptr, frac_var ? dfv : nullptr,
                    cut_row ? dcr : nullptr, dca, dcb, basis ? dbasis : nullptr, x ? dx : nullptr, z ? dz : nullptr, dT,
                    dtot, s);
    if (rc != LPX_OK) return rc;
    auto down = [&](void* dst, const void* src, size_t bytes) {
        return dst ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, s) : cudaSuccess;
    };
    unsigned long long htot = 0;
    LPX_CUDA(down(end, dend, cnt * 4));
    LPX_CUDA(down(n_rounds, dnr, cnt * 4));
    LPX_CUDA(down(n_cuts, dnc, cnt * 4));
    LPX_CUDA(down(lp_status, dls, per * 4));
    LPX_CUDA(down(lp_pivots, dlp, per * 4));
    LPX_CUDA(down(frac_var, dfv, per * 4));
    LPX_CUDA(down(cut_row, dcr, per * 4));
    LPX_CUDA(down(cut_a, dca, per * n * 8));
    LPX_CUDA(down(cut_b, dcb, per * 8));
    LPX_CUDA(down(basis, dbasis, cnt * bstride * 4));
    LPX_CUDA(down(x, dx, cnt * n * 8));
    LPX_CUDA(down(z, dz, cnt * 8));
    LPX_CUDA(down(tableau, dT, cnt * tstride * 8));
    LPX_CUDA(down(&htot, dtot, 8));
    LPX_CUDA(cudaStreamSynchronize(s));
    if (total_pivots) *total_pivots = (long long)htot;
    return LPX_OK;
}

}  // extern "C"
