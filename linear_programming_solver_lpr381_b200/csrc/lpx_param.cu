// lpx_param.cu — parametric analysis of optimal Primal Simplex results (include/lpx.h, "Parametric analysis"): the
// piecewise-linear optimal value z*(theta) along b + theta d or c + theta d, one CTA per query.  Each query's working
// tableau is its base's final tableau plus one direction column g (RHS) or one direction row h (COST); the loop finds
// the next breakpoint with the sensitivity report's tie rule (sens_pick), writes the segment that closes there and
// pivots with the Dual (RHS) or Primal (COST) Simplex rules of cta_simplex_kernel, all without leaving the CTA.
// oracle/orc_param.cpp restates the definition as sequential loops.
//
// The loop is written here from the helpers cta_simplex_kernel uses (cta_stage_ratios, warp_margin_scan_staged,
// warp_margin_scan_cert, cta_pivot) rather than as a branch of that kernel, which keeps its register allocation
// (DESIGN §4.12 gives the same reason for the cutting-plane kernel).
#include <cstring>
#include <vector>

#include "lpx_cta.cuh"
#include "lpx_runtime.hpp"
#include "lpx_sens.cuh"

namespace lpx {

struct ParamBatch {
    int kind, m_in, n, sense, mm;  // mm = m' (rows after EQ expansion)
    int rows, width;               // the working tableau: (m' + 1) x (W + 1) for RHS, (m' + 2) x W for COST
    int seg_cap;
    const int* rel;  // device, nullable = all LE
    const int* base_status;
    const int* base_basis;
    const double* base_T;
    const int* src;  // nullable: query q reads base q
    const double* payload;
    long long pstride;
    int* end;
    int* n_segments;
    int* n_pivots;
    double* segments;  // [seg_cap][4 + 2n] per query
    int* seg_pivots;   // [seg_cap][2] per query
    int* basis;        // m' per query
    double* tableau;   // rows * width per query, compact
    double* work;      // global-memory tableaux (!SMEM_T), stride rows * width
    unsigned long long* total_pivots;
};

template <int THREADS, bool SMEM_T>
__global__ void __launch_bounds__(THREADS) param_kernel(const ParamBatch P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = THREADS / 32;
    const int q = blockIdx.x;
    const bool rk = P.kind == LPX_PARAM_RHS;
    const int n = P.n, mm = P.mm, W = n + mm + 1, rhs = W - 1;
    const int rows = P.rows, width = P.width, ld = SMEM_T ? ((width + 1) & ~1) : width;
    const size_t tsize = (size_t)rows * width;

    const CtaCarve cv = cta_carve(rows, width, SMEM_T);
    double* prow = reinterpret_cast<double*>(smem_raw + cv.prow);
    double* fcol = reinterpret_cast<double*>(smem_raw + cv.fcol);
    SensBest* red = reinterpret_cast<SensBest*>(smem_raw + cv.red);
    int* sbasis = reinterpret_cast<int*>(smem_raw + cv.basis);
    int* ctl = reinterpret_cast<int*>(smem_raw + cv.ctl);
    int* rowof = reinterpret_cast<int*>(smem_raw + cv.zc);  // W ints: basic row of each column, -1 if non-basic
    double* T = SMEM_T ? reinterpret_cast<double*>(smem_raw + cv.T) : P.work + (size_t)q * tsize;

    const long long s = P.src ? P.src[q] : q;
    const double* d = P.payload + (size_t)q * P.pstride;
    const double theta_max = d[rk ? P.m_in : n];
    const int sstride = 4 + 2 * n;
    double* seg = P.segments ? P.segments + (size_t)q * P.seg_cap * sstride : nullptr;
    int* spv = P.seg_pivots ? P.seg_pivots + (size_t)q * P.seg_cap * 2 : nullptr;

    int end = LPX_PARAM_NO_BASE, k = 0;
    if (P.base_status[s] == LPX_OPTIMAL) {
        // ---- the working tableau: the base's, plus g (column W) or h (row m' + 1), in the definition's order ------
        const double* Ts = P.base_T + (size_t)s * (mm + 1) * W;
        const int* bs = P.base_basis + (size_t)s * mm;
        for (int j = tid; j < W; j += THREADS) rowof[j] = -1;
        __syncthreads();
        for (int i = tid; i < mm; i += THREADS) {
            sbasis[i] = bs[i];
            rowof[bs[i]] = i;
        }
        __syncthreads();
        for (int i = warp; i < rows; i += NW) {
            double* Ti = T + (size_t)i * ld;
            for (int j = lane; j < width; j += 32) {
                double v;
                if (rk) {
                    if (j < W) {
                        v = Ts[(size_t)i * W + j];
                    } else {  // g_i: d_i T[i][s1] (EQ: - d_i T[i][s2]) for the constraints in order, from +0
                        v = 0.0;
                        int i1 = 0;
                        for (int c = 0; c < P.m_in; c++) {
                            const bool eq = P.rel && P.rel[c] == 2;
                            const double dc = d[c];
                            if (dc != 0.0) {
                                v = __dadd_rn(v, __dmul_rn(dc, Ts[(size_t)i * W + n + i1]));
                                if (eq) v = __dsub_rn(v, __dmul_rn(dc, Ts[(size_t)i * W + n + i1 + 1]));
                            }
                            i1 += eq ? 2 : 1;
                        }
                    }
                } else if (i <= mm) {
                    v = Ts[(size_t)i * W + j];
                } else {  // h[j]: the COST query's terms applied to a zero row
                    v = 0.0;
                    for (int c = 0; c < n; c++) {
                        const double dc = d[c];
                        if (dc == 0.0) continue;
                        const double delta = P.sense == 1 ? dneg(dc) : dc;
                        if (rowof[c] >= 0) v = __dadd_rn(v, __dmul_rn(delta, Ts[(size_t)rowof[c] * W + j]));
                        if (j == c) v = __dsub_rn(v, delta);
                    }
                }
                Ti[j] = v;
            }
        }
        if (ld > width)
            for (int i = tid; i < rows; i += THREADS) T[(size_t)i * ld + width] = 0.0;  // pad column
        __syncthreads();

        const double* zrow = T + (size_t)mm * ld;
        double th_lo = 0.0;
        while (true) {
            // ---- theta_cand: min -(beta_r / g_r) over g_r < -EPS (RHS), min -(z_k / h_k) over non-basic k with
            // h_k < -EPS (COST); NaN never chosen, ties to the lowest index -----------------------------------------
            SensBest best = sens_empty();
            if (rk) {
                for (int r = tid; r < mm; r += THREADS) {
                    const double g = T[(size_t)r * ld + W];
                    if (g < -LPX_EPS) {
                        SensBest c;
                        c.v = -__ddiv_rn(T[(size_t)r * ld + rhs], g);
                        c.i = r;
                        if (c.v == c.v) sens_pick<false>(best, c);
                    }
                }
            } else {
                const double* hrow = T + (size_t)(mm + 1) * ld;
                for (int j = tid; j < rhs; j += THREADS) {
                    const double h = hrow[j];
                    if (rowof[j] < 0 && h < -LPX_EPS) {
                        SensBest c;
                        c.v = -__ddiv_rn(zrow[j], h);
                        c.i = j;
                        if (c.v == c.v) sens_pick<false>(best, c);
                    }
                }
            }
            best = sens_warp_reduce<false>(best);
            if (lane == 0) red[warp] = best;
            __syncthreads();
            SensBest all = lane < NW ? red[lane] : sens_empty();
            all = sens_warp_reduce<false>(all);
            __syncthreads();  // red is free again
            const double cand = all.i == INT_MAX ? sens_inf() : all.v;
            const double th_end = cand < th_lo ? th_lo : cand;

            int stop = -1, pl = -1, pe = -1;
            double th_hi = th_end;
            if (th_end >= theta_max) {
                stop = LPX_PARAM_REACHED;
                th_hi = theta_max;
            } else if (k + 1 == P.seg_cap) {
                stop = LPX_PARAM_SEG_LIMIT;
            } else if (rk) {
                // row all.i leaves; the entering column by the Dual Simplex rule: min z_j / -a over a < -EPS, margin
                // 1e-12, columns < W - 1
                const int l = all.i;
                const double* lrow = T + (size_t)l * ld;
                for (int j = tid; j < rhs; j += THREADS) {
                    const double a = lrow[j];
                    double r = sens_nan();
                    if (a < -LPX_EPS) r = ddiv_by_pivot(zrow[j], dneg(a));
                    prow[j] = r;
                }
                __syncthreads();
                if (warp == 0) {
                    const int ev = warp_margin_scan_cert(rhs, LPX_MARGIN_DUAL, [&](int j, double& r) {
                        r = prow[j];
                        return r == r;
                    });
                    if (lane == 0) ctl[2] = ev;
                }
                __syncthreads();
                pe = ctl[2];
                if (pe < 0) stop = LPX_PARAM_INFEASIBLE;
                else pl = l;
            } else {
                // column all.i enters; the leaving row by the Primal Simplex rule (ratio margin 1e-9)
                const int e = all.i;
                cta_stage_ratios<THREADS>(T, ld, mm, e, rhs, prow);
                if (warp == 0) {
                    const int lv = warp_margin_scan_staged(mm, LPX_MARGIN_PRIMAL, prow);
                    if (lane == 0) ctl[2] = lv;
                }
                __syncthreads();
                pl = ctl[2];
                if (pl < 0) stop = LPX_PARAM_UNBOUNDED;
                else pe = e;
            }

            // ---- segment k: theta_lo | theta_hi | z0 | dz | x0[n] | dx[n], read before the pivot ------------------
            if (seg) {
                double* rec = seg + (size_t)k * sstride;
                if (tid == 0) {
                    rec[0] = th_lo;
                    rec[1] = th_hi;
                    rec[2] = zrow[rhs];
                    rec[3] = rk ? zrow[W] : T[(size_t)(mm + 1) * ld + rhs];
                }
                for (int j = tid; j < n; j += THREADS) {
                    const int r = rowof[j];
                    rec[4 + j] = r >= 0 ? T[(size_t)r * ld + rhs] : 0.0;
                    rec[4 + n + j] = (rk && r >= 0) ? T[(size_t)r * ld + W] : 0.0;
                }
            }
            if (spv && tid == 0) {
                spv[2 * k] = pl;
                spv[2 * k + 1] = pe;
            }
            k++;
            if (stop >= 0) {
                end = stop;
                break;
            }
            cta_pivot<THREADS, SMEM_T>(T, ld, rows, width, pl, pe, prow, fcol);
            if (tid == 0) {
                rowof[sbasis[pl]] = -1;
                rowof[pe] = pl;
                sbasis[pl] = pe;
            }
            __syncthreads();
            th_lo = th_end;
        }
    }

    // ---- outputs: records past the last segment are zero with pivot (-1, -1); a query without a base gets zeros -----
    const bool ok = end != LPX_PARAM_NO_BASE;
    if (seg)
        for (size_t e = (size_t)k * sstride + tid; e < (size_t)P.seg_cap * sstride; e += THREADS) seg[e] = 0.0;
    if (spv)
        for (int e = 2 * k + tid; e < 2 * P.seg_cap; e += THREADS) spv[e] = -1;
    if (P.basis)
        for (int i = tid; i < mm; i += THREADS) P.basis[(size_t)q * mm + i] = ok ? sbasis[i] : 0;
    if (P.tableau) {
        double* To = P.tableau + (size_t)q * tsize;
        if (!ok) {
            for (size_t e = tid; e < tsize; e += THREADS) To[e] = 0.0;
        } else if (SMEM_T || T != To) {
            cta_copy_out<THREADS>(To, T, ld, rows, width);
        }
    }
    if (tid == 0) {
        P.end[q] = end;
        if (P.n_segments) P.n_segments[q] = k;
        if (P.n_pivots) P.n_pivots[q] = ok ? k - 1 : 0;
        if (P.total_pivots && k > 1) atomicAdd(P.total_pivots, (unsigned long long)(k - 1));
    }
}

static bool known_kind(int kind) { return kind == LPX_PARAM_RHS || kind == LPX_PARAM_COST; }

static int expanded_rows(int m, const int* rel) {
    int mm = 0;
    for (int i = 0; i < m; i++) mm += (rel && rel[i] == 2) ? 2 : 1;
    return mm;
}

static void work_dims(int kind, int n, int mm, int& rows, int& cols) {
    rows = mm + 1 + (kind == LPX_PARAM_COST);
    cols = n + mm + 1 + (kind == LPX_PARAM_RHS);
}

static int check_args(int kind, int count, int m, int n, int sense, int seg_cap, const int* host_rel,
                      const lpx_options& o) {
    if (!known_kind(kind) || count < 0 || m < 1 || n < 1 || (sense != 0 && sense != 1) || seg_cap < 1) {
        set_error("parametric analysis: bad arguments: need kind RHS or COST, count >= 0, m >= 1, n >= 1, sense in "
                  "{0,1}, seg_cap >= 1");
        return LPX_E_BAD_ARGS;
    }
    if (host_rel)
        for (int i = 0; i < m; i++)
            if (host_rel[i] < 0 || host_rel[i] > 2) {
                set_error("bad arguments: rel[i] must be 0 (LE), 1 (GE) or 2 (EQ)");
                return LPX_E_BAD_ARGS;
            }
    if (o.kernel != LPX_KERNEL_AUTO && o.kernel != LPX_KERNEL_CTA_SMEM && o.kernel != LPX_KERNEL_CTA_GLOBAL) {
        set_error("parametric analysis runs on the per-CTA kernels: opt.kernel must be AUTO, CTA_SMEM or CTA_GLOBAL");
        return LPX_E_BAD_ARGS;
    }
    return LPX_OK;
}

// theta_max of every query: >= 0 or +inf; NaN and negative values are refused.
static int check_theta_max(const double* tmax, int count) {
    for (int q = 0; q < count; q++)
        if (!(tmax[q] >= 0.0)) {
            set_error("parametric analysis: theta_max must be >= 0 or +inf (not NaN)");
            return LPX_E_BAD_ARGS;
        }
    return LPX_OK;
}

template <int THREADS, bool SMEM_T>
static int launch_param_variant(const ParamBatch& P, int count, size_t smem, cudaStream_t stream) {
    auto kfn = param_kernel<THREADS, SMEM_T>;
    LPX_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kfn<<<count, THREADS, smem, stream>>>(P);
    LPX_CUDA(cudaGetLastError());
    count_launch();
    return LPX_OK;
}

// Everything on the device already; mm known on the host, arguments and theta_max checked.
static int param_launch(int kind, int count, int m, int n, int sense, const int* rel, int mm, const int* base_status,
                        const int* base_basis, const double* base_T, const int* src, const double* payload,
                        int seg_cap, const lpx_options& o, int* end, int* n_segments, int* n_pivots, double* segments,
                        int* seg_pivots, int* basis, double* tableau, unsigned long long* total_pivots,
                        cudaStream_t stream) {
    int rows, cols;
    work_dims(kind, n, mm, rows, cols);
    const bool fits = cta_fits_smem(rows, cols);
    if (o.kernel == LPX_KERNEL_CTA_SMEM && !fits) {
        set_error("parametric analysis: the working tableau does not fit in shared memory (LPX_KERNEL_CTA_SMEM forced)");
        return LPX_E_CAPACITY;
    }
    const bool smem_T = fits && o.kernel != LPX_KERNEL_CTA_GLOBAL;
    const size_t smem = cta_carve(rows, cols, smem_T).total;
    if (smem > (size_t)max_smem_optin()) {
        set_error("parametric analysis: problem too wide for the per-CTA kernels (work vectors exceed shared memory)");
        return LPX_E_CAPACITY;
    }
    if (count == 0) return LPX_OK;
    const size_t tsize = (size_t)rows * cols;
    double* work = nullptr;
    if (!smem_T) {
        work = tableau ? tableau : ws_dev_as<double>(WS_SCRATCH, (size_t)count * tsize);
        if (!work) return LPX_E_CUDA;
    }
    ParamBatch P;
    std::memset(&P, 0, sizeof P);
    P.kind = kind;
    P.m_in = m;
    P.n = n;
    P.sense = sense;
    P.mm = mm;
    P.rows = rows;
    P.width = cols;
    P.seg_cap = seg_cap;
    P.rel = rel;
    P.base_status = base_status;
    P.base_basis = base_basis;
    P.base_T = base_T;
    P.src = src;
    P.payload = payload;
    P.pstride = (long long)lpx_param_payload_stride(kind, m, n);
    P.end = end;
    P.n_segments = n_segments;
    P.n_pivots = n_pivots;
    P.segments = segments;
    P.seg_pivots = seg_pivots;
    P.basis = basis;
    P.tableau = tableau;
    P.work = work;
    P.total_pivots = total_pivots;

    int threads = o.threads;
    if (threads != 128 && threads != 256 && threads != 512)  // as cta_launch chooses (lpx_cta.cu)
        threads = (!smem_T || tsize >= 8192) ? 512 : 256;
    if (smem_T) {
        if (threads == 128) return launch_param_variant<128, true>(P, count, smem, stream);
        if (threads == 256) return launch_param_variant<256, true>(P, count, smem, stream);
        return launch_param_variant<512, true>(P, count, smem, stream);
    }
    if (threads == 128) return launch_param_variant<128, false>(P, count, smem, stream);
    if (threads == 256) return launch_param_variant<256, false>(P, count, smem, stream);
    return launch_param_variant<512, false>(P, count, smem, stream);
}

}  // namespace lpx

using namespace lpx;

extern "C" {

size_t lpx_param_payload_stride(int kind, int m, int n) {
    if (m < 0 || n < 0) return 0;
    if (kind == LPX_PARAM_RHS) return (size_t)m + 1;
    if (kind == LPX_PARAM_COST) return (size_t)n + 1;
    return 0;
}

size_t lpx_param_segment_stride(int n) { return n < 0 ? 0 : 4 + 2 * (size_t)n; }

int lpx_parametric_dims(int kind, int m, int n, const int* rel, int* rows, int* cols) {
    lpx_options o;
    lpx_default_options(&o);
    int rc = check_args(kind, 0, m, n, 0, 1, rel, o);
    if (rc != LPX_OK) return rc;
    int r, c;
    work_dims(kind, n, expanded_rows(m, rel), r, c);
    if (rows) *rows = r;
    if (cols) *cols = c;
    return LPX_OK;
}

int lpx_parametric_batched_dev(int kind, int count, int m, int n, int sense, const int* rel, const int* base_status,
                               const int* base_basis, const double* base_tableau, const int* src,
                               const double* payload, int seg_cap, const lpx_options* opt, int* end, int* n_segments,
                               int* n_pivots, double* segments, int* seg_pivots, int* basis, double* tableau,
                               unsigned long long* total_pivots, void* stream) {
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    int rc = check_args(kind, count, m, n, sense, seg_cap, nullptr, o);
    if (rc != LPX_OK) return rc;
    if (!base_status || !base_basis || !base_tableau || !payload || !end) {
        set_error("lpx_parametric_batched_dev: base_status, base_basis, base_tableau, payload and end must not be NULL");
        return LPX_E_BAD_ARGS;
    }
    if ((rc = ensure_device()) != LPX_OK) return rc;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    cudaStream_t s = (cudaStream_t)stream;
    // rel (the tableau shape) and theta_max are device data the host has to see once
    int mm = m;
    if (rel) {
        std::vector<int> hrel(m);
        LPX_CUDA(cudaMemcpyAsync(hrel.data(), rel, (size_t)m * 4, cudaMemcpyDeviceToHost, s));
        LPX_CUDA(cudaStreamSynchronize(s));
        if ((rc = check_args(kind, count, m, n, sense, seg_cap, hrel.data(), o)) != LPX_OK) return rc;
        mm = expanded_rows(m, hrel.data());
    }
    if (count > 0) {
        const size_t stride = lpx_param_payload_stride(kind, m, n);
        std::vector<double> tmax(count);
        LPX_CUDA(cudaMemcpy2DAsync(tmax.data(), 8, payload + stride - 1, stride * 8, 8, (size_t)count,
                                   cudaMemcpyDeviceToHost, s));
        LPX_CUDA(cudaStreamSynchronize(s));
        if ((rc = check_theta_max(tmax.data(), count)) != LPX_OK) return rc;
    }
    return param_launch(kind, count, m, n, sense, rel, mm, base_status, base_basis, base_tableau, src, payload, seg_cap,
                        o, end, n_segments, n_pivots, segments, seg_pivots, basis, tableau, total_pivots, s);
}

int lpx_parametric(int kind, int m, int n, int sense, const double* A, const int* rel, const double* b,
                   const double* c, const lpx_options* opt, int count, const double* payload, int seg_cap,
                   int* base_status, int* end, int* n_segments, int* n_pivots, double* segments, int* seg_pivots,
                   int* basis, double* tableau) {
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    int rc = check_args(kind, count, m, n, sense, seg_cap, rel, o);
    if (rc != LPX_OK) return rc;
    if (!A || !b || !c || (count > 0 && (!payload || !end))) {
        set_error("lpx_parametric: A, b, c, payload and end must not be NULL");
        return LPX_E_BAD_ARGS;
    }
    const size_t stride = lpx_param_payload_stride(kind, m, n);
    {
        std::vector<double> tmax(count);
        for (int q = 0; q < count; q++) tmax[q] = payload[(size_t)q * stride + stride - 1];
        if ((rc = check_theta_max(tmax.data(), count)) != LPX_OK) return rc;
    }
    if ((rc = ensure_device()) != LPX_OK) return rc;
    Runtime& r = rt();
    std::lock_guard<std::recursive_mutex> lk(r.mu);
    cudaStream_t s = r.stream;
    const int mm = expanded_rows(m, rel);
    int rows, cols;
    work_dims(kind, n, mm, rows, cols);
    const size_t cnt = (size_t)count, tsize = (size_t)rows * cols, base_tsize = (size_t)(mm + 1) * (n + mm + 1);
    const size_t sstride = lpx_param_segment_stride(n), cap = (size_t)seg_cap;

    // the base: one Primal Simplex solve on the GPU, its final tableau kept on the device
    double* dA = ws_dev_as<double>(WS_A, (size_t)m * n);
    double* db = ws_dev_as<double>(WS_B, m);
    double* dc = ws_dev_as<double>(WS_C, n);
    int* drel = ws_dev_as<int>(WS_REL, m);
    double* dbT = ws_dev_as<double>(WS_RO_BASE_T, base_tsize);
    int* dbI = ws_dev_as<int>(WS_RO_BASE_I, (size_t)mm + 1);  // status, then the basis
    if (!dA || !db || !dc || !drel || !dbT || !dbI) return LPX_E_CUDA;
    LPX_CUDA(cudaMemcpyAsync(dA, A, (size_t)m * n * 8, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemcpyAsync(db, b, (size_t)m * 8, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemcpyAsync(dc, c, (size_t)n * 8, cudaMemcpyHostToDevice, s));
    if (rel) LPX_CUDA(cudaMemcpyAsync(drel, rel, (size_t)m * 4, cudaMemcpyHostToDevice, s));
    lpx_options ob = o;
    ob.kernel = LPX_KERNEL_AUTO;
    rc = lpx_primal_solve_batched_dev(1, m, n, sense, dA, rel ? drel : nullptr, db, dc, &ob, dbI, nullptr, dbI + 1,
                                      nullptr, nullptr, dbT, nullptr, s);
    if (rc != LPX_OK) return rc;
    if (base_status) {
        LPX_CUDA(cudaMemcpyAsync(base_status, dbI, 4, cudaMemcpyDeviceToHost, s));
        LPX_CUDA(cudaStreamSynchronize(s));
    }
    if (count == 0) return LPX_OK;

    // the queries, all against base 0.  ints: src, end, n_segments, n_pivots | seg_pivots | basis;
    // doubles: payload | segments | tableau
    int* di = ws_dev_as<int>(WS_PM_INT, 4 * cnt + cnt * cap * 2 + cnt * mm);
    double* dd = ws_dev_as<double>(WS_PM_DBL, cnt * stride + cnt * cap * sstride + (tableau ? cnt * tsize : 0));
    if (!di || !dd) return LPX_E_CUDA;
    int *dsrc = di, *dend = di + cnt, *dns = di + 2 * cnt, *dnp = di + 3 * cnt, *dspv = di + 4 * cnt,
        *dbasis = dspv + cnt * cap * 2;
    double *dpay = dd, *dseg = dd + cnt * stride, *dT = tableau ? dseg + cnt * cap * sstride : nullptr;
    LPX_CUDA(cudaMemcpyAsync(dpay, payload, cnt * stride * 8, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemsetAsync(dsrc, 0, cnt * 4, s));
    rc = param_launch(kind, count, m, n, sense, rel ? drel : nullptr, mm, dbI, dbI + 1, dbT, dsrc, dpay, seg_cap, o,
                      dend, dns, dnp, dseg, dspv, dbasis, dT, nullptr, s);
    if (rc != LPX_OK) return rc;
    auto down = [&](void* dst, const void* from, size_t bytes) {
        return dst ? cudaMemcpyAsync(dst, from, bytes, cudaMemcpyDeviceToHost, s) : cudaSuccess;
    };
    LPX_CUDA(down(end, dend, cnt * 4));
    LPX_CUDA(down(n_segments, dns, cnt * 4));
    LPX_CUDA(down(n_pivots, dnp, cnt * 4));
    LPX_CUDA(down(segments, dseg, cnt * cap * sstride * 8));
    LPX_CUDA(down(seg_pivots, dspv, cnt * cap * 2 * 4));
    LPX_CUDA(down(basis, dbasis, cnt * mm * 4));
    LPX_CUDA(down(tableau, dT, cnt * tsize * 8));
    LPX_CUDA(cudaStreamSynchronize(s));
    return LPX_OK;
}

}  // extern "C"
