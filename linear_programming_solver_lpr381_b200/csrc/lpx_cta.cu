// lpx_cta.cu — launcher of the one-CTA-per-tableau kernels and the C-ABI entry points built on
// them: lpx_primal_solve, lpx_dual_solve, lpx_primal_solve_batched(_dev).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "lpx_cta.cuh"
#include "lpx_cta_cluster.cuh"
#include "lpx_cta_cond.cuh"
#include "lpx_runtime.hpp"
#include "lpx_stream.hpp"

namespace lpx {

bool cta_fits_smem(int max_rows, int max_width) {
    return cta_carve(max_rows, max_width, true).total <= (size_t)max_smem_optin();
}

template <int THREADS, bool SMEM_T>
static int launch_variant(const CtaBatch& B, int count, size_t smem, cudaStream_t stream) {
    auto kfn = cta_simplex_kernel<THREADS, SMEM_T>;
    LPX_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kfn<<<count, THREADS, smem, stream>>>(B);
    LPX_CUDA(cudaGetLastError());
    count_launch();
    return LPX_OK;
}

bool cta_cluster_fits(int max_rows, int max_width, int cl) {
    return cta_cluster_carve(max_rows, max_width, cl).total <= (size_t)max_smem_optin();
}

// smallest cluster (2 or 4 CTAs) whose combined shared memory holds the tableau; 0 = none
int cta_cluster_size_for(int max_rows, int max_width) {
    // (4 CTAs where 2 would do was measured slower, also at 64 registers for two CTAs per SM: 0.34-0.44 s
    // against 0.27 s on the deep levels of the C4 batch — the cluster barrier grows with the cluster.)
    static const bool prefer4 = getenv("LPX_CLUSTER4") != nullptr;  // experiment switch
    if (prefer4 && cta_cluster_fits(max_rows, max_width, 4)) return 4;
    if (cta_cluster_fits(max_rows, max_width, 2)) return 2;
    if (cta_cluster_fits(max_rows, max_width, 4)) return 4;
    return 0;
}

template <int CL>
static int launch_cluster_variant(const CtaBatch& B, int count, cudaStream_t stream) {
    auto kfn = cta_cluster_simplex_kernel<512, CL>;
    const size_t smem = cta_cluster_carve(B.max_rows, B.max_width, CL).total;
    LPX_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg;
    std::memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3((unsigned)count * CL, 1, 1);
    cfg.blockDim = dim3(512, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    LPX_CUDA(cudaLaunchKernelEx(&cfg, kfn, B));
    count_launch();
    return LPX_OK;
}

int cta_launch(const CtaBatch& B, int count, int kernel_pref, int threads_pref, cudaStream_t stream,
               bool* used_smem) {
    if (count <= 0) return LPX_OK;
    bool smem_T = cta_fits_smem(B.max_rows, B.max_width);
    if (kernel_pref == LPX_KERNEL_CTA_GLOBAL) smem_T = false;
    // Too large for one SM's shared memory: a cluster of 2 or 4 CTAs keeps it on chip
    // (lpx_cta_cluster.cuh); only beyond that does the tableau go to global memory.
    if (kernel_pref == LPX_KERNEL_CTA_CLUSTER || (kernel_pref == LPX_KERNEL_AUTO && !smem_T)) {
        const int cl = cta_cluster_size_for(B.max_rows, B.max_width);
        if (cl == 0 && kernel_pref == LPX_KERNEL_CTA_CLUSTER) {
            set_error("tableau does not fit the shared memory of a 4-CTA cluster (LPX_KERNEL_CTA_CLUSTER forced)");
            return LPX_E_CAPACITY;
        }
        if (cl) {
            if (used_smem) *used_smem = true;
            return cl == 2 ? launch_cluster_variant<2>(B, count, stream) : launch_cluster_variant<4>(B, count, stream);
        }
    }
    if (kernel_pref == LPX_KERNEL_CTA_SMEM && !smem_T) {
        set_error("tableau does not fit in shared memory (LPX_KERNEL_CTA_SMEM forced)");
        return LPX_E_CAPACITY;
    }
    if (!smem_T && !B.tableau && !B.scratch) {
        set_error("internal: global-memory tableau kernel needs scratch");
        return LPX_E_BAD_ARGS;
    }
    const size_t smem = cta_carve(B.max_rows, B.max_width, smem_T).total;
    if (smem > (size_t)max_smem_optin()) {
        set_error("problem too wide for the per-CTA kernels (work vectors exceed shared memory)");
        return LPX_E_CAPACITY;
    }
    if (used_smem) *used_smem = smem_T;
    int threads = threads_pref;
    if (threads != 128 && threads != 256 && threads != 512) {
        // small tableaux: 256; from about 8 k elements on (and for global-memory ones) 512 threads keep more
        // loads in flight and win despite the dearer barriers (measured: 64x128 2.54 -> 2.36 ms per 4096 LPs,
        // 90x120 1.89 -> 1.51 ms per 1184; tools/gpu_probe.py smemshape)
        threads = (!smem_T || (size_t)B.max_rows * B.max_width >= 8192) ? 512 : 256;
    }
    if (smem_T) {
        if (threads == 128) return launch_variant<128, true>(B, count, smem, stream);
        if (threads == 256) return launch_variant<256, true>(B, count, smem, stream);
        return launch_variant<512, true>(B, count, smem, stream);
    }
    if (threads == 128) return launch_variant<128, false>(B, count, smem, stream);
    if (threads == 256) return launch_variant<256, false>(B, count, smem, stream);
    return launch_variant<512, false>(B, count, smem, stream);
}

// condensed-tableau node kernel (lpx_cta_cond.cuh)
bool cta_condensed_fits(int max_rows, int n) { return cond_carve(max_rows, n).total <= (size_t)max_smem_optin(); }
int cta_condensed_ctas_per_sm(int rows, int n) {
    // 227 KB usable per SM, 1 KB reserved per resident CTA; 58 registers x 512 threads allow two CTAs
    const size_t per = cond_carve(rows, n).total + 1024 + 1024;  // + the kernel's static shared memory
    return (int)std::min<size_t>(2, ((size_t)228 * 1024) / per);
}
int cta_condensed_launch(const CtaBatch& B, int count, cudaStream_t stream) {
    if (count <= 0) return LPX_OK;
    const size_t smem = cond_carve(B.max_rows, B.n).total;
    if (smem > (size_t)max_smem_optin()) {
        set_error("internal: condensed tableau does not fit in shared memory");
        return LPX_E_CAPACITY;
    }
    auto kfn = B.dbg ? cta_condensed_kernel<512, true> : cta_condensed_kernel<512, false>;
    LPX_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kfn<<<count, 512, smem, stream>>>(B);
    LPX_CUDA(cudaGetLastError());
    count_launch();
    return LPX_OK;
}

static int expanded_rows(int m, const int* rel) {
    int mm = 0;
    for (int i = 0; i < m; i++) mm += (rel && rel[i] == 2) ? 2 : 1;
    return mm;
}

static int check_problem(int m, int n, int sense, const double* A, const int* rel, const double* b,
                         const double* c) {
    if (m < 1 || n < 1 || !A || !b || !c || (sense != 0 && sense != 1)) {
        set_error("bad arguments: need m >= 1, n >= 1, sense in {0,1}, non-null A, b, c");
        return LPX_E_BAD_ARGS;
    }
    if (rel)
        for (int i = 0; i < m; i++)
            if (rel[i] < 0 || rel[i] > 2) {
                set_error("bad arguments: rel[i] must be 0 (LE), 1 (GE) or 2 (EQ)");
                return LPX_E_BAD_ARGS;
            }
    return LPX_OK;
}

// One LP through the per-CTA kernels; mode 0 primal / 1 dual.
static int solve_single_cta(int mode, int m, int n, int sense, const double* A, const int* rel, const double* b,
                            const double* c, const lpx_options* opt, int* status, int* n_pivots, int* silent,
                            int* pivots, int pivots_cap, int* basis, double* x, double* z, double* tableau,
                            double* history, int history_cap) {
    Runtime& r = rt();
    const int mm = expanded_rows(m, rel);
    const int rows = mm + 1, width = n + mm + 1;
    const size_t tsize = (size_t)rows * width;
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    if (pivots_cap < 0) pivots_cap = 0;
    if (!history) history_cap = 0;

    double* dA = ws_dev_as<double>(WS_A, (size_t)m * n);
    double* db = ws_dev_as<double>(WS_B, m);
    double* dc = ws_dev_as<double>(WS_C, n);
    int* drel = ws_dev_as<int>(WS_REL, m);
    int* dstat = ws_dev_as<int>(WS_STATUS, 4);
    int* dpiv = ws_dev_as<int>(WS_PIVOTS, (size_t)std::max(pivots_cap, 1) * 2);
    int* dbasis = ws_dev_as<int>(WS_BASIS, mm);
    double* dx = ws_dev_as<double>(WS_X, n);
    double* dz = ws_dev_as<double>(WS_Z, 1);
    double* dT = ws_dev_as<double>(WS_TABLEAU, tsize);
    double* dH = history_cap ? ws_dev_as<double>(WS_HISTORY, tsize * history_cap) : nullptr;
    if (!dA || !db || !dc || !drel || !dstat || !dpiv || !dbasis || !dx || !dz || !dT || (history_cap && !dH))
        return LPX_E_CUDA;

    cudaStream_t s = r.stream;
    LPX_CUDA(cudaMemcpyAsync(dA, A, (size_t)m * n * 8, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemcpyAsync(db, b, (size_t)m * 8, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemcpyAsync(dc, c, (size_t)n * 8, cudaMemcpyHostToDevice, s));
    if (rel) LPX_CUDA(cudaMemcpyAsync(drel, rel, (size_t)m * 4, cudaMemcpyHostToDevice, s));

    CtaBatch B;
    std::memset(&B, 0, sizeof B);
    B.A = dA;
    B.b = db;
    B.c = dc;
    B.rel = rel ? drel : nullptr;
    B.m_in = m;
    B.n = n;
    B.sense = sense;
    B.m_base = mm;
    B.mode = mode;
    B.max_iter = o.max_iterations;
    B.max_rows = rows;
    B.max_width = width;
    B.status = dstat;
    B.n_pivots = dstat + 1;
    B.silent = dstat + 2;
    B.n_history = dstat + 3;
    B.pivots = pivots_cap ? dpiv : nullptr;
    B.pivots_cap = pivots_cap;
    B.basis = dbasis;
    B.basis_stride = mm;
    B.x = dx;
    B.z = dz;
    B.tableau = dT;
    B.tableau_stride = (long long)tsize;
    B.history = dH;
    B.history_stride = (long long)(tsize * (size_t)history_cap);
    B.history_cap = history_cap;
    static const bool want_prof = getenv("LPX_CTA_PROF") != nullptr;  // measurement aid, prints to stderr
    long long* d_prof = nullptr;
    if (want_prof) {
        LPX_CUDA(cudaMalloc(&d_prof, 64));
        LPX_CUDA(cudaMemsetAsync(d_prof, 0, 64, s));
        B.dbg = d_prof;
    }
    int rc = cta_launch(B, 1, o.kernel, o.threads, s, nullptr);
    if (rc != LPX_OK) return rc;
    if (want_prof) {
        long long h[8];
        LPX_CUDA(cudaMemcpyAsync(h, d_prof, 64, cudaMemcpyDeviceToHost, s));
        LPX_CUDA(cudaStreamSynchronize(s));
        cudaFree(d_prof);
        const double np = (double)std::max(1LL, h[4]);
        fprintf(stderr, "[cta prof] %lld x %lld tableau, %lld pivots; cycles per pivot: ratios %.0f, scan %.0f, staging %.0f, "
                        "update %.0f\n", h[5], h[6], h[4], h[0] / np, h[1] / np, h[2] / np, h[3] / np);
    }

    int hstat[4] = {0, 0, 0, 0};
    LPX_CUDA(cudaMemcpyAsync(hstat, dstat, sizeof hstat, cudaMemcpyDeviceToHost, s));
    LPX_CUDA(cudaStreamSynchronize(s));
    if (status) *status = hstat[0];
    if (n_pivots) *n_pivots = hstat[1];
    if (silent) *silent = hstat[2];
    const bool solved = hstat[0] >= 0 || hstat[0] == LPX_S_ITER_LIMIT;
    if (pivots && pivots_cap)
        LPX_CUDA(cudaMemcpyAsync(pivots, dpiv, (size_t)std::min(hstat[1], pivots_cap) * 8, cudaMemcpyDeviceToHost, s));
    if (solved) {
        if (basis) LPX_CUDA(cudaMemcpyAsync(basis, dbasis, (size_t)mm * 4, cudaMemcpyDeviceToHost, s));
        if (x) LPX_CUDA(cudaMemcpyAsync(x, dx, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
        if (z) LPX_CUDA(cudaMemcpyAsync(z, dz, 8, cudaMemcpyDeviceToHost, s));
        if (tableau) LPX_CUDA(cudaMemcpyAsync(tableau, dT, tsize * 8, cudaMemcpyDeviceToHost, s));
        if (history && hstat[3] > 0)
            LPX_CUDA(cudaMemcpyAsync(history, dH, tsize * 8 * (size_t)hstat[3], cudaMemcpyDeviceToHost, s));
    }
    LPX_CUDA(cudaStreamSynchronize(s));
    return LPX_OK;
}

static void fill_uniform_batch(CtaBatch& B, int m, int n, int sense, int mm, const lpx_options& o) {
    std::memset(&B, 0, sizeof B);
    B.m_in = m;
    B.n = n;
    B.sense = sense;
    B.m_base = mm;
    B.mode = 0;
    B.max_iter = o.max_iterations;
    B.max_rows = mm + 1;
    B.max_width = n + mm + 1;
    B.strideA = (long long)m * n;
    B.strideB = m;
    B.strideC = n;
    B.basis_stride = mm;
    B.tableau_stride = (long long)(mm + 1) * (n + mm + 1);
}

// Launch of one uniform batch whose row relations are already known on the host (mm = rows after EQ
// expansion, all_le = no '>=' / '=' row): lpx_primal_solve_batched calls this per chunk without the
// device-to-host read of rel (and the stream drain that comes with it) the public _dev entry point needs.
static int batched_dev_launch(int count, int m, int n, int sense, const double* A, const int* drel, int mm, bool all_le,
                              const double* b, const double* c, const lpx_options& o, int* status, int* n_pivots,
                              int* basis, double* x, double* z, double* tableau, unsigned long long* total_pivots,
                              cudaStream_t stream) {
    if (o.kernel == LPX_KERNEL_CTA_REG && !all_le) {
        set_error("LPX_KERNEL_CTA_REG: the register-resident kernel serves all-'<=' problems only");
        return LPX_E_CAPACITY;
    }
    // an all-LE rel array is the same problem as rel == NULL: it keeps the register-resident kernel
    if (o.kernel == LPX_KERNEL_CTA_REG || (o.kernel == LPX_KERNEL_AUTO && all_le && reg_kernel_supports(m, n, mm, false)))
        return reg_launch_batched(count, m, n, sense, A, b, c, o, status, n_pivots, basis, x, z, tableau, total_pivots,
                                  stream);
    CtaBatch B;
    fill_uniform_batch(B, m, n, sense, mm, o);
    B.A = A;
    B.b = b;
    B.c = c;
    B.rel = all_le ? nullptr : drel;
    B.status = status;
    B.n_pivots = n_pivots;
    B.basis = basis;
    B.x = x;
    B.z = z;
    B.tableau = tableau;
    B.total_pivots = total_pivots;
    if (!cta_fits_smem(B.max_rows, B.max_width) || o.kernel == LPX_KERNEL_CTA_GLOBAL) {
        if (!tableau) {
            double* sc = ws_dev_as<double>(WS_SCRATCH, (size_t)count * B.tableau_stride);
            if (!sc) return LPX_E_CUDA;
            B.scratch = sc;
            B.scratch_stride = B.tableau_stride;
        }
    }
    return cta_launch(B, count, o.kernel, o.threads, stream, nullptr);
}

// lpx_primal_solve_batched(_sensitivity): host buffers through a three-stream chunk pipeline.  report (nullable):
// the sensitivity records, computed per chunk on the compute stream from the chunk's tableaux, which then stay
// in a device workspace unless `tableau` asks for them too.
static int primal_batched_pipeline(int count, int m, int n, int sense, const double* A, const int* rel,
                                   const double* b, const double* c, const lpx_options* opt, int* status,
                                   int* n_pivots, int* basis, double* x, double* z, double* tableau, double* report,
                                   long long* total_pivots) {
    int rc = check_problem(m, n, sense, A, rel, b, c);
    if (rc != LPX_OK) return rc;
    if ((rc = ensure_device()) != LPX_OK) return rc;
    Runtime& r = rt();
    std::lock_guard<std::recursive_mutex> lk(r.mu);
    if (total_pivots) *total_pivots = 0;
    if (count == 0) return LPX_OK;
    const int mm = expanded_rows(m, rel);
    const size_t tsize = (size_t)(mm + 1) * (n + mm + 1);
    const size_t cnt = (size_t)count;

    double* dA = ws_dev_as<double>(WS_A, cnt * m * n);
    double* db = ws_dev_as<double>(WS_B, cnt * m);
    double* dc = ws_dev_as<double>(WS_C, cnt * n);
    int* drel = ws_dev_as<int>(WS_REL, m);
    int* dstat = ws_dev_as<int>(WS_STATUS, cnt);
    int* dnp = ws_dev_as<int>(WS_NPIV, cnt);
    int* dbasis = ws_dev_as<int>(WS_BASIS, cnt * mm);
    double* dx = ws_dev_as<double>(WS_X, cnt * n);
    double* dz = ws_dev_as<double>(WS_Z, cnt);
    double* dT = (tableau || report) ? ws_dev_as<double>(WS_TABLEAU, cnt * tsize) : nullptr;
    const size_t rstride = lpx_sensitivity_stride(m, n);
    double* dR = report ? ws_dev_as<double>(WS_SENS, cnt * rstride) : nullptr;
    unsigned long long* dtot = ws_dev_as<unsigned long long>(WS_TOTAL, 1);
    if (!dA || !db || !dc || !drel || !dstat || !dnp || !dbasis || !dx || !dz || ((tableau || report) && !dT) ||
        (report && !dR) || !dtot)
        return LPX_E_CUDA;
    if (rel) LPX_CUDA(cudaMemcpyAsync(drel, rel, (size_t)m * 4, cudaMemcpyHostToDevice, r.h2d));
    LPX_CUDA(cudaMemsetAsync(dtot, 0, 8, r.h2d));

    // Three-stage pipeline over chunks of the batch: H2D | solve | D2H on three streams, so that
    // PCIe traffic in both directions overlaps the kernels.  The result copy is the long pole (the
    // tableaux are 1.5x the inputs), so large batches ramp the chunk size up — 1, 2, 4, 5, 5, ... 32nds —
    // and the first results start down the link after a 32nd of the upload instead of an 8th.
    const int chunks = count >= 1024 ? 8 : (count >= 64 ? 4 : 1);
    static const int ramp[9] = {0, 1, 3, 7, 12, 17, 22, 27, 32};
    auto bound = [&](int k) -> size_t { return chunks == 8 ? cnt * ramp[k] / 32 : cnt * k / chunks; };
    struct Events {  // destroyed on every return path, the LPX_CUDA early returns included
        std::vector<cudaEvent_t> ev;
        ~Events() {
            for (cudaEvent_t e : ev) cudaEventDestroy(e);
        }
        int add(cudaEvent_t* out) {
            LPX_CUDA(cudaEventCreateWithFlags(out, cudaEventDisableTiming));
            ev.push_back(*out);
            return LPX_OK;
        }
    } events;
    std::vector<cudaEvent_t> up(chunks), done(chunks);
    for (int k = 0; k < chunks; k++) {
        if ((rc = events.add(&up[k])) != LPX_OK) return rc;
        if ((rc = events.add(&done[k])) != LPX_OK) return rc;
    }
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    bool all_le = true;
    if (rel)
        for (int i = 0; i < m; i++) all_le = all_le && rel[i] == 0;
    int result = LPX_OK;
    for (int k = 0; k < chunks && result == LPX_OK; k++) {
        const size_t lo = bound(k), hi = bound(k + 1), len = hi - lo;
        if (len == 0) continue;
        LPX_CUDA(cudaMemcpyAsync(dA + lo * m * n, A + lo * m * n, len * m * n * 8, cudaMemcpyHostToDevice, r.h2d));
        LPX_CUDA(cudaMemcpyAsync(db + lo * m, b + lo * m, len * m * 8, cudaMemcpyHostToDevice, r.h2d));
        LPX_CUDA(cudaMemcpyAsync(dc + lo * n, c + lo * n, len * n * 8, cudaMemcpyHostToDevice, r.h2d));
        LPX_CUDA(cudaEventRecord(up[k], r.h2d));
        LPX_CUDA(cudaStreamWaitEvent(r.stream, up[k], 0));
        result = batched_dev_launch((int)len, m, n, sense, dA + lo * m * n, rel ? drel : nullptr, mm, all_le, db + lo * m,
                                    dc + lo * n, o, dstat + lo, dnp + lo, dbasis + lo * mm, dx + lo * n, dz + lo,
                                    dT ? dT + lo * tsize : nullptr, dtot, r.stream);
        if (result == LPX_OK && report)
            result = sens_launch_batched((int)len, m, n, mm, sense, rel ? drel : nullptr, db + lo * m, dc + lo * n,
                                         dstat + lo, dbasis + lo * mm, dT + lo * tsize, dR + lo * rstride, r.stream);
        if (result != LPX_OK) break;
        LPX_CUDA(cudaEventRecord(done[k], r.stream));
        LPX_CUDA(cudaStreamWaitEvent(r.d2h, done[k], 0));
        LPX_CUDA(cudaMemcpyAsync(status + lo, dstat + lo, len * 4, cudaMemcpyDeviceToHost, r.d2h));
        if (n_pivots) LPX_CUDA(cudaMemcpyAsync(n_pivots + lo, dnp + lo, len * 4, cudaMemcpyDeviceToHost, r.d2h));
        if (basis)
            LPX_CUDA(cudaMemcpyAsync(basis + lo * mm, dbasis + lo * mm, len * mm * 4, cudaMemcpyDeviceToHost, r.d2h));
        if (x) LPX_CUDA(cudaMemcpyAsync(x + lo * n, dx + lo * n, len * n * 8, cudaMemcpyDeviceToHost, r.d2h));
        if (z) LPX_CUDA(cudaMemcpyAsync(z + lo, dz + lo, len * 8, cudaMemcpyDeviceToHost, r.d2h));
        if (tableau)
            LPX_CUDA(cudaMemcpyAsync(tableau + lo * tsize, dT + lo * tsize, len * tsize * 8, cudaMemcpyDeviceToHost,
                                     r.d2h));
        if (report)
            LPX_CUDA(cudaMemcpyAsync(report + lo * rstride, dR + lo * rstride, len * rstride * 8, cudaMemcpyDeviceToHost,
                                     r.d2h));
    }
    unsigned long long htot = 0;
    if (result == LPX_OK) {
        cudaError_t e = cudaStreamSynchronize(r.stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(&htot, dtot, 8, cudaMemcpyDeviceToHost, r.d2h);
        if (e == cudaSuccess) e = cudaStreamSynchronize(r.d2h);
        if (e != cudaSuccess) result = cuda_fail(e, "batched pipeline sync", __FILE__, __LINE__);
    } else {
        cudaDeviceSynchronize();
    }
    if (total_pivots) *total_pivots = (long long)htot;
    return result;
}

// opt.kernel AUTO for one LP (lpx_primal_solve, lpx_dual_solve): the per-CTA kernels win while the tableau is small;
// past that a single SM cannot stream it fast enough and the whole-GPU streaming kernels take over.
static int single_auto_kernel(int mm, int n, bool want_history) {
    const size_t elems = (size_t)(mm + 1) * (n + mm + 1);
    int kernel = (cta_fits_smem(mm + 1, n + mm + 1) || elems <= (size_t)96 * 1024) ? LPX_KERNEL_CTA_SMEM
                                                                                    : LPX_KERNEL_STREAM;
    if (kernel == LPX_KERNEL_CTA_SMEM && !cta_fits_smem(mm + 1, n + mm + 1))
        kernel = cta_cluster_size_for(mm + 1, n + mm + 1) ? LPX_KERNEL_CTA_CLUSTER : LPX_KERNEL_CTA_GLOBAL;
    if (want_history && kernel == LPX_KERNEL_STREAM) kernel = LPX_KERNEL_CTA_GLOBAL;
    return kernel;
}

}  // namespace lpx

using namespace lpx;

extern "C" {

int lpx_primal_solve(int m, int n, int sense, const double* A, const int* rel, const double* b, const double* c,
                     const lpx_options* opt, int* status, int* n_pivots, int* pivots, int pivots_cap, int* basis,
                     double* x, double* z, double* tableau, double* history, int history_cap) {
    int rc = check_problem(m, n, sense, A, rel, b, c);
    if (rc != LPX_OK) return rc;
    if ((rc = ensure_device()) != LPX_OK) return rc;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    const int mm = expanded_rows(m, rel);
    int kernel = opt ? opt->kernel : LPX_KERNEL_AUTO;
    if (kernel == LPX_KERNEL_AUTO) kernel = single_auto_kernel(mm, n, history && history_cap > 0);
    if (kernel == LPX_KERNEL_STREAM)
        return stream_solve_host(m, n, sense, A, rel, b, c, opt, status, n_pivots, pivots, pivots_cap, basis, x, z,
                                 tableau, history, history_cap);
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    o.kernel = kernel;
    return solve_single_cta(0, m, n, sense, A, rel, b, c, &o, status, n_pivots, nullptr, pivots, pivots_cap, basis, x,
                            z, tableau, history, history_cap);
}

int lpx_dual_solve(int m, int n, int sense, const double* A, const int* rel, const double* b, const double* c,
                   const lpx_options* opt, int* status, int* n_pivots, int* silent_pivots, int* pivots,
                   int pivots_cap, int* basis, double* x, double* z, double* tableau, double* history,
                   int history_cap) {
    int rc = check_problem(m, n, sense, A, rel, b, c);
    if (rc != LPX_OK) return rc;
    if ((rc = ensure_device()) != LPX_OK) return rc;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    if (o.kernel == LPX_KERNEL_AUTO) o.kernel = single_auto_kernel(expanded_rows(m, rel), n, history && history_cap > 0);
    if (o.kernel == LPX_KERNEL_STREAM)
        return stream_dual_solve_host(m, n, sense, A, rel, b, c, &o, status, n_pivots, silent_pivots, pivots,
                                      pivots_cap, basis, x, z, tableau, history, history_cap);
    return solve_single_cta(1, m, n, sense, A, rel, b, c, &o, status, n_pivots, silent_pivots, pivots, pivots_cap,
                            basis, x, z, tableau, history, history_cap);
}

int lpx_primal_solve_batched_dev(int count, int m, int n, int sense, const double* A, const int* rel,
                                 const double* b, const double* c, const lpx_options* opt, int* status,
                                 int* n_pivots, int* basis, double* x, double* z, double* tableau,
                                 unsigned long long* total_pivots, void* stream) {
    if (count < 0 || m < 1 || n < 1 || !A || !b || !c || !status || (sense != 0 && sense != 1)) {
        set_error("lpx_primal_solve_batched_dev: bad arguments");
        return LPX_E_BAD_ARGS;
    }
    int rc = ensure_device();
    if (rc != LPX_OK) return rc;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    // rel is a device pointer here; the tableau shape needs it on the host
    int mm = m;
    bool all_le = true;
    if (rel) {
        std::vector<int> hrel(m);
        LPX_CUDA(cudaMemcpyAsync(hrel.data(), rel, (size_t)m * 4, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
        LPX_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
        mm = expanded_rows(m, hrel.data());
        for (int i = 0; i < m; i++) all_le = all_le && hrel[i] == 0;
    }
    return batched_dev_launch(count, m, n, sense, A, rel, mm, all_le, b, c, o, status, n_pivots, basis, x, z, tableau,
                              total_pivots, (cudaStream_t)stream);
}

int lpx_primal_solve_batched(int count, int m, int n, int sense, const double* A, const int* rel, const double* b,
                             const double* c, const lpx_options* opt, int* status, int* n_pivots, int* basis,
                             double* x, double* z, double* tableau, long long* total_pivots) {
    if (count < 0 || !status) {
        set_error("lpx_primal_solve_batched: bad arguments");
        return LPX_E_BAD_ARGS;
    }
    return primal_batched_pipeline(count, m, n, sense, A, rel, b, c, opt, status, n_pivots, basis, x, z, tableau, nullptr,
                                   total_pivots);
}

int lpx_primal_solve_sensitivity_batched(int count, int m, int n, int sense, const double* A, const int* rel,
                                         const double* b, const double* c, const lpx_options* opt, int* status,
                                         int* n_pivots, int* basis, double* x, double* z, double* report,
                                         long long* total_pivots) {
    if (count < 0 || !status || !report) {
        set_error("lpx_primal_solve_sensitivity_batched: bad arguments");
        return LPX_E_BAD_ARGS;
    }
    return primal_batched_pipeline(count, m, n, sense, A, rel, b, c, opt, status, n_pivots, basis, x, z, nullptr, report,
                                   total_pivots);
}

}  // extern "C"
