// lpx_reopt.cu — re-optimization of optimal Primal Simplex results (include/lpx.h, "Re-optimization"): what-if
// queries that change b or c, add a constraint or add a variable, re-solved warm from the base's final tableau.
// The host side only sizes the call, builds one warm record per query (which base, which kind) and launches
// cta_simplex_kernel, whose warm prologue builds each query's tableau straight from its base tableau
// (cta_reopt_build, lpx_cta.cuh) and then runs the kind's loop: one read of the base tableau plus the query's pivots.
#include <cstring>
#include <vector>

#include "lpx_cta.cuh"
#include "lpx_runtime.hpp"

namespace lpx {

static int expanded(int m, const int* rel) {
    int mm = 0;
    for (int i = 0; i < m; i++) mm += (rel && rel[i] == 2) ? 2 : 1;
    return mm;
}

static bool known_kind(int kind) { return kind >= LPX_REOPT_RHS && kind <= LPX_REOPT_COL; }

// query q reads base src[q] (q without a map)
__global__ void reopt_records_kernel(int count, int kind, const int* src, const int* base_status, const int* base_basis,
                                     const double* base_T, long long src_tsize, int mm, double* work,
                                     long long out_tsize, WarmNode* rec) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= count) return;
    const long long s = src ? src[q] : q;
    WarmNode w;
    w.T = base_T + s * src_tsize;
    w.basis = base_basis + s * mm;
    w.out_T = work ? work + (size_t)q * out_tsize : nullptr;
    w.out_basis = nullptr;
    w.val = 0.0;
    w.rows = mm + 1;
    w.var = -1;
    w.side = 0;
    w.kind = kind;
    w.base_status = base_status[s];
    rec[q] = w;
}

// The launch behind both entry points; rel / mm already known on the host, payload checked.
static int reopt_launch(int kind, int count, int m, int n, int sense, const int* rel, int mm, const int* base_status,
                        const int* base_basis, const double* base_T, const int* src, const double* payload,
                        const lpx_options& o, int* status, int* n_pivots, int* pivots, int pivots_cap, int* basis,
                        double* x, double* z, double* tableau, unsigned long long* total_pivots, cudaStream_t stream) {
    const int grow_rows = kind == LPX_REOPT_ROW, grow_cols = kind == LPX_REOPT_ROW || kind == LPX_REOPT_COL;
    const int rows = mm + 1 + grow_rows, cols = n + mm + 1 + grow_cols;
    const bool fits = cta_fits_smem(rows, cols);
    if (o.kernel == LPX_KERNEL_CTA_SMEM && !fits) {
        set_error("re-optimization: the query tableau does not fit in shared memory (LPX_KERNEL_CTA_SMEM forced)");
        return LPX_E_CAPACITY;
    }
    const bool smem = fits && o.kernel != LPX_KERNEL_CTA_GLOBAL;
    if (count == 0) return LPX_OK;
    const long long tsize = (long long)rows * cols;
    double* work = nullptr;  // the global-memory build works in the output tableau, or in scratch without one
    if (!smem) {
        work = tableau ? tableau : ws_dev_as<double>(WS_SCRATCH, (size_t)count * tsize);
        if (!work) return LPX_E_CUDA;
    }
    WarmNode* rec = ws_dev_as<WarmNode>(WS_RO_REC, count);
    if (!rec) return LPX_E_CUDA;
    reopt_records_kernel<<<(count + 127) / 128, 128, 0, stream>>>(count, kind, src, base_status, base_basis, base_T,
                                                                  (long long)(mm + 1) * (n + mm + 1), mm, work, tsize,
                                                                  rec);
    LPX_CUDA(cudaGetLastError());
    count_launch();

    CtaBatch B;
    std::memset(&B, 0, sizeof B);
    B.rel = rel;
    B.m_in = m;
    B.n = kind == LPX_REOPT_COL ? n + 1 : n;
    B.sense = sense;
    B.m_base = mm;
    B.max_iter = o.max_iterations;
    B.max_rows = rows;
    B.max_width = cols;
    B.scratch = work;
    B.scratch_stride = tsize;
    B.status = status;
    B.n_pivots = n_pivots;
    B.pivots = pivots_cap > 0 ? pivots : nullptr;
    B.pivots_cap = pivots_cap;
    B.basis = basis;
    B.basis_stride = rows - 1;
    B.x = x;
    B.z = z;
    B.tableau = tableau;
    B.tableau_stride = tsize;
    B.total_pivots = total_pivots;
    B.warm = rec;
    B.reopt_payload = payload;
    B.reopt_stride = (long long)lpx_reopt_payload_stride(kind, m, n);
    return cta_launch(B, count, smem ? LPX_KERNEL_CTA_SMEM : LPX_KERNEL_CTA_GLOBAL, o.threads, stream, nullptr);
}

static int check_kernel(const lpx_options& o) {
    if (o.kernel != LPX_KERNEL_AUTO && o.kernel != LPX_KERNEL_CTA_SMEM && o.kernel != LPX_KERNEL_CTA_GLOBAL) {
        set_error("re-optimization runs on the per-CTA kernels: opt.kernel must be AUTO, CTA_SMEM or CTA_GLOBAL");
        return LPX_E_BAD_ARGS;
    }
    return LPX_OK;
}

static int check_row_rel(const double* rels, int count) {
    for (int q = 0; q < count; q++)
        if (rels[q] != 0.0 && rels[q] != 1.0) {
            set_error("re-optimization: a ROW query's rel must be 0 (LE) or 1 (GE)");
            return LPX_E_BAD_ARGS;
        }
    return LPX_OK;
}

}  // namespace lpx

using namespace lpx;

extern "C" {

size_t lpx_reopt_payload_stride(int kind, int m, int n) {
    if (m < 0 || n < 0) return 0;
    switch (kind) {
    case LPX_REOPT_RHS: return (size_t)m;
    case LPX_REOPT_COST: return (size_t)n;
    case LPX_REOPT_ROW: return (size_t)n + 2;
    case LPX_REOPT_COL: return (size_t)m + 1;
    default: return 0;
    }
}

int lpx_reopt_dims(int kind, int m, int n, const int* rel, int* rows, int* cols) {
    if (!known_kind(kind) || m < 1 || n < 1) {
        set_error("lpx_reopt_dims: bad arguments");
        return LPX_E_BAD_ARGS;
    }
    const int mm = expanded(m, rel);
    if (rows) *rows = mm + 1 + (kind == LPX_REOPT_ROW);
    if (cols) *cols = n + mm + 1 + (kind == LPX_REOPT_ROW || kind == LPX_REOPT_COL);
    return LPX_OK;
}

int lpx_reoptimize_batched_dev(int kind, int count, int m, int n, int sense, const int* rel, const int* base_status,
                               const int* base_basis, const double* base_tableau, const int* src, const double* payload,
                               const lpx_options* opt, int* status, int* n_pivots, int* pivots, int pivots_cap,
                               int* basis, double* x, double* z, double* tableau, unsigned long long* total_pivots,
                               void* stream) {
    if (!known_kind(kind) || count < 0 || m < 1 || n < 1 || (sense != 0 && sense != 1) || !base_status ||
        !base_basis || !base_tableau || !payload || !status || pivots_cap < 0) {
        set_error("lpx_reoptimize_batched_dev: bad arguments");
        return LPX_E_BAD_ARGS;
    }
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    int rc = check_kernel(o);
    if (rc != LPX_OK) return rc;
    if ((rc = ensure_device()) != LPX_OK) return rc;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    cudaStream_t s = (cudaStream_t)stream;
    // rel (the tableau shape) and the ROW relations are device data the host has to see
    int mm = m;
    if (rel) {
        std::vector<int> hrel(m);
        LPX_CUDA(cudaMemcpyAsync(hrel.data(), rel, (size_t)m * 4, cudaMemcpyDeviceToHost, s));
        LPX_CUDA(cudaStreamSynchronize(s));
        mm = expanded(m, hrel.data());
    }
    if (kind == LPX_REOPT_ROW && count > 0) {
        const size_t stride = lpx_reopt_payload_stride(kind, m, n);
        std::vector<double> rels(count);
        LPX_CUDA(cudaMemcpy2DAsync(rels.data(), 8, payload + n, stride * 8, 8, (size_t)count, cudaMemcpyDeviceToHost, s));
        LPX_CUDA(cudaStreamSynchronize(s));
        if ((rc = check_row_rel(rels.data(), count)) != LPX_OK) return rc;
    }
    return reopt_launch(kind, count, m, n, sense, rel, mm, base_status, base_basis, base_tableau, src, payload, o, status,
                        n_pivots, pivots, pivots_cap, basis, x, z, tableau, total_pivots, s);
}

int lpx_reoptimize(int kind, int m, int n, int sense, const double* A, const int* rel, const double* b, const double* c,
                   const lpx_options* opt, int count, const double* payload, int* base_status, int* status,
                   int* n_pivots, int* pivots, int pivots_cap, int* basis, double* x, double* z, double* tableau) {
    if (!known_kind(kind) || m < 1 || n < 1 || (sense != 0 && sense != 1) || !A || !b || !c || count < 0 ||
        (count > 0 && !payload) || pivots_cap < 0) {
        set_error("lpx_reoptimize: bad arguments");
        return LPX_E_BAD_ARGS;
    }
    if (rel)
        for (int i = 0; i < m; i++)
            if (rel[i] < 0 || rel[i] > 2) {
                set_error("bad arguments: rel[i] must be 0 (LE), 1 (GE) or 2 (EQ)");
                return LPX_E_BAD_ARGS;
            }
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    int rc = check_kernel(o);
    if (rc != LPX_OK) return rc;
    const size_t stride = lpx_reopt_payload_stride(kind, m, n);
    if (kind == LPX_REOPT_ROW) {
        std::vector<double> rels(count);
        for (int q = 0; q < count; q++) rels[q] = payload[(size_t)q * stride + n];
        if ((rc = check_row_rel(rels.data(), count)) != LPX_OK) return rc;
    }
    if ((rc = ensure_device()) != LPX_OK) return rc;
    Runtime& r = rt();
    std::lock_guard<std::recursive_mutex> lk(r.mu);
    cudaStream_t s = r.stream;
    const int mm = expanded(m, rel);
    int rows = 0, cols = 0;
    lpx_reopt_dims(kind, m, n, rel, &rows, &cols);
    const size_t cnt = (size_t)count, tsize = (size_t)rows * cols, base_tsize = (size_t)(mm + 1) * (n + mm + 1);
    const int nx = kind == LPX_REOPT_COL ? n + 1 : n;

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

    // the queries, all against base 0
    double* dpay = ws_dev_as<double>(WS_RO_PAY, cnt * stride);
    int* dsrc = ws_dev_as<int>(WS_RO_SRC, cnt);
    int* dstat = ws_dev_as<int>(WS_STATUS, cnt);
    int* dnp = ws_dev_as<int>(WS_NPIV, cnt);
    int* dpiv = pivots_cap ? ws_dev_as<int>(WS_PIVOTS, cnt * pivots_cap * 2) : nullptr;
    int* dbasis = ws_dev_as<int>(WS_BASIS, cnt * (rows - 1));
    double* dx = ws_dev_as<double>(WS_X, cnt * nx);
    double* dz = ws_dev_as<double>(WS_Z, cnt);
    double* dT = tableau ? ws_dev_as<double>(WS_TABLEAU, cnt * tsize) : nullptr;
    if (!dpay || !dsrc || !dstat || !dnp || (pivots_cap && !dpiv) || !dbasis || !dx || !dz || (tableau && !dT))
        return LPX_E_CUDA;
    LPX_CUDA(cudaMemcpyAsync(dpay, payload, cnt * stride * 8, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemsetAsync(dsrc, 0, cnt * 4, s));
    if (dpiv) LPX_CUDA(cudaMemsetAsync(dpiv, 0xff, cnt * pivots_cap * 8, s));  // unused entries read -1
    rc = reopt_launch(kind, count, m, n, sense, rel ? drel : nullptr, mm, dbI, dbI + 1, dbT, dsrc, dpay, o, dstat, dnp,
                      dpiv, pivots_cap, dbasis, dx, dz, dT, nullptr, s);
    if (rc != LPX_OK) return rc;
    if (status) LPX_CUDA(cudaMemcpyAsync(status, dstat, cnt * 4, cudaMemcpyDeviceToHost, s));
    if (n_pivots) LPX_CUDA(cudaMemcpyAsync(n_pivots, dnp, cnt * 4, cudaMemcpyDeviceToHost, s));
    if (pivots && dpiv) LPX_CUDA(cudaMemcpyAsync(pivots, dpiv, cnt * pivots_cap * 8, cudaMemcpyDeviceToHost, s));
    if (basis) LPX_CUDA(cudaMemcpyAsync(basis, dbasis, cnt * (rows - 1) * 4, cudaMemcpyDeviceToHost, s));
    if (x) LPX_CUDA(cudaMemcpyAsync(x, dx, cnt * nx * 8, cudaMemcpyDeviceToHost, s));
    if (z) LPX_CUDA(cudaMemcpyAsync(z, dz, cnt * 8, cudaMemcpyDeviceToHost, s));
    if (tableau) LPX_CUDA(cudaMemcpyAsync(tableau, dT, cnt * tsize * 8, cudaMemcpyDeviceToHost, s));
    LPX_CUDA(cudaStreamSynchronize(s));
    return LPX_OK;
}

}  // extern "C"
