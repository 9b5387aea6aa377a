// lpx_sens.cu — sensitivity report kernels and their entry points: lpx_sensitivity_stride,
// lpx_sensitivity_batched_dev (final tableaux already on the device), the session launcher behind
// lpx_session_sensitivity, and the two-phase session launcher behind lpx_session_two_phase_sensitivity.  lpx_primal_solve_sensitivity_batched (lpx_cta.cu) runs the batched kernel per chunk.
#include <algorithm>
#include <vector>

#include "lpx_runtime.hpp"
#include "lpx_sens.cuh"
#include "lpx_stream.hpp"

namespace lpx {

struct SensBatch {
    int m, n, mm, W, sense;
    const int* rel;  // nullable: all rows '<='
    const double* b;
    const double* c;
    const int* status;
    const int* basis;
    const double* tableau;
    double* report;
};

#define LPX_SENS_THREADS 256

static size_t sens_smem(const SensBatch& S, bool stage) {
    const size_t flags = ((size_t)S.W + S.m) * 4;
    return (stage ? (size_t)(S.mm + 1) * S.W * 8 : 0) + flags;
}

// One CTA per LP.  With STAGE the tableau is first copied into shared memory with coalesced loads; without it
// (tableaux larger than shared memory) the same code reads global memory.  Warps take the m constraints (a
// column reduction over the m' rows, lanes over rows) and then the n decision variables (a row reduction over the
// columns, lanes over columns).
template <bool STAGE>
__global__ void __launch_bounds__(LPX_SENS_THREADS) sens_batched_kernel(SensBatch S) {
    extern __shared__ __align__(16) unsigned char sens_smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = LPX_SENS_THREADS / 32;
    const int m = S.m, n = S.n, mm = S.mm, W = S.W;
    const size_t stride = 4 * (size_t)m + 3 * (size_t)n;
    const long long k = blockIdx.x;
    double* rep = S.report + k * stride;
    if (S.status[k] != LPX_OPTIMAL) {
        for (size_t e = tid; e < stride; e += LPX_SENS_THREADS) rep[e] = sens_nan();
        return;
    }
    const size_t tsize = (size_t)(mm + 1) * W;
    const double* Tg = S.tableau + k * tsize;
    double* Ts = reinterpret_cast<double*>(sens_smem_raw);
    int* rowof = reinterpret_cast<int*>(sens_smem_raw + (STAGE ? tsize * 8 : 0));
    int* rmap = rowof + W;
    if (STAGE) {
        size_t e = tid;
        for (; e + 3 * LPX_SENS_THREADS < tsize; e += 4 * LPX_SENS_THREADS) {
            const double v0 = Tg[e], v1 = Tg[e + LPX_SENS_THREADS], v2 = Tg[e + 2 * LPX_SENS_THREADS],
                         v3 = Tg[e + 3 * LPX_SENS_THREADS];
            Ts[e] = v0;
            Ts[e + LPX_SENS_THREADS] = v1;
            Ts[e + 2 * LPX_SENS_THREADS] = v2;
            Ts[e + 3 * LPX_SENS_THREADS] = v3;
        }
        for (; e < tsize; e += LPX_SENS_THREADS) Ts[e] = Tg[e];
    }
    const double* T = STAGE ? Ts : Tg;
    for (int j = tid; j < W; j += LPX_SENS_THREADS) rowof[j] = -1;
    if (tid == 0) {
        int r = 0;
        for (int i = 0; i < m; i++) {
            const bool eq = S.rel && S.rel[i] == 2;
            rmap[i] = eq ? -r - 1 : r;
            r += eq ? 2 : 1;
        }
    }
    __syncthreads();
    const int* basis = S.basis + k * mm;
    for (int r = tid; r < mm; r += LPX_SENS_THREADS) rowof[basis[r]] = r;
    __syncthreads();

    const double* z = T + (size_t)mm * W;
    const double* bk = S.b + k * m;
    const double* ck = S.c + k * n;
    for (int i = warp; i < m; i += nwarps) {
        const int e = rmap[i], c1 = n + sens_row1(e), c2 = c1 + 1;
        SensBest lo = sens_empty(), hi = sens_empty();
        for (int r = lane; r < mm; r += 32) {
            const double* Tr = T + (size_t)r * W;
            const double g = e < 0 ? __dsub_rn(Tr[c1], Tr[c2]) : Tr[c1];
            sens_rhs_candidate(lo, hi, Tr[W - 1], g, r);
        }
        lo = sens_warp_reduce<true>(lo);
        hi = sens_warp_reduce<false>(hi);
        if (lane == 0) {
            const double u = e < 0 ? __dsub_rn(z[c1], z[c2]) : z[c1];
            const int rs = rowof[c1];
            const double slack = rs >= 0 ? T[(size_t)rs * W + W - 1] : 0.0;
            sens_write_constraint(rep, m, i, S.sense, u, slack, lo, hi, bk[i]);
        }
    }
    for (int j = warp; j < n; j += nwarps) sens_variable_warp(T, W, W, mm, n, m, j, S.sense, rowof, ck[j], rep);
}

int sens_launch_batched(int count, int m, int n, int mm, int sense, const int* rel, const double* b, const double* c,
                        const int* status, const int* basis, const double* tableau, double* report,
                        cudaStream_t stream) {
    if (count <= 0) return LPX_OK;
    SensBatch S;
    S.m = m;
    S.n = n;
    S.mm = mm;
    S.W = n + mm + 1;
    S.sense = sense;
    S.rel = rel;
    S.b = b;
    S.c = c;
    S.status = status;
    S.basis = basis;
    S.tableau = tableau;
    S.report = report;
    const bool stage = sens_smem(S, true) <= (size_t)max_smem_optin();
    const size_t smem = sens_smem(S, stage);
    if (smem > (size_t)max_smem_optin()) {
        set_error("sensitivity: problem too wide for the per-LP kernel (column flags exceed shared memory)");
        return LPX_E_CAPACITY;
    }
    auto kfn = stage ? sens_batched_kernel<true> : sens_batched_kernel<false>;
    LPX_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kfn<<<count, LPX_SENS_THREADS, smem, stream>>>(S);
    LPX_CUDA(cudaGetLastError());
    count_launch();
    return LPX_OK;
}

// ---- session: one large LP in HBM, rows ld doubles apart ---------------------------------------------------

struct SensSession {
    int m, n, mm, W, sense, chunk_rows, nchunks;
    int ld;
    const int* rmap;  // m entries, encoded as sens_row1 reads them
    const double* b;
    const double* c;
    const int* basis;
    const double* T;
    int* rowof;         // W
    SensBest* partial;  // nchunks x m x {lo, hi}
    double* report;     // device, one stride
};

__global__ void __launch_bounds__(1024) sens_session_rowof_kernel(SensSession S) {
    for (int j = threadIdx.x; j < S.W; j += 1024) S.rowof[j] = -1;
    __syncthreads();
    for (int r = threadIdx.x; r < S.mm; r += 1024) S.rowof[S.basis[r]] = r;
}

// Row pass: one warp per decision variable, coalesced along its basic row and the z-row.
__global__ void __launch_bounds__(256) sens_session_row_kernel(SensSession S) {
    const int j = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (j >= S.n) return;
    sens_variable_warp(S.T, S.ld, S.W, S.mm, S.n, S.m, j, S.sense, S.rowof, S.c[j], S.report);
}

// Column pass over the slack block: thread per constraint (adjacent threads read adjacent slack columns), one
// chunk of chunk_rows rows per blockIdx.y; each chunk leaves its (value, index) partials for the combine.
__global__ void __launch_bounds__(256) sens_session_col_kernel(SensSession S) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= S.m) return;
    const int e = S.rmap[i], c1 = S.n + sens_row1(e), c2 = c1 + 1;
    const int r0 = blockIdx.y * S.chunk_rows, r1 = min(S.mm, r0 + S.chunk_rows);
    SensBest lo = sens_empty(), hi = sens_empty();
    for (int r = r0; r < r1; r++) {
        const double* Tr = S.T + (size_t)r * S.ld;
        const double g = e < 0 ? __dsub_rn(Tr[c1], Tr[c2]) : Tr[c1];
        sens_rhs_candidate(lo, hi, Tr[S.W - 1], g, r);
    }
    SensBest* p = S.partial + 2 * ((size_t)blockIdx.y * S.m + i);
    p[0] = lo;
    p[1] = hi;
}

// Combine of the column-pass partials (chunks in row order, same tie rule), plus shadow price and slack.
__global__ void __launch_bounds__(256) sens_session_combine_kernel(SensSession S) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= S.m) return;
    SensBest lo = sens_empty(), hi = sens_empty();
    for (int ch = 0; ch < S.nchunks; ch++) {
        const SensBest* p = S.partial + 2 * ((size_t)ch * S.m + i);
        sens_pick<true>(lo, p[0]);
        sens_pick<false>(hi, p[1]);
    }
    const int e = S.rmap[i], c1 = S.n + sens_row1(e), c2 = c1 + 1;
    const double* z = S.T + (size_t)S.mm * S.ld;
    const double u = e < 0 ? __dsub_rn(z[c1], z[c2]) : z[c1];
    const int rs = S.rowof[c1];
    const double slack = rs >= 0 ? S.T[(size_t)rs * S.ld + S.W - 1] : 0.0;
    sens_write_constraint(S.report, S.m, i, S.sense, u, slack, lo, hi, S.b[i]);
}

size_t sens_session_partial_bytes(int m, int mm) {
    const int chunks = (mm + LPX_SENS_CHUNK_ROWS - 1) / LPX_SENS_CHUNK_ROWS;
    return (size_t)chunks * m * 2 * sizeof(SensBest);
}

int sens_session_launch(int m, int n, int mm, size_t ld, int sense, const int* rmap, const double* b, const double* c,
                        const int* basis, const double* T, int* rowof, void* partial, double* report,
                        cudaStream_t stream) {
    SensSession S;
    S.m = m;
    S.n = n;
    S.mm = mm;
    S.W = n + mm + 1;
    S.sense = sense;
    S.chunk_rows = LPX_SENS_CHUNK_ROWS;
    S.nchunks = (mm + LPX_SENS_CHUNK_ROWS - 1) / LPX_SENS_CHUNK_ROWS;
    S.ld = (int)ld;
    S.rmap = rmap;
    S.b = b;
    S.c = c;
    S.basis = basis;
    S.T = T;
    S.rowof = rowof;
    S.partial = static_cast<SensBest*>(partial);
    S.report = report;
    const unsigned cblocks = (unsigned)((m + 255) / 256);
    sens_session_rowof_kernel<<<1, 1024, 0, stream>>>(S);
    sens_session_row_kernel<<<(n + 7) / 8, 256, 0, stream>>>(S);
    sens_session_col_kernel<<<dim3(cblocks, (unsigned)S.nchunks, 1), 256, 0, stream>>>(S);
    sens_session_combine_kernel<<<cblocks, 256, 0, stream>>>(S);
    LPX_CUDA(cudaGetLastError());
    count_launch(4);
    return LPX_OK;
}

// ---- two-phase session: the report of "Sensitivity analysis of a two-phase result" on the full-width tableau -------
// (objective row m, W = the session's width).  info = flip | slk | art, m ints each, as the session's open wrote them.

struct TwoPhaseSensRows {
    const int* flip;
    const int* slk;
    const int* art;
    int ns;  // n + s: columns from ns to W - 2 are artificials
};

__global__ void __launch_bounds__(1024) tp_sens_rowof_kernel(SensSession S, int ns) {
    for (int j = threadIdx.x; j < S.W; j += 1024) S.rowof[j] = j < ns ? -1 : S.m;  // never in a cost range
    __syncthreads();
    for (int r = threadIdx.x; r < S.mm; r += 1024) S.rowof[S.basis[r]] = r;
}

// Column pass over the unit columns u_i: thread per constraint, one chunk of chunk_rows rows per blockIdx.y.  A row
// whose basic variable is an artificial (a redundant row) bounds both sides.
__global__ void __launch_bounds__(256) tp_sens_col_kernel(SensSession S, TwoPhaseSensRows R) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= S.m) return;
    const int u = R.art[i] >= 0 ? R.art[i] : R.slk[i];
    const bool f = R.flip[i] != 0;
    const int r0 = blockIdx.y * S.chunk_rows, r1 = min(S.mm, r0 + S.chunk_rows);
    SensBest lo = sens_empty(), hi = sens_empty();
    for (int r = r0; r < r1; r++) {
        const double* Tr = S.T + (size_t)r * S.ld;
        const double g = sens_sign(Tr[u], f);
        if (S.basis[r] < R.ns) sens_rhs_candidate(lo, hi, Tr[S.W - 1], g, r);
        else sens_rhs_candidate_both(lo, hi, Tr[S.W - 1], g, r);
    }
    SensBest* p = S.partial + 2 * ((size_t)blockIdx.y * S.m + i);
    p[0] = lo;
    p[1] = hi;
}

// Combine of the chunks in row order, plus shadow price and slack.
__global__ void __launch_bounds__(256) tp_sens_combine_kernel(SensSession S, TwoPhaseSensRows R) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= S.m) return;
    SensBest lo = sens_empty(), hi = sens_empty();
    for (int ch = 0; ch < S.nchunks; ch++) {
        const SensBest* p = S.partial + 2 * ((size_t)ch * S.m + i);
        sens_pick<true>(lo, p[0]);
        sens_pick<false>(hi, p[1]);
    }
    const int u = R.art[i] >= 0 ? R.art[i] : R.slk[i];
    const double* z = S.T + (size_t)S.mm * S.ld;
    const int rs = R.slk[i] >= 0 ? S.rowof[R.slk[i]] : -1;
    const double slack = rs >= 0 ? S.T[(size_t)rs * S.ld + S.W - 1] : 0.0;
    sens_write_constraint(S.report, S.m, i, S.sense, sens_sign(z[u], R.flip[i] != 0), slack, lo, hi, S.b[i]);
}

int tp_sens_session_launch(int m, int n, int ns, int W, size_t ld, int sense, const int* info, const double* b,
                           const double* c, const int* basis, const double* T, int* rowof, void* partial,
                           double* report, cudaStream_t stream) {
    SensSession S;
    S.m = m;
    S.n = n;
    S.mm = m;
    S.W = W;
    S.sense = sense;
    S.chunk_rows = LPX_SENS_CHUNK_ROWS;
    S.nchunks = (m + LPX_SENS_CHUNK_ROWS - 1) / LPX_SENS_CHUNK_ROWS;
    S.ld = (int)ld;
    S.rmap = nullptr;
    S.b = b;
    S.c = c;
    S.basis = basis;
    S.T = T;
    S.rowof = rowof;
    S.partial = static_cast<SensBest*>(partial);
    S.report = report;
    const TwoPhaseSensRows R{info, info + m, info + 2 * m, ns};
    const unsigned cblocks = (unsigned)((m + 255) / 256);
    tp_sens_rowof_kernel<<<1, 1024, 0, stream>>>(S, ns);
    sens_session_row_kernel<<<(n + 7) / 8, 256, 0, stream>>>(S);
    tp_sens_col_kernel<<<dim3(cblocks, (unsigned)S.nchunks, 1), 256, 0, stream>>>(S, R);
    tp_sens_combine_kernel<<<cblocks, 256, 0, stream>>>(S, R);
    LPX_CUDA(cudaGetLastError());
    count_launch(4);
    return LPX_OK;
}

}  // namespace lpx

using namespace lpx;

extern "C" {

size_t lpx_sensitivity_stride(int m, int n) {
    if (m < 0 || n < 0) return 0;
    return 4 * (size_t)m + 3 * (size_t)n;
}

int lpx_sensitivity_batched_dev(int count, int m, int n, int sense, const int* rel, const double* b, const double* c,
                                const int* status, const int* basis, const double* tableau, double* report,
                                void* stream) {
    if (count < 0 || m < 1 || n < 1 || (sense != 0 && sense != 1) || !b || !c || !status || !basis || !tableau ||
        !report) {
        set_error("lpx_sensitivity_batched_dev: bad arguments");
        return LPX_E_BAD_ARGS;
    }
    int rc = ensure_device();
    if (rc != LPX_OK) return rc;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    // rel is a device pointer; the tableau shape needs the EQ count on the host
    int mm = m;
    if (rel) {
        std::vector<int> hrel(m);
        LPX_CUDA(cudaMemcpyAsync(hrel.data(), rel, (size_t)m * 4, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
        LPX_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
        for (int i = 0; i < m; i++) mm += hrel[i] == 2;
    }
    return sens_launch_batched(count, m, n, mm, sense, rel, b, c, status, basis, tableau, report, (cudaStream_t)stream);
}

}  // extern "C"
