// lpx_twophase.cu — two-phase Primal Simplex (include/lpx.h, "Two-phase Simplex"), one CTA per LP: the normalised
// tableau with its slack and artificial columns and the Phase I row is built in the CTA from (A, b, c, rel); Phase I,
// the feasibility test, the drive-out of basic artificials and Phase II all run without leaving it.
// oracle/orc_twophase.cpp restates the definition as sequential loops.
//
// The loops are written here from the helpers cta_simplex_kernel uses (warp_argmin_below, cta_stage_ratios,
// warp_margin_scan_staged, cta_pivot) rather than as a branch of that kernel, which keeps its register allocation
// (DESIGN §4.12 gives the same reason for the cutting-plane kernel).
//
// two_phase_sens_kernel is the same solve with the sensitivity report of include/lpx.h ("Sensitivity analysis of a
// two-phase result") as its epilogue, read from the full-width tableau before the CTA ends: the artificial columns
// hold B^-1 e_i of the rows whose unit column they are, and the compact output tableau drops them.
#include <cstring>
#include <vector>

#include "lpx_cta.cuh"
#include "lpx_runtime.hpp"
#include "lpx_sens.cuh"

namespace lpx {

struct TwoPhaseBatch {
    const double* A;  // [count][m][n]
    const double* b;  // [count][m]
    const double* c;  // [count][n]
    const int* rel;   // device, nullable = all LE; shared by the batch
    int m, n, sense;
    int s;            // slack columns: the non-EQ rows
    int max_width;    // n + s + m + 1: the widest tableau (every row with an artificial)
    int max_iter;
    int* status;
    int* phase1;      // nullable, as every output below
    int* n_pivots;
    int* pivots;      // [pivots_cap][2] per LP
    int pivots_cap;
    int* basis;       // [m] per LP
    double* x;        // [n] per LP
    double* z;
    double* tableau;  // [m + 1][n + s + 1] per LP
    double* work;     // global-memory tableaux (!SMEM_T), stride (m + 2) * max_width
    unsigned long long* total_pivots;
};

// The report of one OPTIMAL LP from its final full-width tableau T (rows ld doubles apart, objective row m, RHS
// column W - 1).  rowof takes W ints of scratch that is dead after the solve; sbasis / flip / slk / art as the solve
// left them.  Constraints: one warp per row i, lanes over the rows r (column reduction along the unit column u_i);
// decision variables: one warp per variable, lanes over the columns (sens_variable_warp).
template <int THREADS>
__device__ __forceinline__ void two_phase_report(const double* T, int ld, int m, int n, int ns, int W, int sense,
                                                 const int* sbasis, const int* flip, const int* slk, const int* art,
                                                 int* rowof, const double* bi, const double* ci, double* rep) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = THREADS / 32;
    const int rhs = W - 1;
    for (int j = tid; j < W; j += THREADS) rowof[j] = j < ns ? -1 : m;  // an artificial never enters a cost range
    __syncthreads();
    for (int r = tid; r < m; r += THREADS) rowof[sbasis[r]] = r;
    __syncthreads();
    const double* z = T + (size_t)m * ld;
    for (int i = warp; i < m; i += NW) {
        const int u = art[i] >= 0 ? art[i] : slk[i];
        const bool f = flip[i] != 0;
        SensBest lo = sens_empty(), hi = sens_empty();
        for (int r = lane; r < m; r += 32) {
            const double* Tr = T + (size_t)r * ld;
            const double g = sens_sign(Tr[u], f);
            if (sbasis[r] < ns) sens_rhs_candidate(lo, hi, Tr[rhs], g, r);
            else sens_rhs_candidate_both(lo, hi, Tr[rhs], g, r);
        }
        lo = sens_warp_reduce<true>(lo);
        hi = sens_warp_reduce<false>(hi);
        if (lane == 0) {
            const int rs = slk[i] >= 0 ? rowof[slk[i]] : -1;
            const double slack = rs >= 0 ? T[(size_t)rs * ld + rhs] : 0.0;
            sens_write_constraint(rep, m, i, sense, sens_sign(z[u], f), slack, lo, hi, bi[i]);
        }
    }
    for (int j = warp; j < n; j += NW) sens_variable_warp(T, ld, W, m, n, m, j, sense, rowof, ci[j], rep);
}

// REPORT: write the sensitivity record of LP p to report + p * (4m + 3n) (NaNs unless OPTIMAL).
template <int THREADS, bool SMEM_T, bool REPORT>
__device__ __forceinline__ void two_phase_body(const TwoPhaseBatch& P, double* report) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = THREADS / 32;
    const int p = blockIdx.x;
    const int m = P.m, n = P.n, ns = n + P.s, rows = m + 2;  // ns: the structural and slack columns

    const CtaCarve cv = cta_carve(rows, P.max_width, SMEM_T);
    double* prow = reinterpret_cast<double*>(smem_raw + cv.prow);
    double* fcol = reinterpret_cast<double*>(smem_raw + cv.fcol);
    int* art = reinterpret_cast<int*>(smem_raw + cv.rsrc);   // artificial column of each row, -1 if none
    int* flip = reinterpret_cast<int*>(smem_raw + cv.rsgn);  // 1: the row is negated (b_i < 0)
    int* slk = reinterpret_cast<int*>(smem_raw + cv.zc);     // slack column of each row, -1 for EQ
    int* sbasis = reinterpret_cast<int*>(smem_raw + cv.basis);
    int* ctl = reinterpret_cast<int*>(smem_raw + cv.ctl);
    double* dsh = reinterpret_cast<double*>(smem_raw + cv.red);  // [0]: S, the artificial rows' normalised b

    const double* Ai = P.A + (size_t)p * m * n;
    const double* bi = P.b + (size_t)p * m;
    const double* ci = P.c + (size_t)p * n;

    // ---- normalisation and column numbering: slack / artificial indices by ballot prefix over the rows; S summed
    // in row order by one lane (fcol holds the normalised b until the first pivot) ------------------------------------
    if (warp == 0) {
        int sk = n, ak = ns;
        for (int base = 0; base < m; base += 32) {
            const int i = base + lane;
            int rl = 0, f = 0;
            double bv = 0.0;
            if (i < m) {
                rl = P.rel ? P.rel[i] : 0;
                bv = bi[i];
                f = bv < 0.0;
            }
            const int rn = (f && rl != 2) ? 1 - rl : rl;  // the relation after normalisation
            const unsigned below = (1u << lane) - 1u;
            const unsigned hs = __ballot_sync(0xffffffffu, i < m && rl != 2);
            const unsigned ha = __ballot_sync(0xffffffffu, i < m && rn != 0);
            if (i < m) {
                flip[i] = f;
                slk[i] = rl != 2 ? sk + __popc(hs & below) : -1;
                art[i] = rn != 0 ? ak + __popc(ha & below) : -1;
                fcol[i] = f ? dneg(bv) : bv;
            }
            sk += __popc(hs);
            ak += __popc(ha);
        }
        __syncwarp();
        if (lane == 0) {
            double S = 0.0;
            for (int i = 0; i < m; i++)
                if (art[i] >= 0) S = __dadd_rn(S, fcol[i]);
            ctl[0] = ak - ns;
            dsh[0] = S;
        }
    }
    __syncthreads();
    const int W = ns + ctl[0] + 1, rhs = W - 1, ld = SMEM_T ? ((W + 1) & ~1) : W;
    double* T = SMEM_T ? reinterpret_cast<double*>(smem_raw + cv.T) : P.work + (size_t)p * rows * P.max_width;

    // ---- rows 0..m: the normalised constraints and the objective row as BuildTableau writes it ----------------------
    for (int i = warp; i <= m; i += NW) {
        double* Ti = T + (size_t)i * ld;
        if (i < m) {
            const bool f = flip[i] != 0;
            const int sc = slk[i], ac = art[i];
            const double sv = ac >= 0 ? -1.0 : 1.0;  // a row with both a slack and an artificial is GE
            const double* Ar = Ai + (size_t)i * n;
            for (int j = lane; j < W; j += 32) {
                double v;
                if (j < n) v = f ? dneg(Ar[j]) : Ar[j];
                else if (j == rhs) v = f ? dneg(bi[i]) : bi[i];
                else if (j == sc) v = sv;
                else if (j == ac) v = 1.0;
                else v = 0.0;
                Ti[j] = v;
            }
        } else {
            for (int j = lane; j < W; j += 32) {
                double v = 0.0;
                if (j < n) {
                    double cj = ci[j];
                    if (P.sense == 1) cj = dneg(cj);  // Min -> Max
                    v = dneg(cj);                     // T[m,j] = -C[j]
                }
                Ti[j] = v;
            }
        }
    }
    for (int i = tid; i < m; i += THREADS) sbasis[i] = art[i] >= 0 ? art[i] : slk[i];
    __syncthreads();
    // ---- row m+1: the artificial rows subtracted from +0 in row order, on the non-artificial columns and the RHS -----
    {
        double* wrow = T + (size_t)(m + 1) * ld;
        for (int j = tid; j < W; j += THREADS) {
            double v = 0.0;
            if (j < ns || j == rhs)
                for (int i = 0; i < m; i++)
                    if (art[i] >= 0) v = __dsub_rn(v, T[(size_t)i * ld + j]);
            wrow[j] = v;
        }
        if (ld > W)
            for (int i = tid; i < rows; i += THREADS) T[(size_t)i * ld + W] = 0.0;  // pad column
    }
    __syncthreads();

    int n_piv = 0, p1 = 0;
    int* plog = P.pivots ? P.pivots + (size_t)p * P.pivots_cap * 2 : nullptr;
    auto pivot_on = [&](int l, int e, int nrows) {
        cta_pivot<THREADS, SMEM_T>(T, ld, nrows, W, l, e, prow, fcol);
        if (tid == 0) {
            sbasis[l] = e;
            if (plog && n_piv < P.pivots_cap) {
                plog[2 * n_piv] = e;
                plog[2 * n_piv + 1] = l;
            }
        }
        n_piv++;
    };
    // Primal Simplex on objective row zr over columns 0..ncols-1, pivots on rows 0..nrows-1.
    // Returns why it stopped: 0 = the iteration limit, 1 = no entering column, 2 = no leaving row.
    auto simplex = [&](int zr, int ncols, int nrows, bool phase1) -> int {
        while (true) {
            if (n_piv >= P.max_iter) return 0;  // "iter > MaxIterations" before the column is chosen
            if (warp == 0) {
                const int e = warp_argmin_below(T + (size_t)zr * ld, ncols, -LPX_EPS);
                if (lane == 0) ctl[3] = e;
            }
            __syncthreads();
            const int e = ctl[3];
            if (e < 0) return 1;
            cta_stage_ratios<THREADS>(T, ld, m, e, rhs, prow);
            if (warp == 0) {
                const int lv = warp_margin_scan_staged(m, LPX_MARGIN_PRIMAL, prow);
                if (lane == 0) ctl[2] = lv;
            }
            __syncthreads();
            const int l = ctl[2];
            if (l < 0) return 2;
            pivot_on(l, e, nrows);
            if (phase1) p1++;
        }
    };

    int status;
    const int why1 = simplex(m + 1, W - 1, rows, true);  // Phase I: every column, artificials included
    __syncthreads();
    const double w = T[(size_t)(m + 1) * ld + rhs];
    const double tol = __dmul_rn(1e-9, __dadd_rn(1.0, dsh[0]));
    if (why1 == 0) {
        status = LPX_S_ITER_LIMIT;
    } else if (!(w >= -tol)) {
        status = LPX_INFEASIBLE;
    } else {
        // ---- drive-out: a basic artificial leaves for the lowest non-artificial column with |T[r][j]| > EPS -------
        for (int r = 0; r < m; r++) {
            if (sbasis[r] < ns) continue;
            if (warp == 0) {
                const double* Tr = T + (size_t)r * ld;
                int e = -1;
                for (int base = 0; base < ns && e < 0; base += 32) {
                    const int j = base + lane;
                    const unsigned h = __ballot_sync(0xffffffffu, j < ns && fabs(Tr[j]) > LPX_EPS);
                    if (h) e = base + __ffs(h) - 1;
                }
                if (lane == 0) ctl[2] = e;
            }
            __syncthreads();
            const int e = ctl[2];
            if (e >= 0) {  // else the row is redundant and its artificial stays basic
                pivot_on(r, e, rows);
                p1++;
            }
            __syncthreads();
        }
        const int why2 = simplex(m, ns, m + 1, false);  // Phase II: row m, the non-artificial columns
        status = why2 == 0 ? LPX_S_ITER_LIMIT : (why2 == 1 ? LPX_OPTIMAL : LPX_UNBOUNDED);
    }
    __syncthreads();

    // ---- outputs: the tableau where the solve stopped ---------------------------------------------------------------
    if (P.basis)
        for (int i = tid; i < m; i += THREADS) P.basis[(size_t)p * m + i] = sbasis[i];
    if (P.x) {
        double* xo = P.x + (size_t)p * n;
        for (int j = tid; j < n; j += THREADS) xo[j] = 0.0;
        __syncthreads();
        for (int i = tid; i < m; i += THREADS)  // distinct rows, distinct basic variables
            if (sbasis[i] < n) xo[sbasis[i]] = T[(size_t)i * ld + rhs];
    }
    if (P.z && tid == 0) P.z[p] = T[(size_t)m * ld + rhs];
    if (plog)
        for (int k = 2 * min(n_piv, P.pivots_cap) + tid; k < 2 * P.pivots_cap; k += THREADS) plog[k] = -1;
    if (P.tableau) {
        const int oc = ns + 1, total = (m + 1) * oc;
        double* To = P.tableau + (size_t)p * total;
        for (int k = tid; k < total; k += THREADS) {
            const int i = k / oc, j = k - i * oc;
            To[k] = T[(size_t)i * ld + (j < ns ? j : rhs)];
        }
    }
    if constexpr (REPORT) {
        double* rep = report + (size_t)p * (4 * (size_t)m + 3 * (size_t)n);
        if (status != LPX_OPTIMAL) {
            for (int e = tid; e < 4 * m + 3 * n; e += THREADS) rep[e] = sens_nan();
        } else {
            // prow (max_width + 2 doubles) is dead once the solve has stopped: rowof's W ints fit in it
            two_phase_report<THREADS>(T, ld, m, n, ns, W, P.sense, sbasis, flip, slk, art, reinterpret_cast<int*>(prow),
                                      bi, ci, rep);
        }
    }
    if (tid == 0) {
        P.status[p] = status;
        if (P.phase1) P.phase1[p] = p1;
        if (P.n_pivots) P.n_pivots[p] = n_piv;
        if (P.total_pivots && n_piv) atomicAdd(P.total_pivots, (unsigned long long)n_piv);
    }
}

template <int THREADS, bool SMEM_T>
__global__ void __launch_bounds__(THREADS, 1) two_phase_kernel(const TwoPhaseBatch P) {
    two_phase_body<THREADS, SMEM_T, false>(P, nullptr);
}

template <int THREADS, bool SMEM_T>
__global__ void __launch_bounds__(THREADS, 1) two_phase_sens_kernel(const TwoPhaseBatch P, double* report) {
    two_phase_body<THREADS, SMEM_T, true>(P, report);
}

static int slack_count(int m, const int* rel) {
    int s = 0;
    for (int i = 0; i < m; i++) s += (rel && rel[i] == 2) ? 0 : 1;
    return s;
}

static int check_args(int count, int m, int n, int sense, int pivots_cap, const int* host_rel, const lpx_options& o) {
    if (count < 0 || m < 1 || n < 1 || (sense != 0 && sense != 1) || pivots_cap < 0) {
        set_error("two-phase simplex: bad arguments: need count >= 0, m >= 1, n >= 1, sense in {0,1}, pivots_cap >= 0");
        return LPX_E_BAD_ARGS;
    }
    if (host_rel)
        for (int i = 0; i < m; i++)
            if (host_rel[i] < 0 || host_rel[i] > 2) {
                set_error("bad arguments: rel[i] must be 0 (LE), 1 (GE) or 2 (EQ)");
                return LPX_E_BAD_ARGS;
            }
    if (o.kernel != LPX_KERNEL_AUTO && o.kernel != LPX_KERNEL_CTA_SMEM && o.kernel != LPX_KERNEL_CTA_GLOBAL) {
        set_error("two-phase simplex runs on the per-CTA kernels: opt.kernel must be AUTO, CTA_SMEM or CTA_GLOBAL");
        return LPX_E_BAD_ARGS;
    }
    return LPX_OK;
}

template <int THREADS, bool SMEM_T>
static int launch_two_phase_variant(const TwoPhaseBatch& P, double* report, int count, size_t smem,
                                    cudaStream_t stream) {
    if (report) {
        auto kfn = two_phase_sens_kernel<THREADS, SMEM_T>;
        LPX_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kfn<<<count, THREADS, smem, stream>>>(P, report);
    } else {
        auto kfn = two_phase_kernel<THREADS, SMEM_T>;
        LPX_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kfn<<<count, THREADS, smem, stream>>>(P);
    }
    LPX_CUDA(cudaGetLastError());
    count_launch();
    return LPX_OK;
}

// Everything on the device already; s (slack columns) known on the host, arguments checked.  report (nullable): run the
// report builds, whose epilogue needs no shared memory beyond the solve's carve, so the fit decision is the same.
static int two_phase_launch(int count, int m, int n, int sense, int s, const double* A, const int* rel,
                            const double* b, const double* c, const lpx_options& o, int* status, int* phase1,
                            int* n_pivots, int* pivots, int pivots_cap, int* basis, double* x, double* z,
                            double* tableau, unsigned long long* total_pivots, double* report, cudaStream_t stream) {
    // the width takes a = m artificials: a depends on each LP's b, while rel is shared by the batch
    const int rows = m + 2, max_width = n + s + m + 1;
    const bool fits = cta_fits_smem(rows, max_width);
    if (o.kernel == LPX_KERNEL_CTA_SMEM && !fits) {
        set_error("two-phase simplex: the tableau does not fit in shared memory (LPX_KERNEL_CTA_SMEM forced)");
        return LPX_E_CAPACITY;
    }
    const bool smem_T = fits && o.kernel != LPX_KERNEL_CTA_GLOBAL;
    const size_t smem = cta_carve(rows, max_width, smem_T).total;
    if (smem > (size_t)max_smem_optin()) {
        set_error("two-phase simplex: problem too wide for the per-CTA kernels (work vectors exceed shared memory)");
        return LPX_E_CAPACITY;
    }
    if (count == 0) return LPX_OK;
    const size_t tsize = (size_t)rows * max_width;
    double* work = nullptr;
    if (!smem_T) {
        work = ws_dev_as<double>(WS_SCRATCH, (size_t)count * tsize);
        if (!work) return LPX_E_CUDA;
    }
    TwoPhaseBatch P;
    std::memset(&P, 0, sizeof P);
    P.A = A;
    P.b = b;
    P.c = c;
    P.rel = rel;
    P.m = m;
    P.n = n;
    P.sense = sense;
    P.s = s;
    P.max_width = max_width;
    P.max_iter = o.max_iterations;
    P.status = status;
    P.phase1 = phase1;
    P.n_pivots = n_pivots;
    P.pivots = pivots_cap > 0 ? pivots : nullptr;
    P.pivots_cap = pivots_cap;
    P.basis = basis;
    P.x = x;
    P.z = z;
    P.tableau = tableau;
    P.work = work;
    P.total_pivots = total_pivots;

    int threads = o.threads;
    if (threads != 128 && threads != 256 && threads != 512)  // as cta_launch chooses (lpx_cta.cu)
        threads = (!smem_T || tsize >= 8192) ? 512 : 256;
    if (smem_T) {
        if (threads == 128) return launch_two_phase_variant<128, true>(P, report, count, smem, stream);
        if (threads == 256) return launch_two_phase_variant<256, true>(P, report, count, smem, stream);
        return launch_two_phase_variant<512, true>(P, report, count, smem, stream);
    }
    if (threads == 128) return launch_two_phase_variant<128, false>(P, report, count, smem, stream);
    if (threads == 256) return launch_two_phase_variant<256, false>(P, report, count, smem, stream);
    return launch_two_phase_variant<512, false>(P, report, count, smem, stream);
}

}  // namespace lpx

using namespace lpx;

extern "C" {

int lpx_two_phase_dims(int m, int n, const int* rel, int* rows, int* cols) {
    lpx_options o;
    lpx_default_options(&o);
    int rc = check_args(0, m, n, 0, 0, rel, o);
    if (rc != LPX_OK) return rc;
    if (rows) *rows = m + 1;
    if (cols) *cols = n + slack_count(m, rel) + 1;
    return LPX_OK;
}

int lpx_two_phase_solve_batched_dev(int count, int m, int n, int sense, const double* A, const int* rel,
                                    const double* b, const double* c, const lpx_options* opt, int* status,
                                    int* phase1_pivots, int* n_pivots, int* pivots, int pivots_cap, int* basis,
                                    double* x, double* z, double* tableau, unsigned long long* total_pivots,
                                    void* stream) {
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    int rc = check_args(count, m, n, sense, pivots_cap, nullptr, o);
    if (rc != LPX_OK) return rc;
    if (!A || !b || !c || !status) {
        set_error("lpx_two_phase_solve_batched_dev: A, b, c and status must not be NULL");
        return LPX_E_BAD_ARGS;
    }
    if ((rc = ensure_device()) != LPX_OK) return rc;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    cudaStream_t s = (cudaStream_t)stream;
    // rel is a device pointer; the tableau shape needs it on the host
    int ns = m;
    if (rel) {
        std::vector<int> hrel(m);
        LPX_CUDA(cudaMemcpyAsync(hrel.data(), rel, (size_t)m * 4, cudaMemcpyDeviceToHost, s));
        LPX_CUDA(cudaStreamSynchronize(s));
        if ((rc = check_args(count, m, n, sense, pivots_cap, hrel.data(), o)) != LPX_OK) return rc;
        ns = slack_count(m, hrel.data());
    }
    return two_phase_launch(count, m, n, sense, ns, A, rel, b, c, o, status, phase1_pivots, n_pivots, pivots,
                            pivots_cap, basis, x, z, tableau, total_pivots, nullptr, s);
}

int lpx_two_phase_solve_batched(int count, int m, int n, int sense, const double* A, const int* rel, const double* b,
                                const double* c, const lpx_options* opt, int* status, int* phase1_pivots,
                                int* n_pivots, int* pivots, int pivots_cap, int* basis, double* x, double* z,
                                double* tableau, long long* total_pivots) {
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    int rc = check_args(count, m, n, sense, pivots_cap, rel, o);
    if (rc != LPX_OK) return rc;
    if (!A || !b || !c || !status) {
        set_error("lpx_two_phase_solve_batched: A, b, c and status must not be NULL");
        return LPX_E_BAD_ARGS;
    }
    if ((rc = ensure_device()) != LPX_OK) return rc;
    Runtime& r = rt();
    std::lock_guard<std::recursive_mutex> lk(r.mu);
    cudaStream_t s = r.stream;
    if (total_pivots) *total_pivots = 0;
    if (count == 0) return LPX_OK;
    const int ns = slack_count(m, rel);
    const size_t cnt = (size_t)count, cap = pivots ? (size_t)pivots_cap : 0, tsize = (size_t)(m + 1) * (n + ns + 1);

    double* dA = ws_dev_as<double>(WS_A, cnt * m * n);
    double* db = ws_dev_as<double>(WS_B, cnt * m);
    double* dc = ws_dev_as<double>(WS_C, cnt * n);
    int* drel = ws_dev_as<int>(WS_REL, m);
    // ints: status, phase1, n_pivots | pivots | basis;  doubles: x | z | tableau
    int* di = ws_dev_as<int>(WS_TP_INT, 3 * cnt + cnt * cap * 2 + cnt * m);
    double* dd = ws_dev_as<double>(WS_TP_DBL, cnt * n + cnt + (tableau ? cnt * tsize : 0));
    unsigned long long* dtot = ws_dev_as<unsigned long long>(WS_TOTAL, 1);
    if (!dA || !db || !dc || !drel || !di || !dd || !dtot) return LPX_E_CUDA;
    int *dst = di, *dp1 = di + cnt, *dnp = di + 2 * cnt, *dpiv = di + 3 * cnt, *dbasis = dpiv + cnt * cap * 2;
    double *dx = dd, *dz = dd + cnt * n, *dT = tableau ? dz + cnt : nullptr;

    LPX_CUDA(cudaMemcpyAsync(dA, A, cnt * m * n * 8, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemcpyAsync(db, b, cnt * m * 8, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemcpyAsync(dc, c, cnt * n * 8, cudaMemcpyHostToDevice, s));
    if (rel) LPX_CUDA(cudaMemcpyAsync(drel, rel, (size_t)m * 4, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemsetAsync(dtot, 0, 8, s));
    rc = two_phase_launch(count, m, n, sense, ns, dA, rel ? drel : nullptr, db, dc, o, dst, phase1_pivots ? dp1 : nullptr,
                          n_pivots ? dnp : nullptr, cap ? dpiv : nullptr, (int)cap, basis ? dbasis : nullptr,
                          x ? dx : nullptr, z ? dz : nullptr, dT, dtot, nullptr, s);
    if (rc != LPX_OK) return rc;
    auto down = [&](void* dst_h, const void* src, size_t bytes) {
        return dst_h ? cudaMemcpyAsync(dst_h, src, bytes, cudaMemcpyDeviceToHost, s) : cudaSuccess;
    };
    unsigned long long htot = 0;
    LPX_CUDA(down(status, dst, cnt * 4));
    LPX_CUDA(down(phase1_pivots, dp1, cnt * 4));
    LPX_CUDA(down(n_pivots, dnp, cnt * 4));
    if (cap) LPX_CUDA(down(pivots, dpiv, cnt * cap * 2 * 4));
    LPX_CUDA(down(basis, dbasis, cnt * m * 4));
    LPX_CUDA(down(x, dx, cnt * n * 8));
    LPX_CUDA(down(z, dz, cnt * 8));
    LPX_CUDA(down(tableau, dT, cnt * tsize * 8));
    LPX_CUDA(down(&htot, dtot, 8));
    LPX_CUDA(cudaStreamSynchronize(s));
    if (total_pivots) *total_pivots = (long long)htot;
    return LPX_OK;
}

int lpx_two_phase_solve_sensitivity_batched_dev(int count, int m, int n, int sense, const double* A, const int* rel,
                                                const double* b, const double* c, const lpx_options* opt, int* status,
                                                int* phase1_pivots, int* n_pivots, int* basis, double* x, double* z,
                                                double* report, unsigned long long* total_pivots, void* stream) {
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    int rc = check_args(count, m, n, sense, 0, nullptr, o);
    if (rc != LPX_OK) return rc;
    if (!A || !b || !c || !status || !report) {
        set_error("lpx_two_phase_solve_sensitivity_batched_dev: A, b, c, status and report must not be NULL");
        return LPX_E_BAD_ARGS;
    }
    if ((rc = ensure_device()) != LPX_OK) return rc;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    cudaStream_t s = (cudaStream_t)stream;
    int ns = m;
    if (rel) {
        std::vector<int> hrel(m);
        LPX_CUDA(cudaMemcpyAsync(hrel.data(), rel, (size_t)m * 4, cudaMemcpyDeviceToHost, s));
        LPX_CUDA(cudaStreamSynchronize(s));
        if ((rc = check_args(count, m, n, sense, 0, hrel.data(), o)) != LPX_OK) return rc;
        ns = slack_count(m, hrel.data());
    }
    return two_phase_launch(count, m, n, sense, ns, A, rel, b, c, o, status, phase1_pivots, n_pivots, nullptr, 0, basis,
                            x, z, nullptr, total_pivots, report, s);
}

int lpx_two_phase_solve_sensitivity_batched(int count, int m, int n, int sense, const double* A, const int* rel,
                                            const double* b, const double* c, const lpx_options* opt, int* status,
                                            int* phase1_pivots, int* n_pivots, int* basis, double* x, double* z,
                                            double* report, long long* total_pivots) {
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    int rc = check_args(count, m, n, sense, 0, rel, o);
    if (rc != LPX_OK) return rc;
    if (!A || !b || !c || !status || !report) {
        set_error("lpx_two_phase_solve_sensitivity_batched: A, b, c, status and report must not be NULL");
        return LPX_E_BAD_ARGS;
    }
    if ((rc = ensure_device()) != LPX_OK) return rc;
    Runtime& r = rt();
    std::lock_guard<std::recursive_mutex> lk(r.mu);
    cudaStream_t s = r.stream;
    if (total_pivots) *total_pivots = 0;
    if (count == 0) return LPX_OK;
    const int ns = slack_count(m, rel);
    const size_t cnt = (size_t)count, stride = 4 * (size_t)m + 3 * (size_t)n;

    double* dA = ws_dev_as<double>(WS_A, cnt * m * n);
    double* db = ws_dev_as<double>(WS_B, cnt * m);
    double* dc = ws_dev_as<double>(WS_C, cnt * n);
    int* drel = ws_dev_as<int>(WS_REL, m);
    // ints: status, phase1, n_pivots | basis;  doubles: x | z | report
    int* di = ws_dev_as<int>(WS_TP_INT, 3 * cnt + cnt * m);
    double* dd = ws_dev_as<double>(WS_TP_DBL, cnt * n + cnt + cnt * stride);
    unsigned long long* dtot = ws_dev_as<unsigned long long>(WS_TOTAL, 1);
    if (!dA || !db || !dc || !drel || !di || !dd || !dtot) return LPX_E_CUDA;
    int *dst = di, *dp1 = di + cnt, *dnp = di + 2 * cnt, *dbasis = di + 3 * cnt;
    double *dx = dd, *dz = dd + cnt * n, *drep = dz + cnt;

    LPX_CUDA(cudaMemcpyAsync(dA, A, cnt * m * n * 8, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemcpyAsync(db, b, cnt * m * 8, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemcpyAsync(dc, c, cnt * n * 8, cudaMemcpyHostToDevice, s));
    if (rel) LPX_CUDA(cudaMemcpyAsync(drel, rel, (size_t)m * 4, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemsetAsync(dtot, 0, 8, s));
    rc = two_phase_launch(count, m, n, sense, ns, dA, rel ? drel : nullptr, db, dc, o, dst, phase1_pivots ? dp1 : nullptr,
                          n_pivots ? dnp : nullptr, nullptr, 0, basis ? dbasis : nullptr, x ? dx : nullptr,
                          z ? dz : nullptr, nullptr, dtot, drep, s);
    if (rc != LPX_OK) return rc;
    auto down = [&](void* dst_h, const void* src, size_t bytes) {
        return dst_h ? cudaMemcpyAsync(dst_h, src, bytes, cudaMemcpyDeviceToHost, s) : cudaSuccess;
    };
    unsigned long long htot = 0;
    LPX_CUDA(down(status, dst, cnt * 4));
    LPX_CUDA(down(phase1_pivots, dp1, cnt * 4));
    LPX_CUDA(down(n_pivots, dnp, cnt * 4));
    LPX_CUDA(down(basis, dbasis, cnt * m * 4));
    LPX_CUDA(down(x, dx, cnt * n * 8));
    LPX_CUDA(down(z, dz, cnt * 8));
    LPX_CUDA(down(report, drep, cnt * stride * 8));
    LPX_CUDA(down(&htot, dtot, 8));
    LPX_CUDA(cudaStreamSynchronize(s));
    if (total_pivots) *total_pivots = (long long)htot;
    return LPX_OK;
}

}  // extern "C"
