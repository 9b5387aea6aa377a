// lpx_stream.cu — ONE large dense tableau spread over the whole GPU (BASELINE config 3:
// 4096 x 8192 -> 4097 x 12289 doubles = 403 MB, far beyond L2).  Each pivot is
//
//   select  (1 CTA)   exact ChooseLeaving on two compact 4097-vectors, normalise the pivot row,
//                     update the z-row in registers and pick the NEXT entering column
//   update  (grid)    one HBM pass: T[i,j] -= f[i] * p[j], 128-bit loads/stores, the pivot row
//                     held in registers per column strip; the pass also captures the next
//                     entering column and the RHS into compact vectors for the next select
//
// so the tableau is read and written exactly once per pivot: 2 * 8 * rows * cols algorithmic
// bytes (SURVEY.md §8d).  Replaces R/Models/PrimalSimplex.cs:92-124 (loop), :205-257 (rules).
//
// HBM layout: row-major, leading dimension padded to a multiple of 16 doubles (128 B) so every
// row starts on a 128-byte line and double2 accesses are aligned; pad columns hold zeros.
#include <algorithm>
#include <cstring>
#include <limits>
#include <vector>

#include "lpx_common.cuh"
#include "lpx_runtime.hpp"
#include "lpx_stream.hpp"

namespace lpx {

struct StreamCtl {
    int status;   // LPX_RUNNING until decided
    int pivots;   // pivots performed
    int enter;    // entering column of the next pivot (-1: optimal)
    int leave;    // leaving row of the pivot being applied
    int active;   // 1: the update kernel has a pivot to apply
    int capture;  // entering column of the pivot after this one (-1: none)
    int k;        // index of the pivot being applied
    int block_cnt;  // blocked protocol: pivots decided by the last look-ahead, applied by the next pass
    int blk_in[2];   // pipelined protocol, per block parity: tableau buffer the block's pass reads
    int blk_cnt[2];  // pipelined protocol, per block parity: pivots decided for the block
};

struct StreamParams {
    double* T;
    int ld, rows, width, m, n;
    double* colbuf;  // 2 x colstride: entering column of pivot k lives in buffer k & 1
    int colstride;
    double* rhsbuf;  // rows
    double* prow;    // ld
    double* ratio;   // m
    int* basis;
    int* pivlog;
    int pivlog_cap;
    StreamCtl* ctl;
    int max_iter;
    ArgMin* partial;  // per prep-CTA argmin of the look-ahead z-row (multi-CTA protocol)
    int npartial;     // 0: single-CTA select protocol (very tall tableaux)
    // blocked look-ahead protocol (lpx_stream_block.cuh)
    double* Fbuf;  // kblock x colstride factor columns
    double* Pbuf;  // kblock x ld normalised pivot rows
    int* Lbuf;     // kblock leaving rows
    int kblock;    // 0: per-pivot protocol
    unsigned long long* dbg;  // optional phase timestamps (development aid)
    double* T1;    // second tableau buffer (pipelined protocol: passes are out of place)
    double* zbuf;  // ld: z-row after every decided pivot, handed from look-ahead to look-ahead
};

#define LPX_PREP_THREADS 1024

__device__ __forceinline__ double dneg_s(double v) {
    return __longlong_as_double(__double_as_longlong(v) ^ (long long)0x8000000000000000ULL);
}

template <int THREADS>
__device__ __forceinline__ int block_min_int(int v, int* sred) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = __reduce_min_sync(0xffffffffu, v);
    if (lane == 0) sred[warp] = v;
    __syncthreads();
    if (warp == 0) {
        int w = lane < THREADS / 32 ? sred[lane] : INT_MAX;
        w = __reduce_min_sync(0xffffffffu, w);
        if (lane == 0) sred[32] = w;
    }
    __syncthreads();
    const int r = sred[32];
    __syncthreads();
    return r;
}

// ---- setup kernels --------------------------------------------------------------------------

// First offending constraint in the reference's order (PrimalSimplex.cs:66-77).
__global__ void __launch_bounds__(1024) stream_validate_kernel(StreamCtl* ctl, const double* b, int m_in,
                                                               int first_ge) {
    __shared__ int sred[34];
    int cand = INT_MAX;
    for (int r = threadIdx.x; r < m_in; r += 1024)
        if (b[r] < -1e-9) {
            cand = r;
            break;
        }
    cand = block_min_int<1024>(cand, sred);
    if (threadIdx.x == 0) {
        int st = LPX_RUNNING;
        if (first_ge != INT_MAX || cand != INT_MAX) st = (first_ge <= cand) ? LPX_S_GE_ROW : LPX_S_NEG_RHS;
        ctl->status = st;
        ctl->pivots = 0;
        ctl->enter = -1;
        ctl->leave = -1;
        ctl->active = 0;
        ctl->capture = -1;
        ctl->k = 0;
        ctl->block_cnt = 0;
        ctl->blk_in[0] = ctl->blk_in[1] = 0;
        ctl->blk_cnt[0] = ctl->blk_cnt[1] = 0;
    }
}

// BuildTableau (PrimalSimplex.cs:179-203) with the EQ expansion folded in through a row map.
__global__ void __launch_bounds__(256) stream_build_kernel(StreamParams P, const double* A, const double* b,
                                                           const double* c, const int* rsrc, const int* rsgn,
                                                           int sense) {
    const int n = P.n, m = P.m, rhs = P.width - 1;
    for (int i = blockIdx.x; i < P.rows; i += gridDim.x) {
        double* Ti = P.T + (size_t)i * P.ld;
        if (i < m) {
            const int src = rsrc[i];
            const bool flip = rsgn[i] != 0;
            const double* Ar = A + (size_t)src * n;
            for (int j = threadIdx.x; j < P.ld; j += 256) {
                double v = 0.0;
                if (j < n) v = neg_if(Ar[j], flip);
                else if (j == rhs) v = neg_if(b[src], flip);
                else if (j == n + i) v = 1.0;
                Ti[j] = v;
            }
            if (threadIdx.x == 0) P.basis[i] = n + i;
        } else {
            for (int j = threadIdx.x; j < P.ld; j += 256) {
                double v = 0.0;
                if (j < n) {
                    double cj = c[j];
                    if (sense == 1) cj = dneg_s(cj);
                    v = dneg_s(cj);
                }
                Ti[j] = v;
            }
        }
    }
}

// ChooseEntering on the initial z-row.
__global__ void __launch_bounds__(1024) stream_first_kernel(StreamParams P) {
    __shared__ ArgMin red[34];
    if (P.ctl->status != LPX_RUNNING) return;
    const int e = block_argmin_below<1024>(P.T + (size_t)P.m * P.ld, P.width - 1, -LPX_EPS, red);
    if (threadIdx.x == 0) P.ctl->enter = e;
}

// Compact copies of the entering column and of the RHS (only needed before the first pivot; from
// then on the update pass captures them on the fly).
__global__ void __launch_bounds__(256) stream_gather_kernel(StreamParams P) {
    if (P.ctl->status != LPX_RUNNING) return;
    const int e = P.ctl->enter;
    if (P.zbuf)
        for (int j = blockIdx.x * 256 + threadIdx.x; j < P.ld; j += gridDim.x * 256)
            P.zbuf[j] = P.T[(size_t)P.m * P.ld + j];
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= P.rows) return;
    const double* Ti = P.T + (size_t)i * P.ld;
    if (e >= 0) P.colbuf[i] = Ti[e];
    P.rhsbuf[i] = Ti[P.width - 1];
}

// ---- per-pivot kernels ------------------------------------------------------------------------

// FORCE: the ratio margin of DualSimplex.ForceDualFeasibility (1e-12) instead of PrimalSimplex's (1e-9), for the silent
// Primal Simplex pivots that open a Dual Simplex session (session_dual_silent_phase).
template <bool FORCE>
__global__ void __launch_bounds__(1024) stream_select_kernel(StreamParams P, int probe_only) {
    constexpr double margin = FORCE ? LPX_MARGIN_DUAL : LPX_MARGIN_PRIMAL;
    __shared__ ArgMin red[34];
    __shared__ int ired[34];
    StreamCtl* ctl = P.ctl;
    const int tid = threadIdx.x;
    if (tid == 0) ctl->active = 0;
    if (ctl->status != LPX_RUNNING) return;
    const int k = ctl->pivots;
    if (k >= P.max_iter) {  // "if (iter > MaxIterations) throw" comes before the optimality test
        if (tid == 0) ctl->status = LPX_S_ITER_LIMIT;
        return;
    }
    const int e = ctl->enter;
    if (e < 0) {
        if (tid == 0) ctl->status = LPX_OPTIMAL;
        return;
    }
    const int m = P.m;
    const double* col = P.colbuf + (size_t)(k & 1) * P.colstride;

    // ChooseLeaving.  Ratios first (NaN marks "not eligible": NaN < x is false) ...
    for (int i = tid; i < m; i += 1024) {
        const double a = col[i];
        double r = __longlong_as_double(0x7ff8000000000000LL);
        if (a > LPX_EPS) r = ddiv_by_pos(P.rhsbuf[i], a);
        P.ratio[i] = r;
    }
    __syncthreads();
    // ... then the reference's sequential rule "take i if ratio < best - margin", reproduced exactly:
    // repeatedly find the FIRST row after the last accepted one that beats the running best.
    // The number of rounds is the number of accepted updates (about ln m on random data).
    const int R = (m + 1023) / 1024;
    const int lo = tid * R, hi = min(m, lo + R);
    double best = __longlong_as_double(0x7ff0000000000000LL);
    int row = -1, start = 0;
    while (true) {
        const double thr = __dsub_rn(best, margin);
        int cand = INT_MAX;
        for (int i = max(lo, start); i < hi; i++)
            if (P.ratio[i] < thr) {
                cand = i;
                break;
            }
        cand = block_min_int<1024>(cand, ired);
        if (cand == INT_MAX) break;
        best = P.ratio[cand];
        row = cand;
        start = cand + 1;
    }
    if (row < 0) {
        if (tid == 0) ctl->status = LPX_UNBOUNDED;
        return;
    }
    if (probe_only) return;

    // Normalise the pivot row (true division), write it back, and on the way compute the updated
    // z-row entries z_j - f_z * p_j to choose the NEXT entering column (ChooseEntering).
    const int l = row;
    const double piv = col[l], fz = col[m];
    double* Tl = P.T + (size_t)l * P.ld;
    const double* Tz = P.T + (size_t)m * P.ld;
    ArgMin a;
    a.v = -LPX_EPS;
    a.i = INT_MAX;
    const int ncand = P.width - 1;
    for (int j = tid; j < P.ld; j += 1024) {
        const double pj = ddiv_by_pos(Tl[j], piv);
        P.prow[j] = pj;
        Tl[j] = pj;
        if (j < ncand) {
            const double zn = __dsub_rn(Tz[j], __dmul_rn(fz, pj));
            if (zn < a.v) {
                a.v = zn;
                a.i = j;
            }
        }
    }
    a = warp_argmin(a);
    const int lane = tid & 31, warp = tid >> 5;
    if (lane == 0) red[warp] = a;
    __syncthreads();
    if (warp == 0) {
        ArgMin b2 = red[lane];
        b2 = warp_argmin(b2);
        if (lane == 0) {
            const int en = b2.i == INT_MAX ? -1 : b2.i;
            double* out = P.colbuf + (size_t)((k + 1) & 1) * P.colstride;
            if (en >= 0) out[l] = P.prow[en];
            P.rhsbuf[l] = P.prow[P.width - 1];
            P.basis[l] = e;
            if (k < P.pivlog_cap) {
                P.pivlog[2 * k] = e;
                P.pivlog[2 * k + 1] = l;
            }
            ctl->leave = l;
            ctl->capture = en;
            ctl->k = k;
            ctl->pivots = k + 1;
            ctl->enter = en;
            ctl->active = 1;
        }
    }
}

// Multi-CTA replacement of stream_select_kernel (the single CTA took ~30 us per pivot, 18 % of the
// step).  grid = one thread per tableau column.  EVERY CTA repeats the exact ratio test on the two
// compact vectors (64 KB from L2, ratios parked in shared memory, rows interleaved over the
// threads so the scan is bank-conflict free), then normalises its own 256 columns of the pivot
// row and reduces its slice of the look-ahead z-row to one (value, column) pair.  The update
// kernel combines the pairs.  Field ownership keeps the CTAs race-free: prep CTAs only READ
// status/pivots/enter; CTA 0 writes leave/k/active (and a terminal status, which makes every
// other CTA return as well); pivots/enter are advanced by the update kernel.
__global__ void __launch_bounds__(LPX_PREP_THREADS) stream_prep_kernel(StreamParams P, int probe_only) {
    extern __shared__ double s_ratio[];
    __shared__ ArgMin red[34];
    __shared__ int ired[34];
    constexpr int TH = LPX_PREP_THREADS;
    StreamCtl* ctl = P.ctl;
    const int tid = threadIdx.x;
    const bool lead = blockIdx.x == 0 && tid == 0;
    const int status = ctl->status;
    const int k = ctl->pivots;
    const int e = ctl->enter;
    if (lead) ctl->active = 0;
    if (status != LPX_RUNNING) return;
    if (k >= P.max_iter) {
        if (lead) ctl->status = LPX_S_ITER_LIMIT;
        return;
    }
    if (e < 0) {
        if (lead) ctl->status = LPX_OPTIMAL;
        return;
    }
    const int m = P.m;
    const double* col = P.colbuf + (size_t)(k & 1) * P.colstride;
    // all loads of a batch are issued before the first division: dependent global loads in a
    // loop (load a, branch, load rhs, divide) cost ~1.4k cycles per row and made this phase 10 us
    for (int base = 0; base < m; base += 4 * TH) {
        double a[4], bb[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int i = base + u * TH + tid;
            a[u] = i < m ? col[i] : 0.0;
            bb[u] = i < m ? P.rhsbuf[i] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int i = base + u * TH + tid;
            double r = __longlong_as_double(0x7ff8000000000000LL);  // NaN: never eligible
            if (a[u] > LPX_EPS) r = ddiv_by_pos(bb[u], a[u]);
            if (i < m) s_ratio[i] = r;
        }
    }
    __syncthreads();
    double best = __longlong_as_double(0x7ff0000000000000LL);
    int row = -1, start = 0;
    while (true) {
        const double thr = __dsub_rn(best, LPX_MARGIN_PRIMAL);
        int cand = INT_MAX;
        // this thread's rows are tid, tid+TH, ...: its first hit at or after `start`
        int i = tid;
        if (start > tid) i = tid + ((start - tid + TH - 1) / TH) * TH;
        for (; i < m; i += TH)
            if (s_ratio[i] < thr) {
                cand = i;
                break;
            }
        cand = block_min_int<TH>(cand, ired);
        if (cand == INT_MAX) break;
        best = s_ratio[cand];
        row = cand;
        start = cand + 1;
    }
    if (row < 0) {
        if (lead) ctl->status = LPX_UNBOUNDED;
        return;
    }
    if (probe_only) return;

    const int l = row;
    const double piv = col[l], fz = col[m];
    const int j = blockIdx.x * TH + tid;
    ArgMin a;
    a.v = -LPX_EPS;
    a.i = INT_MAX;
    if (j < P.ld) {
        double* Tl = P.T + (size_t)l * P.ld;
        const double pj = ddiv_by_pos(Tl[j], piv);
        if (j < P.width - 1) {
            const double zn = __dsub_rn(P.T[(size_t)m * P.ld + j], __dmul_rn(fz, pj));
            if (zn < a.v) {
                a.v = zn;
                a.i = j;
            }
        }
        P.prow[j] = pj;
        Tl[j] = pj;
    }
    a = warp_argmin(a);
    const int lane = tid & 31, warp = tid >> 5;
    if (lane == 0) red[warp] = a;
    __syncthreads();
    if (warp == 0) {
        ArgMin b2;
        b2.v = -LPX_EPS;
        b2.i = INT_MAX;
        if (lane < TH / 32) b2 = red[lane];
        b2 = warp_argmin(b2);
        if (lane == 0) P.partial[blockIdx.x] = b2;
    }
    if (lead) {
        P.basis[l] = e;
        if (k < P.pivlog_cap) {
            P.pivlog[2 * k] = e;
            P.pivlog[2 * k + 1] = l;
        }
        ctl->leave = l;
        ctl->k = k;
        ctl->active = 1;
    }
}

// The HBM pass.  grid = (column strips of 512, row chunks); each thread owns two adjacent
// columns for its CTA's rows, so p[j] stays in registers and f[i] is a broadcast load.
// The sweep direction alternates with the pivot parity: the rows written last by pivot k are
// read first by pivot k+1, while they are still in the 126 MB L2.
template <int UNROLL>
__global__ void __launch_bounds__(256, 4) stream_update_kernel(StreamParams P) {
    StreamCtl* ctl = P.ctl;
    if (ctl->active == 0) return;
    const int l = ctl->leave, k = ctl->k;
    int cap;
    if (P.npartial > 0) {
        // combine the prep CTAs' look-ahead argmins: the next entering column (ChooseEntering)
        __shared__ int s_cap;
        if (threadIdx.x < 32) {
            ArgMin a;
            a.v = -LPX_EPS;
            a.i = INT_MAX;
            for (int i = threadIdx.x; i < P.npartial; i += 32) a = argmin_pick(a, P.partial[i]);
            a = warp_argmin(a);
            if (threadIdx.x == 0) s_cap = a.i == INT_MAX ? -1 : a.i;
        }
        __syncthreads();
        cap = s_cap;
        if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) {
            // pivot-row entries of the two captured vectors, then advance the pivot counter
            double* outl = P.colbuf + (size_t)((k + 1) & 1) * P.colstride;
            if (cap >= 0) outl[l] = P.prow[cap];
            P.rhsbuf[l] = P.prow[P.width - 1];
            ctl->capture = cap;
            ctl->enter = cap;
            ctl->pivots = k + 1;
        }
    } else {
        cap = ctl->capture;
    }
    const int j0 = (blockIdx.x * 256 + threadIdx.x) * 2;
    if (j0 >= P.ld) return;
    const double* __restrict__ f = P.colbuf + (size_t)(k & 1) * P.colstride;
    double* __restrict__ out = P.colbuf + (size_t)((k + 1) & 1) * P.colstride;
    const int rpc = (P.rows + gridDim.y - 1) / gridDim.y;
    const int r0 = blockIdx.y * rpc;
    const int r1 = min(P.rows, r0 + rpc);
    const int cnt = r1 - r0;
    if (cnt <= 0) return;
    const double2 p = *reinterpret_cast<const double2*>(P.prow + j0);
    const int rhs = P.width - 1;
    const int cx = (cap == j0) ? 0 : ((cap == j0 + 1) ? 1 : -1);
    const int rx = (rhs == j0) ? 0 : ((rhs == j0 + 1) ? 1 : -1);
    const bool rev = (k & 1) != 0;
    double* __restrict__ Tc = P.T + j0;
    const size_t ld = (size_t)P.ld;

    for (int q = 0; q < cnt; q += UNROLL) {
        double2 t[UNROLL];
        double fi[UNROLL];
        int ri[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; u++) {
            const int qq = q + u;
            ri[u] = qq < cnt ? (rev ? r1 - 1 - qq : r0 + qq) : -1;
            if (ri[u] >= 0) {
                t[u] = *reinterpret_cast<const double2*>(Tc + (size_t)ri[u] * ld);
                fi[u] = f[ri[u]];
            }
        }
#pragma unroll
        for (int u = 0; u < UNROLL; u++) {
            if (ri[u] >= 0 && ri[u] != l) {
                double2 v;
                v.x = __dsub_rn(t[u].x, __dmul_rn(fi[u], p.x));
                v.y = __dsub_rn(t[u].y, __dmul_rn(fi[u], p.y));
                *reinterpret_cast<double2*>(Tc + (size_t)ri[u] * ld) = v;
                if (cx >= 0) out[ri[u]] = cx == 0 ? v.x : v.y;
                if (rx >= 0) P.rhsbuf[ri[u]] = rx == 0 ? v.x : v.y;
            }
        }
    }
}

}  // namespace lpx

#include "lpx_stream_block.cuh"
#include "lpx_stream_pipe.cuh"
#include "lpx_stream_reopt.cuh"
#include "lpx_stream_dual.cuh"
#include "lpx_stream_param.cuh"
#include "lpx_stream_twophase.cuh"


// ---- session object -----------------------------------------------------------------------------

using namespace lpx;

struct lpx_session {
    StreamParams P{};
    int m_in = 0, n = 0, sense = 0;
    lpx_options opt{};
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    void* buffers[32] = {};
    int nbuf = 0;
    // sensitivity report: copies of b and c, the constraint -> slack row map, and (on first use) the work buffers
    double* sens_b = nullptr;
    double* sens_c = nullptr;
    int* sens_rmap = nullptr;
    std::vector<int> rmap;  // host copy of sens_rmap: constraint i -> expanded row i1 (EQ: -i1 - 1)
    bool sens_ok = true;    // false for ROW / COL re-optimization queries and their descendants
    bool dual = false;      // Dual Simplex rules (RHS / ROW re-optimization queries, Dual Simplex sessions)
    bool dual_model = false;  // opened by lpx_dual_session_open(_dev): DualSimplex.Solve on the model
    int silent = 0;           // ForceDualFeasibility pivots performed inside lpx_dual_session_open
    int* sens_rowof = nullptr;
    void* sens_partial = nullptr;
    double* sens_report = nullptr;
    dim3 grid_update;
    dim3 grid_block;
    bool la_cluster = false;  // look-ahead on a thread-block cluster (else one CTA)
    int rpc_block = 0;        // rows per CTA of the blocked pass
    // pipelined protocol: look-ahead of block B+1 overlaps the pass of block B
    bool pipe = false;
    cudaStream_t streamL = nullptr;
    cudaEvent_t evL[2] = {nullptr, nullptr}, evP[2] = {nullptr, nullptr}, evStart = nullptr;
    long long blocks = 0;  // blocks launched so far (parity selects the buffer halves)
    dim3 grid_pipe;
    int rpc_pipe = 0;
    int device = 0;
    // two-phase session (lpx_two_phase_session_open): its look-ahead and the compact output width n + s
    bool two_phase = false;
    TwoPhaseLa tla{};
    size_t tla_smem = 0;
    int tp_ns = 0;
    int* tp_info = nullptr;  // device flip | slk | art (m ints each): lpx_session_two_phase_sensitivity reads them
};

namespace lpx {

static void* sess_alloc(lpx_session* s, size_t bytes) {
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes ? bytes : 16);
    if (e != cudaSuccess) {
        cuda_fail(e, "cudaMalloc(session)", __FILE__, __LINE__);
        return nullptr;
    }
    s->buffers[s->nbuf++] = p;
    return p;
}

static void sess_free(lpx_session* s) {
    if (!s) return;
    if (s->stream) cudaStreamSynchronize(s->stream);
    for (int i = 0; i < s->nbuf; i++) cudaFree(s->buffers[i]);
    if (s->streamL) {
        cudaStreamSynchronize(s->streamL);
        cudaStreamDestroy(s->streamL);
    }
    for (int k = 0; k < 2; k++) {
        if (s->evL[k]) cudaEventDestroy(s->evL[k]);
        if (s->evP[k]) cudaEventDestroy(s->evP[k]);
    }
    if (s->evStart) cudaEventDestroy(s->evStart);
    if (s->own_stream && s->stream) cudaStreamDestroy(s->stream);
    delete s;
}

static void launch_select(lpx_session* s, int probe_only) {
    if (s->dual)
        stream_dual_select_kernel<<<1, 1024, 0, s->stream>>>(s->P, probe_only);
    else if (s->P.npartial > 0)
        stream_prep_kernel<<<s->P.npartial, LPX_PREP_THREADS, (size_t)s->P.m * 8, s->stream>>>(s->P, probe_only);
    else
        stream_select_kernel<false><<<1, 1024, 0, s->stream>>>(s->P, probe_only);
}

static int launch_pair(lpx_session* s, int probe_only) {
    launch_select(s, probe_only);
    count_launch();
    if (!probe_only) {
        stream_update_kernel<4><<<s->grid_update, 256, 0, s->stream>>>(s->P);
        count_launch();
    }
    LPX_CUDA(cudaGetLastError());
    return LPX_OK;
}

static size_t lookahead_smem(const StreamParams& P) { return ((size_t)P.ld + 3 * (size_t)P.colstride) * 8; }

// One block of the look-ahead protocol: decide up to `budget` pivots, then one HBM pass.
static size_t lookahead_cluster_smem(const StreamParams& P) {
    const size_t cw = ((((size_t)P.ld + LPX_LA_CLUSTER - 1) / LPX_LA_CLUSTER) + 1) & ~(size_t)1;
    const size_t q = ((size_t)P.m + LPX_LA_THREADS - 1) / LPX_LA_THREADS;
    return (cw + 2 * (size_t)P.colstride + q * LPX_LA_THREADS) * 8;
}

static void launch_lookahead(lpx_session* s, int budget) {
    if (s->two_phase)
        stream_two_phase_lookahead_kernel<<<1, 1024, s->tla_smem, s->stream>>>(s->P, s->tla, budget);
    else if (s->dual)
        stream_dual_lookahead_kernel<<<1, 1024, dual_lookahead_smem(s->P), s->stream>>>(s->P, budget);
    else if (s->la_cluster)
        stream_lookahead_cluster_kernel<<<LPX_LA_CLUSTER, LPX_LA_THREADS, lookahead_cluster_smem(s->P), s->stream>>>(
            s->P, budget);
    else
        stream_lookahead_kernel<<<1, 1024, lookahead_smem(s->P), s->stream>>>(s->P, budget);
}

// pass variants: LDG/STG kernels <KMAX, doubles per thread, rows in flight> or the TMA-staged kernel
typedef void (*BlockPassFn)(StreamParams, int);
// the TMA-staged kernel is the default (measured 143 us vs 182 us per 8-pivot pass at 4097 x 12289)
static bool block_pass_is_tma(int variant) { return variant == 3 || variant == 0; }
static BlockPassFn block_pass_fn(int variant, int kblock) {
    // variant: 0 auto; 1: two doubles/thread; 2: one; 3: TMA-staged
    if (block_pass_is_tma(variant))
        return kblock <= 8 ? stream_update_block_tma_kernel<8> : stream_update_block_tma_kernel<16>;
    if (kblock <= 8) return variant == 2 ? stream_update_block_kernel<8, 1, 4> : stream_update_block_kernel<8, 2, 4>;
    return variant == 2 ? stream_update_block_kernel<16, 1, 4> : stream_update_block_kernel<16, 2, 2>;
}
static size_t block_pass_smem(int variant, int kblock, int rpc) {
    const int kmax = kblock <= 8 ? 8 : 16;
    if (block_pass_is_tma(variant))
        return (size_t)LPX_TMA_STAGES * (kblock <= 8 ? sizeof(TmaTile<8>) : sizeof(TmaTile<16>)) + 128;
    return (size_t)kmax * rpc * 8 + (size_t)((rpc + 15) & ~15);
}
static BlockPassFn block_pass_fn(const lpx_session* s) { return block_pass_fn(s->opt.stream_pass_variant, s->P.kblock); }
static size_t block_pass_smem(const lpx_session* s) {
    return block_pass_smem(s->opt.stream_pass_variant, s->P.kblock, s->rpc_block);
}
static void launch_block_pass(lpx_session* s) {
    block_pass_fn(s)<<<s->grid_block, 256, block_pass_smem(s), s->stream>>>(s->P, s->rpc_block);
}

// Rows per CTA and grid of the blocked pass over P (P.kblock > 0), sized to one resident wave; sets the pass
// kernel's shared-memory attribute.
static void size_block_pass(const StreamParams& P, int variant, int* rpc_out, dim3* grid_out) {
    if (block_pass_is_tma(variant)) {
        // TMA-staged pass: strips of 256 columns, row chunks (multiples of 8 rows) sized to one wave
        const size_t smem = block_pass_smem(variant, P.kblock, 0);
        cudaFuncSetAttribute(block_pass_fn(variant, P.kblock), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        int got = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&got, block_pass_fn(variant, P.kblock), 256, smem);
        if (got < 1) got = 1;
        const int bstrips = (P.ld + LPX_TMA_COLS - 1) / LPX_TMA_COLS;
        int ch = std::max(1, (sm_count() * got) / bstrips);
        int rpc = (P.rows + ch - 1) / ch;
        rpc = (rpc + 7) & ~7;
        *rpc_out = rpc;
        *grid_out = dim3(bstrips, (P.rows + rpc - 1) / rpc, 1);
        cudaGetLastError();
        return;
    }
    // blocked pass: column strips x row chunks sized to one resident wave; the factor slices of a
    // chunk must fit in shared memory next to the other resident CTAs
    const int vec = variant == 2 ? 1 : 2;
    const int bstrips = (P.ld / vec + 255) / 256;
    int best_rpc = 0;
    for (int want_occ = 4; want_occ >= 1 && !best_rpc; want_occ--) {
        int ch = std::max(1, (sm_count() * want_occ) / bstrips);
        ch = std::min(ch, P.rows);
        const int rpc = (P.rows + ch - 1) / ch;
        const size_t smem = block_pass_smem(variant, P.kblock, rpc);
        if (smem > (size_t)max_smem_optin()) continue;
        cudaFuncSetAttribute(block_pass_fn(variant, P.kblock), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        int got = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&got, block_pass_fn(variant, P.kblock), 256, smem);
        if (got >= want_occ || want_occ == 1) best_rpc = rpc;
    }
    if (!best_rpc) best_rpc = 64;
    *rpc_out = best_rpc;
    cudaFuncSetAttribute(block_pass_fn(variant, P.kblock), cudaFuncAttributeMaxDynamicSharedMemorySize,
                         (int)block_pass_smem(variant, P.kblock, best_rpc));
    cudaGetLastError();
    *grid_out = dim3(bstrips, (P.rows + best_rpc - 1) / best_rpc, 1);
}

static bool create_priority_stream(cudaStream_t* st) {
    int lo = 0, hi = 0;
    if (cudaDeviceGetStreamPriorityRange(&lo, &hi) != cudaSuccess) hi = 0;
    return cudaStreamCreateWithPriority(st, cudaStreamNonBlocking, hi) == cudaSuccess;  // hi = greatest priority
}

static size_t pipe_pass_smem() { return (size_t)LPX_TMA_STAGES * sizeof(TmaTile<LPX_PIPE_K>) + 128; }

// The pipelined protocol.  Dependencies (B = block index):
//   look-ahead(B) after look-ahead(B-1) and pass(B-2)   [it overwrites the buffer halves of block B-2]
//   pass(B)       after look-ahead(B)   and pass(B-1)   [it reads what pass(B-1) wrote]
// so look-ahead(B+1) runs while pass(B) streams the tableau.  The look-ahead is a cluster of 8 CTAs
// that each need a whole SM; pass(B) and look-ahead(B+1) become ready at the same moment, so the
// look-ahead is enqueued FIRST and on a higher-priority stream: it takes its 8 SMs, the pass (whose
// grid is sized for the remaining SMs) fills the rest.
static int enqueue_pipe_lookahead(lpx_session* s, long long B, int budget, cudaStream_t sl) {
    const int par = (int)(B & 1);
    LPX_CUDA(cudaStreamWaitEvent(sl, s->evL[par ^ 1], 0));
    LPX_CUDA(cudaStreamWaitEvent(sl, s->evP[par], 0));
    stream_lookahead_pipe_kernel<<<LPX_LA_CLUSTER, LPX_LA_THREADS, lookahead_cluster_smem(s->P), sl>>>(s->P, budget, par, 1);
    LPX_CUDA(cudaEventRecord(s->evL[par], sl));
    count_launch();
    return LPX_OK;
}
static int enqueue_pipe_pass(lpx_session* s, long long B) {
    const int par = (int)(B & 1);
    LPX_CUDA(cudaStreamWaitEvent(s->stream, s->evL[par], 0));
    LPX_CUDA(cudaStreamWaitEvent(s->stream, s->evP[par ^ 1], 0));
    stream_update_pipe_tma_kernel<LPX_PIPE_K><<<s->grid_pipe, 256, pipe_pass_smem(), s->stream>>>(s->P, s->rpc_pipe, par);
    LPX_CUDA(cudaEventRecord(s->evP[par], s->stream));
    count_launch();
    return LPX_OK;
}
// `pivots` more pivots: blocks B0 .. B0+nb-1, enqueued as LA(B0), [LA(B0+1), pass(B0)], ..., pass(B0+nb-1)
static int launch_pipe_blocks(lpx_session* s, int pivots, bool serialize) {
    const int K = s->P.kblock;
    const int nb = (pivots + K - 1) / K;
    if (nb <= 0) return LPX_OK;
    cudaStream_t sl = serialize ? s->stream : s->streamL;
    const long long B0 = s->blocks;
    int left = pivots, rc;
    if ((rc = enqueue_pipe_lookahead(s, B0, std::min(left, K), sl)) != LPX_OK) return rc;
    left -= std::min(left, K);
    for (int i = 1; i < nb; i++) {
        if ((rc = enqueue_pipe_lookahead(s, B0 + i, std::min(left, K), sl)) != LPX_OK) return rc;
        left -= std::min(left, K);
        if ((rc = enqueue_pipe_pass(s, B0 + i - 1)) != LPX_OK) return rc;
    }
    if ((rc = enqueue_pipe_pass(s, B0 + nb - 1)) != LPX_OK) return rc;
    LPX_CUDA(cudaGetLastError());
    s->blocks += nb;
    return LPX_OK;
}

// Resolve the status of the tableau as it stands (all passes applied), no pivot.
static int launch_pipe_probe(lpx_session* s) {
    const int par = (int)(s->blocks & 1);
    LPX_CUDA(cudaStreamWaitEvent(s->stream, s->evL[par ^ 1], 0));
    stream_lookahead_pipe_kernel<<<LPX_LA_CLUSTER, LPX_LA_THREADS, lookahead_cluster_smem(s->P), s->stream>>>(s->P, 0, par, 0);
    LPX_CUDA(cudaGetLastError());
    count_launch();
    return LPX_OK;
}

// tableau buffer that holds the current tableau once every launched pass has finished
static int pipe_current_buffer(const lpx_session* s, const StreamCtl& h) {
    if (!s->pipe || s->blocks == 0) return 0;
    const int q = (int)((s->blocks - 1) & 1);
    return h.blk_in[q] ^ (h.blk_cnt[q] > 0 ? 1 : 0);
}

static int launch_block(lpx_session* s, int budget) {
    launch_lookahead(s, budget);
    count_launch();
    if (budget > 0) {
        launch_block_pass(s);
        count_launch();
    }
    LPX_CUDA(cudaGetLastError());
    return LPX_OK;
}

// A session of mm tableau rows (after EQ expansion) and n decision variables, shared by the sessions built from
// (A, b, c) and the re-optimization queries built from a base: the stream, the sizing, every buffer, the protocol
// and the launch grids.  dual: the Dual Simplex rules (limit 10000 dual pivots; the pivot log also holds the up to
// 100 silent pivots of a Dual Simplex session) with the blocked dual look-ahead (stream_dual_lookahead_kernel + the
// blocked pass) or, for stream_protocol 1 / 2 or when its carve does not fit, the per-pivot protocol
// (stream_dual_select_kernel + stream_update_kernel<4>); otherwise opt's Primal Simplex protocol.  m_in / n: the
// model's constraints and variables (b, c).  xcol / xrow: room for one more column past the width (ld) or one more
// row below the z-row (rows, colstride): the direction column g / row h of a parametric working session.  xlog: room
// for that many more pairs in the pivot log.
static lpx_session* session_new(int m_in, int n, int sense, int mm, const lpx_options* opt, bool dual, int xcol = 0,
                                int xrow = 0, int xlog = 0) {
    lpx_session* s = new lpx_session();
    lpx_default_options(&s->opt);
    if (opt) s->opt = *opt;
    s->m_in = m_in;
    s->n = n;
    s->sense = sense;
    s->dual = dual;
    s->device = rt().device;
    if (cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking) != cudaSuccess) {
        set_error("cudaStreamCreate failed");
        delete s;
        return nullptr;
    }
    s->own_stream = true;

    StreamParams& P = s->P;
    P.m = mm;
    P.n = n;
    P.rows = mm + 1 + xrow;
    P.width = n + mm + 1;
    P.ld = (P.width + xcol + 15) & ~15;
    P.colstride = (P.rows + 15) & ~15;
    P.max_iter = dual ? LPX_DUAL_MAX_ITER : s->opt.max_iterations;
    P.pivlog_cap = std::max(1, std::min(P.max_iter, 1 << 20)) + (dual ? LPX_DUAL_SILENT_MAX : 0) + xlog;
    const size_t tbytes = (size_t)P.rows * P.ld * 8;
    P.T = (double*)sess_alloc(s, tbytes);
    P.colbuf = (double*)sess_alloc(s, (size_t)2 * P.colstride * 8);
    P.rhsbuf = (double*)sess_alloc(s, (size_t)P.colstride * 8);
    P.prow = (double*)sess_alloc(s, (size_t)P.ld * 8);
    // the primal ratio test runs over rows, the dual one over columns
    P.ratio = (double*)sess_alloc(s, (size_t)(dual ? std::max(P.colstride, P.ld) : P.colstride) * 8);
    P.basis = (int*)sess_alloc(s, (size_t)mm * 4);
    P.pivlog = (int*)sess_alloc(s, (size_t)P.pivlog_cap * 8);
    P.ctl = (StreamCtl*)sess_alloc(s, sizeof(StreamCtl));
    // multi-CTA prep when the ratio vector fits in one CTA's shared memory (m <= ~25 K rows)
    const int prep_ctas = (P.ld + LPX_PREP_THREADS - 1) / LPX_PREP_THREADS;
    const size_t prep_smem = (size_t)mm * 8;
    P.npartial = (prep_smem + 2048 <= (size_t)max_smem_optin()) ? prep_ctas : 0;
    P.partial = (ArgMin*)sess_alloc(s, (size_t)prep_ctas * sizeof(ArgMin));
    // blocked look-ahead protocol: needs z-row + three row-length vectors in one CTA's shared memory.
    // stream_protocol: 0 auto, 1 single-CTA select per pivot, 2 multi-CTA prep per pivot.  stream_block: pivots per pass.
    P.kblock = 0;
    // stream_protocol == 3 forces the single-CTA look-ahead (tests); otherwise the cluster version is preferred.
    const bool blocked_wanted =
        !dual && (s->opt.stream_protocol == 0 || s->opt.stream_protocol == 3 || s->opt.stream_protocol == 4);
    if (blocked_wanted) {
        const int kb = s->opt.stream_block > 0 ? std::min(s->opt.stream_block, LPX_BLOCK_KMAX) : 8;
        if (s->opt.stream_protocol != 3 && lookahead_cluster_smem(P) + 24 * 1024 <= (size_t)max_smem_optin() &&
            (LPX_LA_CLUSTER <= 8 ||
             (cudaFuncSetAttribute(stream_lookahead_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) ==
                  cudaSuccess &&
              cudaFuncSetAttribute(stream_lookahead_pipe_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) ==
                  cudaSuccess)) &&
            cudaFuncSetAttribute(stream_lookahead_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)lookahead_cluster_smem(P)) == cudaSuccess) {
            P.kblock = kb;
            s->la_cluster = true;
        } else if (lookahead_smem(P) + 4096 <= (size_t)max_smem_optin() &&
                   cudaFuncSetAttribute(stream_lookahead_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)lookahead_smem(P)) == cudaSuccess) {
            P.kblock = kb;
        }
        cudaGetLastError();
    }
    if (dual && (s->opt.stream_protocol == 0 || s->opt.stream_protocol == 3 || s->opt.stream_protocol == 4)) {
        // blocked dual look-ahead: one CTA, not pipelined; z-row + compact RHS + one column in shared memory
        const int kb = s->opt.stream_block > 0 ? std::min(s->opt.stream_block, LPX_BLOCK_KMAX) : 8;
        if (dual_lookahead_smem(P) + 4096 <= (size_t)max_smem_optin() &&
            cudaFuncSetAttribute(stream_dual_lookahead_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)dual_lookahead_smem(P)) == cudaSuccess)
            P.kblock = kb;
        cudaGetLastError();
    }
    if (dual || s->opt.stream_protocol == 1) P.npartial = 0;
    // stream_protocol 0: pipelined when the cluster look-ahead is available and the block size allows it
    // (<= 8 pivots per block); 4 forces the non-pipelined blocked protocol.
    const bool want_pipe = s->opt.stream_protocol == 0 && s->la_cluster && P.kblock > 0 && P.kblock <= LPX_PIPE_K;
    // factor columns and pivot rows of the blocks in flight, in ONE allocation: the look-ahead re-reads all
    // pending entries for every pivot it decides, so they are pinned in L2 (access policy window below)
    const size_t fbytes = (size_t)LPX_BLOCK_KMAX * P.colstride * 8, pbytes = (size_t)LPX_BLOCK_KMAX * P.ld * 8;
    P.Fbuf = (double*)sess_alloc(s, fbytes + pbytes);
    P.Pbuf = P.Fbuf ? P.Fbuf + (size_t)LPX_BLOCK_KMAX * P.colstride : nullptr;
    P.Lbuf = (int*)sess_alloc(s, (size_t)LPX_BLOCK_KMAX * 4);
    P.dbg = (unsigned long long*)sess_alloc(s, 16 * 8);
    P.T1 = nullptr;
    P.zbuf = nullptr;
    if (want_pipe) {
        P.T1 = (double*)sess_alloc(s, tbytes);
        P.zbuf = (double*)sess_alloc(s, (size_t)P.ld * 8);
        bool ok = P.T1 && P.zbuf &&
                  cudaFuncSetAttribute(stream_lookahead_pipe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)lookahead_cluster_smem(P)) == cudaSuccess &&
                  cudaFuncSetAttribute(stream_update_pipe_tma_kernel<LPX_PIPE_K>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pipe_pass_smem()) == cudaSuccess &&
                  create_priority_stream(&s->streamL);
        for (int k = 0; k < 2 && ok; k++)
            ok = cudaEventCreateWithFlags(&s->evL[k], cudaEventDisableTiming) == cudaSuccess &&
                 cudaEventCreateWithFlags(&s->evP[k], cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&s->evStart, cudaEventDisableTiming) == cudaSuccess;
        if (ok && !getenv("LPX_NO_L2_PIN")) {
            // The pass streams 800 MB through L2 per block and would evict the 2 MB of pending factor columns /
            // pivot rows the concurrent look-ahead needs again for each of its 8 pivots (16 dependent round
            // trips per block, each queueing behind a saturated HBM).  Keep them resident: a persisting-L2
            // carve-out and an access-policy window on both streams.  Best effort: failures are ignored.
            cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, (size_t)8 << 20);
            cudaStreamAttrValue av;
            std::memset(&av, 0, sizeof av);
            av.accessPolicyWindow.base_ptr = P.Fbuf;
            av.accessPolicyWindow.num_bytes = fbytes + pbytes;
            av.accessPolicyWindow.hitRatio = 1.0f;
            av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
            av.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
            cudaStreamSetAttribute(s->streamL, cudaStreamAttributeAccessPolicyWindow, &av);
            cudaStreamSetAttribute(s->stream, cudaStreamAttributeAccessPolicyWindow, &av);
        }
        cudaGetLastError();
        s->pipe = ok;
        if (!ok) P.zbuf = nullptr;  // fall back to the non-pipelined blocked protocol
    }
    if (P.npartial > 0 && prep_smem > 40 * 1024 &&
        cudaFuncSetAttribute(stream_prep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)prep_smem) !=
            cudaSuccess)
        P.npartial = 0;
    s->sens_b = (double*)sess_alloc(s, (size_t)m_in * 8);
    s->sens_c = (double*)sess_alloc(s, (size_t)n * 8);
    s->sens_rmap = (int*)sess_alloc(s, (size_t)m_in * 4);
    if (!P.T || !P.colbuf || !P.rhsbuf || !P.prow || !P.ratio || !P.basis || !P.pivlog || !P.ctl || !P.partial || !P.Fbuf ||
        !P.Pbuf || !P.Lbuf || !s->sens_b || !s->sens_c || !s->sens_rmap) {
        sess_free(s);
        return nullptr;
    }
    if (cudaMemsetAsync(P.colbuf, 0, (size_t)2 * P.colstride * 8, s->stream) != cudaSuccess ||
        cudaMemsetAsync(P.rhsbuf, 0, (size_t)P.colstride * 8, s->stream) != cudaSuccess) {
        cuda_fail(cudaGetLastError(), "session setup", __FILE__, __LINE__);
        sess_free(s);
        return nullptr;
    }
    // update grid: column strips x row chunks sized to one resident wave
    int occ = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, stream_update_kernel<4>, 256, 0);
    if (occ < 1) occ = 1;
    const int strips = (P.ld / 2 + 255) / 256;
    int chunks = (sm_count() * occ) / strips;
    chunks = std::max(1, std::min(chunks, P.rows));
    s->grid_update = dim3(strips, chunks, 1);
    if (s->pipe) {
        int got = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&got, stream_update_pipe_tma_kernel<LPX_PIPE_K>, 256, pipe_pass_smem());
        if (got < 1) got = 1;
        // the look-ahead cluster of the next block occupies LPX_LA_CLUSTER SMs while the pass runs
        const int sms = sm_count() > 4 * LPX_LA_CLUSTER ? sm_count() - LPX_LA_CLUSTER : sm_count();
        const int bstrips = (P.ld + LPX_TMA_COLS - 1) / LPX_TMA_COLS;
        const int ch = std::max(1, (sms * got) / bstrips);
        int rpc = (P.rows + ch - 1) / ch;
        rpc = (rpc + 7) & ~7;
        s->rpc_pipe = rpc;
        s->grid_pipe = dim3(bstrips, (P.rows + rpc - 1) / rpc, 1);
        cudaGetLastError();
    }
    if (P.kblock > 0) size_block_pass(P, s->opt.stream_pass_variant, &s->rpc_block, &s->grid_block);
    return s;
}

// The silent phase of a Dual Simplex session (DualSimplex.ForceDualFeasibility): at most 100 Primal Simplex pivots with
// the ratio margin 1e-12, on the per-pivot single-CTA primal protocol.  It ends, with no status, on no entering column,
// no leaving row or the guard; the select kernel marks those OPTIMAL / UNBOUNDED / ITER_LIMIT (with max_iter = 100
// during the phase) and makes every later launch of the phase a no-op, so the 100 pairs are enqueued at once and the
// control block is re-armed for the Dual Simplex loop afterwards.  Runs synchronously, inside open.
static int session_dual_silent_phase(lpx_session* s) {
    StreamParams F = s->P;
    F.max_iter = LPX_DUAL_SILENT_MAX;
    F.npartial = 0;
    cudaStream_t st = s->stream;
    stream_first_kernel<<<1, 1024, 0, st>>>(F);
    stream_gather_kernel<<<(F.rows + 255) / 256, 256, 0, st>>>(F);
    count_launch(2);
    for (int k = 0; k < LPX_DUAL_SILENT_MAX; k++) {
        stream_select_kernel<true><<<1, 1024, 0, st>>>(F, 0);
        stream_update_kernel<4><<<s->grid_update, 256, 0, st>>>(F);
        count_launch(2);
    }
    LPX_CUDA(cudaGetLastError());
    StreamCtl h;
    LPX_CUDA(cudaMemcpyAsync(&h, F.ctl, sizeof h, cudaMemcpyDeviceToHost, st));
    LPX_CUDA(cudaStreamSynchronize(st));
    s->silent = h.pivots;
    h.status = LPX_RUNNING;
    h.enter = -1;
    h.leave = -1;
    h.active = 0;
    h.capture = -1;
    h.block_cnt = 0;
    LPX_CUDA(cudaMemcpyAsync(F.ctl, &h, sizeof h, cudaMemcpyHostToDevice, st));
    LPX_CUDA(cudaStreamSynchronize(st));
    s->P.max_iter = s->silent + LPX_DUAL_MAX_ITER;  // the limit counts Dual Simplex pivots only
    return LPX_OK;
}

// A, b, c: device pointers valid until this call returns (setup runs synchronously).  dual: a Dual Simplex session
// (DualSimplex.Solve); hb is then b on the host, for the row signs of DualSimplex.PrepareForTableau.
static lpx_session* session_create(int m, int n, int sense, const double* dA, const int* rel, const double* db,
                                   const double* dc, const lpx_options* opt, bool dual = false,
                                   const double* hb = nullptr) {
    if (ensure_device() != LPX_OK) return nullptr;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    // row map of the EQ expansion, and the first '>=' row, both known from rel on the host.  Dual Simplex row signs
    // (PrepareForTableau): an EQ row as given, then negated; a GE row negated, then negated back when the negated b is
    // below -1e-9 (so flipped unless -b < -1e-9); an LE row negated when b < -1e-9.  No GE / negative-RHS validation.
    std::vector<int> rsrc, rsgn, rmap;
    int first_ge = INT_MAX;
    for (int r = 0; r < m; r++) {
        const int rl = rel ? rel[r] : 0;
        if (rl == 1 && first_ge == INT_MAX) first_ge = r;
        rmap.push_back(rl == 2 ? -(int)rsrc.size() - 1 : (int)rsrc.size());
        rsrc.push_back(r);
        int flip = 0;
        if (dual && rl == 1) flip = !(-hb[r] < -LPX_EPS);
        if (dual && rl == 0) flip = hb[r] < -LPX_EPS;
        rsgn.push_back(flip);
        if (rl == 2) {
            rsrc.push_back(r);
            rsgn.push_back(1);
        }
    }
    const int mm = (int)rsrc.size();
    lpx_session* s = session_new(m, n, sense, mm, opt, dual);
    if (!s) return nullptr;
    s->rmap = rmap;
    s->dual_model = dual;
    s->sens_ok = !dual;
    StreamParams& P = s->P;
    int* drsrc = (int*)sess_alloc(s, (size_t)mm * 4);
    int* drsgn = (int*)sess_alloc(s, (size_t)mm * 4);
    if (!drsrc || !drsgn) {
        sess_free(s);
        return nullptr;
    }
    cudaStream_t st = s->stream;
    bool ok = true;
    ok = ok && cudaMemcpyAsync(drsrc, rsrc.data(), (size_t)mm * 4, cudaMemcpyHostToDevice, st) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(drsgn, rsgn.data(), (size_t)mm * 4, cudaMemcpyHostToDevice, st) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(s->sens_b, db, (size_t)m * 8, cudaMemcpyDeviceToDevice, st) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(s->sens_c, dc, (size_t)n * 8, cudaMemcpyDeviceToDevice, st) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(s->sens_rmap, rmap.data(), (size_t)m * 4, cudaMemcpyHostToDevice, st) == cudaSuccess;
    if (ok && dual) {
        // validate with no constraints only resets StreamCtl to RUNNING, 0 pivots
        stream_validate_kernel<<<1, 1024, 0, st>>>(P.ctl, nullptr, 0, INT_MAX);
        const int bgrid = std::min(P.rows, sm_count() * 8);
        stream_build_kernel<<<bgrid, 256, 0, st>>>(P, dA, db, dc, drsrc, drsgn, sense);
        count_launch(2);
        ok = cudaGetLastError() == cudaSuccess && session_dual_silent_phase(s) == LPX_OK;
    } else if (ok) {
        stream_validate_kernel<<<1, 1024, 0, st>>>(P.ctl, db, m, first_ge);
        const int bgrid = std::min(P.rows, sm_count() * 8);
        stream_build_kernel<<<bgrid, 256, 0, st>>>(P, dA, db, dc, drsrc, drsgn, sense);
        stream_first_kernel<<<1, 1024, 0, st>>>(P);
        stream_gather_kernel<<<(P.rows + 255) / 256, 256, 0, st>>>(P);
        count_launch(4);
        ok = cudaGetLastError() == cudaSuccess && cudaStreamSynchronize(st) == cudaSuccess;
    }
    if (!ok) {
        cuda_fail(cudaGetLastError(), "session setup", __FILE__, __LINE__);
        sess_free(s);
        return nullptr;
    }
    return s;
}

// The terms of a change d[m_in] of b (RHS and COL edits, the parametric RHS direction), in the definition's order:
// d_i * T[r][s1], and for an EQ row - d_i * T[r][s2].
static void slack_terms(const lpx_session* base, const double* d, std::vector<ReoptTerm>& terms) {
    for (int i = 0; i < base->m_in; i++) {
        if (d[i] == 0.0) continue;
        const int r = base->rmap[i];
        const int s1 = base->n + (r < 0 ? -r - 1 : r);
        terms.push_back(ReoptTerm{d[i], s1, 0});
        if (r < 0) terms.push_back(ReoptTerm{d[i], s1 + 1, 1});
    }
}

// The terms of a change d[n] of c in the model's sense (COST edits, the parametric COST direction): delta_j with the
// basic row of column j (-1: non-basic).  bb: the base's basis.
static void cost_terms(const lpx_session* base, const std::vector<int>& bb, const double* d,
                       std::vector<ReoptTerm>& terms) {
    const int n = base->n;
    std::vector<int> rowof(n, -1);
    for (int r = 0; r < (int)bb.size(); r++)
        if (bb[r] < n) rowof[bb[r]] = r;
    for (int j = 0; j < n; j++) {
        if (d[j] == 0.0) continue;
        terms.push_back(ReoptTerm{base->sense == 1 ? -d[j] : d[j], rowof[j], j});
    }
}

// lpx_session_reoptimize: the query session of one what-if edit of an optimal base session (include/lpx.h,
// "Re-optimization").  The terms of the edit are listed on the host in the definition's order; the build kernel
// writes the query's tableau straight from the base's current buffer, then the query's protocol is armed as a new
// session's is.  The base is only read, and is idle once this returns (setup runs synchronously).
static lpx_session* session_reoptimize(const lpx_session* base, int kind, const double* pay, const lpx_options* opt) {
    if (base->dual_model) {
        set_error("lpx_session_reoptimize: the base is a Dual Simplex session; re-optimization is defined for Primal "
                  "Simplex results");
        return nullptr;
    }
    const StreamParams& B = base->P;
    const int m_in = base->m_in, n = base->n, mb = B.m;
    StreamCtl h;
    std::vector<int> bb(mb);
    std::vector<double> hb(m_in), hc(n);
    if (cudaMemcpyAsync(&h, B.ctl, sizeof h, cudaMemcpyDeviceToHost, base->stream) != cudaSuccess ||
        cudaMemcpyAsync(bb.data(), B.basis, (size_t)mb * 4, cudaMemcpyDeviceToHost, base->stream) != cudaSuccess ||
        cudaMemcpyAsync(hb.data(), base->sens_b, (size_t)m_in * 8, cudaMemcpyDeviceToHost, base->stream) != cudaSuccess ||
        cudaMemcpyAsync(hc.data(), base->sens_c, (size_t)n * 8, cudaMemcpyDeviceToHost, base->stream) != cudaSuccess ||
        cudaStreamSynchronize(base->stream) != cudaSuccess) {
        cuda_fail(cudaGetLastError(), "lpx_session_reoptimize: reading the base", __FILE__, __LINE__);
        return nullptr;
    }
    if (h.status != LPX_OPTIMAL) {
        set_error("lpx_session_reoptimize: the base session's status is " + std::to_string(h.status) +
                  ", not LPX_OPTIMAL (step or sync it to OPTIMAL first)");
        return nullptr;
    }
    const double* Tb = (base->pipe && pipe_current_buffer(base, h)) ? B.T1 : B.T;
    const bool ge = kind == LPX_REOPT_ROW && pay[n] == 1.0;
    // the terms, and the query's basis, model vectors (b, c: what the sensitivity report of an RHS / COST query
    // reads) and constraint map
    std::vector<ReoptTerm> terms;
    std::vector<int> qb(bb), qmap(base->rmap);
    std::vector<double> qbv(hb), qcv(hc);
    double zstart = 0.0;
    if (kind == LPX_REOPT_RHS) {
        slack_terms(base, pay, terms);
        for (int i = 0; i < m_in; i++) qbv[i] = hb[i] + pay[i];
    } else if (kind == LPX_REOPT_COST) {
        cost_terms(base, bb, pay, terms);
        for (int j = 0; j < n; j++) qcv[j] = hc[j] + pay[j];
    } else if (kind == LPX_REOPT_ROW) {
        for (int r = 0; r < mb; r++) {
            const int j = bb[r];
            if (j >= n || pay[j] == 0.0) continue;
            terms.push_back(ReoptTerm{ge ? -pay[j] : pay[j], r, 0});
        }
        qb.push_back(B.width - 1);  // the new slack is basic in the new row
        qmap.push_back(mb);
        qbv.push_back(ge ? -pay[n + 1] : pay[n + 1]);
    } else {
        slack_terms(base, pay, terms);
        const double cp = base->sense == 1 ? -pay[m_in] : pay[m_in];
        zstart = -cp;
        for (int& j : qb)
            if (j >= n) j++;
        qcv.push_back(pay[m_in]);
    }
    const bool dual = kind == LPX_REOPT_RHS || kind == LPX_REOPT_ROW;
    const int qm_in = (int)qmap.size(), qn = kind == LPX_REOPT_COL ? n + 1 : n, qmm = (int)qb.size();
    lpx_session* s = session_new(qm_in, qn, base->sense, qmm, opt ? opt : &base->opt, dual);
    if (!s) return nullptr;
    s->rmap = qmap;
    s->sens_ok = base->sens_ok && (kind == LPX_REOPT_RHS || kind == LPX_REOPT_COST);
    const size_t stride = lpx_reopt_payload_stride(kind, m_in, n);
    ReoptTerm* dterms = (ReoptTerm*)sess_alloc(s, std::max<size_t>(terms.size(), 1) * sizeof(ReoptTerm));
    double* dpay = (double*)sess_alloc(s, stride * 8);
    if (!dterms || !dpay) {
        sess_free(s);
        return nullptr;
    }
    StreamParams& P = s->P;
    cudaStream_t st = s->stream;
    bool ok = true;
    ok = ok && (terms.empty() || cudaMemcpyAsync(dterms, terms.data(), terms.size() * sizeof(ReoptTerm),
                                                 cudaMemcpyHostToDevice, st) == cudaSuccess);
    ok = ok && cudaMemcpyAsync(dpay, pay, stride * 8, cudaMemcpyHostToDevice, st) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(P.basis, qb.data(), (size_t)qmm * 4, cudaMemcpyHostToDevice, st) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(s->sens_b, qbv.data(), (size_t)qm_in * 8, cudaMemcpyHostToDevice, st) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(s->sens_c, qcv.data(), (size_t)qn * 8, cudaMemcpyHostToDevice, st) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(s->sens_rmap, qmap.data(), (size_t)qm_in * 4, cudaMemcpyHostToDevice, st) == cudaSuccess;
    if (ok) {
        // validate with no constraints only resets StreamCtl to RUNNING, 0 pivots
        stream_validate_kernel<<<1, 1024, 0, st>>>(P.ctl, nullptr, 0, INT_MAX);
        const int strips = (P.ld + 255) / 256;
        const int groups = std::max(1, std::min(P.rows, sm_count() * 8 / strips));
        stream_reopt_build_kernel<<<dim3(strips, groups, 1), 256, 0, st>>>(P, Tb, B.ld, B.width, mb, n, kind, dterms,
                                                                            (int)terms.size(), dpay, zstart, ge ? 1 : 0);
        if (!dual) {
            stream_first_kernel<<<1, 1024, 0, st>>>(P);
            count_launch();
        }
        stream_gather_kernel<<<(P.rows + 255) / 256, 256, 0, st>>>(P);  // dual: no entering column, the RHS only
        count_launch(3);
        ok = cudaGetLastError() == cudaSuccess && cudaStreamSynchronize(st) == cudaSuccess;
    }
    if (!ok) {
        cuda_fail(cudaGetLastError(), "lpx_session_reoptimize: setup", __FILE__, __LINE__);
        sess_free(s);
        return nullptr;
    }
    return s;
}

// Where a single-CTA look-ahead keeps its vectors: in dynamic shared memory, in the order given, each one that fits next
// to those placed before it; the others in global memory (`scratch`, every vector's home back to back in that order,
// which L2 holds).  Every shape runs: at worst every vector is in global memory.  Returns the dynamic shared-memory
// bytes.
static size_t vec_place(const size_t* len, const int* order, int nv, double* scratch, double** gvec, int* soff) {
    const size_t cap = ((size_t)max_smem_optin() - 4096) / 8;  // 4 KB for the kernel's static shared memory
    size_t used = 0, g = 0;
    for (int k = 0; k < nv; k++) {
        const int v = order[k];
        gvec[v] = scratch + g;
        g += len[v];
        soff[v] = -1;
        if (used + len[v] <= cap) {
            soff[v] = (int)used;
            used += len[v];
        }
    }
    return used * 8;
}

// The parametric look-ahead's vectors (scratch: 2 ld + 3 colstride doubles).
static size_t param_place(const StreamParams& P, bool cost, double* scratch, ParamLa& A) {
    size_t len[PV_N];
    len[PV_Z] = P.ld;
    len[PV_HG] = cost ? P.ld : P.colstride;
    len[PV_RHS] = P.colstride;
    len[PV_COL] = P.colstride;
    len[PV_RATIO] = cost ? P.colstride : P.ld;
    const int order[PV_N] = {PV_RHS, PV_COL, PV_HG, PV_RATIO, PV_Z};
    return vec_place(len, order, PV_N, scratch, A.gvec, A.soff);
}

// lpx_session_parametric with its arguments checked.  A working session of the working shape (RHS: ld with room for
// g at column W, P.width = W so every rule still finds the RHS at W - 1; COST: h as row m' + 1, P.rows = m' + 2 with
// the z-row still at P.m = m') is built from the base's current buffer; then blocks of stream_param_lookahead_kernel
// + the blocked pass are enqueued in chunks behind the device status word (ParamState::end), one synchronise per
// chunk, and the outputs are copied out.  The base is only read.
static int session_parametric(const lpx_session* base, int kind, const double* pay, int seg_cap, const lpx_options* opt,
                              int* end, int* n_segments, int* n_pivots, double* segments, int* seg_pivots, int* basis,
                              double* tableau) {
    const StreamParams& B = base->P;
    const int n = base->n, mb = B.m, W = B.width;
    const bool cost = kind == LPX_PARAM_COST;
    const int rows = mb + 1 + (cost ? 1 : 0), cols = W + (cost ? 0 : 1);
    const size_t sstride = lpx_param_segment_stride(n), cap = (size_t)seg_cap;
    StreamCtl h;
    std::vector<int> bb(mb);
    LPX_CUDA(cudaMemcpyAsync(&h, B.ctl, sizeof h, cudaMemcpyDeviceToHost, base->stream));
    LPX_CUDA(cudaMemcpyAsync(bb.data(), B.basis, (size_t)mb * 4, cudaMemcpyDeviceToHost, base->stream));
    LPX_CUDA(cudaStreamSynchronize(base->stream));
    if (h.status != LPX_OPTIMAL) {
        *end = LPX_PARAM_NO_BASE;
        if (n_segments) *n_segments = 0;
        if (n_pivots) *n_pivots = 0;
        if (segments) std::fill(segments, segments + cap * sstride, 0.0);
        if (seg_pivots) std::fill(seg_pivots, seg_pivots + 2 * cap, -1);
        if (basis) std::fill(basis, basis + mb, 0);
        if (tableau) std::fill(tableau, tableau + (size_t)rows * cols, 0.0);
        return LPX_OK;
    }
    const double* Tb = (base->pipe && pipe_current_buffer(base, h)) ? B.T1 : B.T;
    std::vector<ReoptTerm> terms;
    if (cost)
        cost_terms(base, bb, pay, terms);
    else
        slack_terms(base, pay, terms);
    // the working session always runs the parametric look-ahead and the blocked pass; protocol 4 (blocked, not
    // pipelined) keeps session_new from allocating the pipelined protocol's second tableau
    lpx_options o = opt ? *opt : base->opt;
    o.stream_protocol = 4;
    lpx_session* s = session_new(base->m_in, n, base->sense, mb, &o, false, cost ? 0 : 1, cost ? 1 : 0);
    if (!s) return LPX_E_CUDA;
    StreamParams& P = s->P;
    P.kblock = o.stream_block > 0 ? std::min(o.stream_block, LPX_BLOCK_KMAX) : 8;
    size_block_pass(P, o.stream_pass_variant, &s->rpc_block, &s->grid_block);
    double* dvec = (double*)sess_alloc(s, (2 * (size_t)P.ld + 3 * (size_t)P.colstride) * 8);
    ParamState* dstate = (ParamState*)sess_alloc(s, sizeof(ParamState));
    int* disb = cost ? (int*)sess_alloc(s, (size_t)W * 4) : nullptr;
    ReoptTerm* dterms = (ReoptTerm*)sess_alloc(s, std::max<size_t>(terms.size(), 1) * sizeof(ReoptTerm));
    double* dseg = segments ? (double*)sess_alloc(s, cap * sstride * 8) : nullptr;
    int* dspv = seg_pivots ? (int*)sess_alloc(s, cap * 2 * 4) : nullptr;
    if (!dvec || !dstate || (cost && !disb) || !dterms || (segments && !dseg) || (seg_pivots && !dspv)) {
        sess_free(s);
        return LPX_E_CUDA;
    }
    ParamLa A{};
    const size_t smem = param_place(P, cost, dvec, A);
    A.isb = disb;
    A.st = dstate;
    A.seg = dseg;
    A.spv = dspv;
    A.seg_cap = seg_cap;
    A.n = n;
    A.theta_max = pay[lpx_param_payload_stride(kind, base->m_in, n) - 1];
    void (*la)(StreamParams, ParamLa) = cost ? stream_param_lookahead_kernel<true> : stream_param_lookahead_kernel<false>;
    const ParamState h0{0.0, 0, -1};
    std::vector<int> isb(cost ? W : 0, 0);
    for (int r = 0; r < mb && cost; r++) isb[bb[r]] = 1;
    cudaStream_t st = s->stream;
    bool ok = cudaFuncSetAttribute(la, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess;
    ok = ok && (terms.empty() || cudaMemcpyAsync(dterms, terms.data(), terms.size() * sizeof(ReoptTerm),
                                                 cudaMemcpyHostToDevice, st) == cudaSuccess);
    ok = ok && cudaMemcpyAsync(dstate, &h0, sizeof h0, cudaMemcpyHostToDevice, st) == cudaSuccess;
    ok = ok && (!cost || cudaMemcpyAsync(disb, isb.data(), (size_t)W * 4, cudaMemcpyHostToDevice, st) == cudaSuccess);
    ok = ok && cudaMemcpyAsync(P.basis, bb.data(), (size_t)mb * 4, cudaMemcpyHostToDevice, st) == cudaSuccess;
    ok = ok && (!dseg || cudaMemsetAsync(dseg, 0, cap * sstride * 8, st) == cudaSuccess);
    ok = ok && (!dspv || cudaMemsetAsync(dspv, 0xff, cap * 2 * 4, st) == cudaSuccess);  // (-1, -1)
    if (ok) {
        // validate with no constraints only resets StreamCtl (0 pivots, block_cnt 0)
        stream_validate_kernel<<<1, 1024, 0, st>>>(P.ctl, nullptr, 0, INT_MAX);
        const int strips = (P.ld + 255) / 256;
        const int groups = std::max(1, std::min(P.rows, sm_count() * 8 / strips));
        stream_param_build_kernel<<<dim3(strips, groups, 1), 256, 0, st>>>(P, Tb, B.ld, mb, cost ? 1 : 0, dterms,
                                                                           (int)terms.size());
        count_launch(2);
        if (!cost) {
            stream_param_g_kernel<<<(P.rows + LPX_PARAM_G_THREADS - 1) / LPX_PARAM_G_THREADS, LPX_PARAM_G_THREADS, 0,
                                    st>>>(P, Tb, B.ld, dterms, (int)terms.size());
            count_launch();
        }
        ok = cudaGetLastError() == cudaSuccess;
    }
    // every block but the last decides K pivots, and there are at most seg_cap - 1 of them
    const long long max_blocks = (cap - 1 + P.kblock - 1) / P.kblock + 1;
    long long launched = 0;
    int chunk = 1;
    ParamState hs = h0;
    while (ok) {
        const int todo = (int)std::min<long long>(chunk, max_blocks - launched);
        for (int b = 0; b < todo; b++) {
            la<<<1, 1024, smem, st>>>(P, A);
            launch_block_pass(s);
            count_launch(2);
        }
        launched += todo;
        ok = cudaGetLastError() == cudaSuccess &&
             cudaMemcpyAsync(&hs, dstate, sizeof hs, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
             cudaStreamSynchronize(st) == cudaSuccess;
        if (!ok || hs.end >= 0) break;
        if (launched >= max_blocks) {
            set_error("lpx_session_parametric: the analysis did not end within seg_cap segments");
            sess_free(s);
            return LPX_E_CUDA;
        }
        chunk = std::min(2 * chunk, 64);
    }
    if (ok) {
        *end = hs.end;
        if (n_segments) *n_segments = hs.k;
        if (n_pivots) *n_pivots = hs.k - 1;
        auto down = [&](void* dst, const void* from, size_t bytes) {
            return !dst || cudaMemcpyAsync(dst, from, bytes, cudaMemcpyDeviceToHost, st) == cudaSuccess;
        };
        ok = down(segments, dseg, cap * sstride * 8) && down(seg_pivots, dspv, cap * 2 * 4) &&
             down(basis, P.basis, (size_t)mb * 4) &&
             (!tableau || cudaMemcpy2DAsync(tableau, (size_t)cols * 8, P.T, (size_t)P.ld * 8, (size_t)cols * 8, rows,
                                            cudaMemcpyDeviceToHost, st) == cudaSuccess) &&
             cudaStreamSynchronize(st) == cudaSuccess;
    }
    if (!ok) {
        cuda_fail(cudaGetLastError(), "lpx_session_parametric", __FILE__, __LINE__);
        sess_free(s);
        return LPX_E_CUDA;
    }
    sess_free(s);
    return LPX_OK;
}

// lpx_two_phase_session_open(_dev) with its arguments checked.  A, b, c: device pointers valid until this returns
// (setup runs synchronously); rel, hb: host.  The normalisation, the column numbering, a, W and S come from rel and b on
// the host; the session has m + 2 rows of width W and always runs the two-phase look-ahead with the blocked pass.
static lpx_session* session_two_phase(int m, int n, int sense, const double* dA, const int* rel, const double* db,
                                      const double* dc, const double* hb, const lpx_options* opt) {
    std::vector<int> info((size_t)4 * m);  // flip | slk | art | the artificial rows in row order
    int* flip = info.data();
    int *slk = flip + m, *art = slk + m, *arows = art + m;
    int ns = n;
    for (int i = 0; i < m; i++) ns += (rel && rel[i] == 2) ? 0 : 1;
    int sk = n, a = 0;
    double S = 0.0;
    for (int i = 0; i < m; i++) {
        const int rl = rel ? rel[i] : 0;
        flip[i] = hb[i] < 0.0;
        const int rn = (flip[i] && rl != 2) ? 1 - rl : rl;
        slk[i] = rl != 2 ? sk++ : -1;
        art[i] = -1;
        if (rn != 0) {
            art[i] = ns + a;
            arows[a++] = i;
            S += flip[i] ? -hb[i] : hb[i];
        }
    }
    const int W = ns + a + 1;
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    o.stream_protocol = 4;  // blocked, not pipelined: session_new allocates no second tableau and no L2 window
    // W - (n + m + 1) >= 0 more columns: every EQ row has an artificial, so s + a >= m
    lpx_session* s = session_new(m, n, sense, m, &o, false, W - (n + m + 1), 1, m);
    if (!s) return nullptr;
    s->two_phase = true;
    s->sens_ok = false;
    s->tp_ns = ns;
    StreamParams& P = s->P;
    P.width = W;
    P.kblock = o.stream_block > 0 ? std::min(o.stream_block, LPX_BLOCK_KMAX) : 8;
    size_block_pass(P, o.stream_pass_variant, &s->rpc_block, &s->grid_block);
    double* dvec = (double*)sess_alloc(s, ((size_t)P.ld + 3 * (size_t)P.colstride) * 8);
    TwoPhaseState* dstate = (TwoPhaseState*)sess_alloc(s, sizeof(TwoPhaseState));
    int* dinfo = (int*)sess_alloc(s, info.size() * 4);
    if (!dvec || !dstate || !dinfo) {
        sess_free(s);
        return nullptr;
    }
    size_t len[TV_N];
    len[TV_Z] = P.ld;
    len[TV_RHS] = P.colstride;
    len[TV_COL] = P.colstride;
    len[TV_RATIO] = P.colstride;
    const int order[TV_N] = {TV_RHS, TV_COL, TV_RATIO, TV_Z};
    s->tla_smem = vec_place(len, order, TV_N, dvec, s->tla.gvec, s->tla.soff);
    s->tla.st = dstate;
    s->tla.ns = ns;
    s->tp_info = dinfo;
    const TwoPhaseRows R{dinfo, dinfo + m, dinfo + 2 * m, dinfo + 3 * m, a};
    TwoPhaseState h0{};
    h0.phase = 1;
    h0.S = S;
    cudaStream_t st = s->stream;
    bool ok = cudaFuncSetAttribute(stream_two_phase_lookahead_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)s->tla_smem) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(dinfo, info.data(), info.size() * 4, cudaMemcpyHostToDevice, st) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(dstate, &h0, sizeof h0, cudaMemcpyHostToDevice, st) == cudaSuccess;
    // the model's b and c, for the sensitivity report
    ok = ok && cudaMemcpyAsync(s->sens_b, db, (size_t)m * 8, cudaMemcpyDeviceToDevice, st) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(s->sens_c, dc, (size_t)n * 8, cudaMemcpyDeviceToDevice, st) == cudaSuccess;
    if (ok) {
        // validate with no constraints only resets StreamCtl to RUNNING, 0 pivots, no entering column
        stream_validate_kernel<<<1, 1024, 0, st>>>(P.ctl, nullptr, 0, INT_MAX);
        const int strips = (P.ld + 255) / 256;
        const int groups = std::max(1, std::min(P.rows, sm_count() * 8 / strips));
        stream_two_phase_build_kernel<<<dim3(strips, groups, 1), 256, 0, st>>>(P, dA, db, dc, R, sense, ns);
        stream_gather_kernel<<<(P.rows + 255) / 256, 256, 0, st>>>(P);  // the compact RHS
        count_launch(3);
        ok = cudaGetLastError() == cudaSuccess && cudaStreamSynchronize(st) == cudaSuccess;
    }
    if (!ok) {
        cuda_fail(cudaGetLastError(), "lpx_two_phase_session_open: setup", __FILE__, __LINE__);
        sess_free(s);
        return nullptr;
    }
    return s;
}

int stream_solve_host(int m, int n, int sense, const double* A, const int* rel, const double* b, const double* c,
                      const lpx_options* opt, int* status, int* n_pivots, int* pivots, int pivots_cap, int* basis,
                      double* x, double* z, double* tableau, double* history, int history_cap) {
    if (history && history_cap > 0) {
        set_error("per-iteration history is not available on the streaming kernel; use LPX_KERNEL_CTA_GLOBAL");
        return LPX_E_CAPACITY;
    }
    lpx_session* s = lpx_session_open(m, n, sense, A, rel, b, c, opt);
    if (!s) return LPX_E_CUDA;
    int st = LPX_RUNNING, np = 0, rc = LPX_OK;
    while (st == LPX_RUNNING && rc == LPX_OK) rc = lpx_session_step(s, 512, &st, &np);
    if (rc == LPX_OK) {
        if (status) *status = st;
        if (n_pivots) *n_pivots = np;
        if (pivots && pivots_cap > 0) rc = lpx_session_read_pivots(s, pivots, pivots_cap);
        const bool solved = st >= 0 || st == LPX_S_ITER_LIMIT;
        if (rc == LPX_OK && solved && (basis || x || z)) rc = lpx_session_read_solution(s, basis, x, z);
        if (rc == LPX_OK && solved && tableau) rc = lpx_session_read_tableau(s, tableau);
    }
    lpx_session_close(s);
    return rc;
}

// lpx_dual_solve with kernel = LPX_KERNEL_STREAM: one Dual Simplex session stepped to its terminal status.
int stream_dual_solve_host(int m, int n, int sense, const double* A, const int* rel, const double* b, const double* c,
                           const lpx_options* opt, int* status, int* n_pivots, int* silent_pivots, int* pivots,
                           int pivots_cap, int* basis, double* x, double* z, double* tableau, double* history,
                           int history_cap) {
    if (history && history_cap > 0) {
        set_error("per-iteration history is not available on the streaming kernel; use LPX_KERNEL_CTA_GLOBAL");
        return LPX_E_CAPACITY;
    }
    lpx_session* s = lpx_dual_session_open(m, n, sense, A, rel, b, c, opt);
    if (!s) return LPX_E_CUDA;
    int st = LPX_RUNNING, np = 0, rc = LPX_OK;
    while (st == LPX_RUNNING && rc == LPX_OK) rc = lpx_session_step(s, 512, &st, &np);
    if (rc == LPX_OK) {
        if (status) *status = st;
        if (n_pivots) *n_pivots = np;
        if (silent_pivots) *silent_pivots = s->silent;
        if (pivots && pivots_cap > 0) rc = lpx_session_read_pivots(s, pivots, pivots_cap);
        const bool solved = st >= 0 || st == LPX_S_ITER_LIMIT;
        if (rc == LPX_OK && solved && (basis || x || z)) rc = lpx_session_read_solution(s, basis, x, z);
        if (rc == LPX_OK && solved && tableau) rc = lpx_session_read_tableau(s, tableau);
    }
    lpx_session_close(s);
    return rc;
}

}  // namespace lpx

#include "lpx_revised_stream.cuh"

extern "C" {

static bool dual_open_args_ok(const char* who, int m, int n, int sense, const double* A, const int* rel,
                              const double* b, const double* c) {
    bool ok = m >= 1 && n >= 1 && A && b && c && (sense == 0 || sense == 1);
    for (int i = 0; ok && rel && i < m; i++) ok = rel[i] >= 0 && rel[i] <= 2;
    if (!ok) set_error(std::string(who) + ": bad arguments (need m >= 1, n >= 1, sense 0 / 1, non-null A, b, c, rel[i] "
                                          "in 0..2)");
    return ok;
}

lpx_session* lpx_dual_session_open_dev(int m, int n, int sense, const double* A, const int* rel, const double* b,
                                       const double* c, const lpx_options* opt) {
    if (!dual_open_args_ok("lpx_dual_session_open_dev", m, n, sense, A, rel, b, c)) return nullptr;
    if (ensure_device() != LPX_OK) return nullptr;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    // the row signs need b on the host
    std::vector<double> hb(m);
    cudaStream_t st = rt().stream;
    if (cudaMemcpyAsync(hb.data(), b, (size_t)m * 8, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess) {
        cuda_fail(cudaGetLastError(), "lpx_dual_session_open_dev: reading b", __FILE__, __LINE__);
        return nullptr;
    }
    return session_create(m, n, sense, A, rel, b, c, opt, true, hb.data());
}

lpx_session* lpx_dual_session_open(int m, int n, int sense, const double* A, const int* rel, const double* b,
                                   const double* c, const lpx_options* opt) {
    if (!dual_open_args_ok("lpx_dual_session_open", m, n, sense, A, rel, b, c)) return nullptr;
    if (ensure_device() != LPX_OK) return nullptr;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    double *dA = nullptr, *db = nullptr, *dc = nullptr;
    lpx_session* s = nullptr;
    if (cudaMalloc(&dA, (size_t)m * n * 8) == cudaSuccess && cudaMalloc(&db, (size_t)m * 8) == cudaSuccess &&
        cudaMalloc(&dc, (size_t)n * 8) == cudaSuccess &&
        cudaMemcpy(dA, A, (size_t)m * n * 8, cudaMemcpyHostToDevice) == cudaSuccess &&
        cudaMemcpy(db, b, (size_t)m * 8, cudaMemcpyHostToDevice) == cudaSuccess &&
        cudaMemcpy(dc, c, (size_t)n * 8, cudaMemcpyHostToDevice) == cudaSuccess) {
        s = session_create(m, n, sense, dA, rel, db, dc, opt, true, b);
    } else {
        cuda_fail(cudaGetLastError(), "lpx_dual_session_open: staging inputs", __FILE__, __LINE__);
    }
    cudaFree(dA);
    cudaFree(db);
    cudaFree(dc);
    return s;
}

lpx_session* lpx_two_phase_session_open_dev(int m, int n, int sense, const double* A, const int* rel, const double* b,
                                            const double* c, const lpx_options* opt) {
    if (!dual_open_args_ok("lpx_two_phase_session_open_dev", m, n, sense, A, rel, b, c)) return nullptr;
    if (ensure_device() != LPX_OK) return nullptr;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    // the normalisation and the column numbering need b on the host
    std::vector<double> hb(m);
    cudaStream_t st = rt().stream;
    if (cudaMemcpyAsync(hb.data(), b, (size_t)m * 8, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess) {
        cuda_fail(cudaGetLastError(), "lpx_two_phase_session_open_dev: reading b", __FILE__, __LINE__);
        return nullptr;
    }
    return session_two_phase(m, n, sense, A, rel, b, c, hb.data(), opt);
}

lpx_session* lpx_two_phase_session_open(int m, int n, int sense, const double* A, const int* rel, const double* b,
                                        const double* c, const lpx_options* opt) {
    if (!dual_open_args_ok("lpx_two_phase_session_open", m, n, sense, A, rel, b, c)) return nullptr;
    if (ensure_device() != LPX_OK) return nullptr;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    double *dA = nullptr, *db = nullptr, *dc = nullptr;
    lpx_session* s = nullptr;
    cudaStream_t st = rt().stream;
    if (cudaMalloc(&dA, (size_t)m * n * 8) == cudaSuccess && cudaMalloc(&db, (size_t)m * 8) == cudaSuccess &&
        cudaMalloc(&dc, (size_t)n * 8) == cudaSuccess &&
        cudaMemcpyAsync(dA, A, (size_t)m * n * 8, cudaMemcpyHostToDevice, st) == cudaSuccess &&
        cudaMemcpyAsync(db, b, (size_t)m * 8, cudaMemcpyHostToDevice, st) == cudaSuccess &&
        cudaMemcpyAsync(dc, c, (size_t)n * 8, cudaMemcpyHostToDevice, st) == cudaSuccess &&
        cudaStreamSynchronize(st) == cudaSuccess) {
        s = session_two_phase(m, n, sense, dA, rel, db, dc, b, opt);
    } else {
        cuda_fail(cudaGetLastError(), "lpx_two_phase_session_open: staging inputs", __FILE__, __LINE__);
    }
    cudaFree(dA);
    cudaFree(db);
    cudaFree(dc);
    return s;
}

int lpx_session_two_phase_info(lpx_session* s, int* phase, int* phase1_pivots) {
    if (!s) {
        set_error("lpx_session_two_phase_info: null session");
        return LPX_E_BAD_ARGS;
    }
    TwoPhaseState h{};
    if (s->two_phase) {
        LPX_CUDA(cudaMemcpyAsync(&h, s->tla.st, sizeof h, cudaMemcpyDeviceToHost, s->stream));
        LPX_CUDA(cudaStreamSynchronize(s->stream));
    }
    if (phase) *phase = h.phase;
    if (phase1_pivots) *phase1_pivots = h.p1;
    return LPX_OK;
}

int lpx_session_silent_pivots(const lpx_session* s, int* silent) {
    if (!s || !silent) {
        set_error("lpx_session_silent_pivots: bad arguments");
        return LPX_E_BAD_ARGS;
    }
    *silent = s->silent;
    return LPX_OK;
}

lpx_session* lpx_session_open_dev(int m, int n, int sense, const double* A, const int* rel, const double* b,
                                  const double* c, const lpx_options* opt) {
    if (m < 1 || n < 1 || !A || !b || !c || (sense != 0 && sense != 1)) {
        set_error("lpx_session_open_dev: bad arguments");
        return nullptr;
    }
    return session_create(m, n, sense, A, rel, b, c, opt);
}

lpx_session* lpx_session_open(int m, int n, int sense, const double* A, const int* rel, const double* b,
                              const double* c, const lpx_options* opt) {
    if (m < 1 || n < 1 || !A || !b || !c || (sense != 0 && sense != 1)) {
        set_error("lpx_session_open: bad arguments");
        return nullptr;
    }
    if (ensure_device() != LPX_OK) return nullptr;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    double *dA = nullptr, *db = nullptr, *dc = nullptr;
    lpx_session* s = nullptr;
    if (cudaMalloc(&dA, (size_t)m * n * 8) == cudaSuccess && cudaMalloc(&db, (size_t)m * 8) == cudaSuccess &&
        cudaMalloc(&dc, (size_t)n * 8) == cudaSuccess &&
        cudaMemcpy(dA, A, (size_t)m * n * 8, cudaMemcpyHostToDevice) == cudaSuccess &&
        cudaMemcpy(db, b, (size_t)m * 8, cudaMemcpyHostToDevice) == cudaSuccess &&
        cudaMemcpy(dc, c, (size_t)n * 8, cudaMemcpyHostToDevice) == cudaSuccess) {
        s = session_create(m, n, sense, dA, rel, db, dc, opt);
    } else {
        cuda_fail(cudaGetLastError(), "lpx_session_open: staging inputs", __FILE__, __LINE__);
    }
    cudaFree(dA);
    cudaFree(db);
    cudaFree(dc);
    return s;
}

lpx_session* lpx_session_reoptimize(const lpx_session* base, int kind, const double* payload, const lpx_options* opt) {
    if (!base || !payload || kind < LPX_REOPT_RHS || kind > LPX_REOPT_COL) {
        set_error("lpx_session_reoptimize: bad arguments (NULL base or payload, or an unknown kind)");
        return nullptr;
    }
    if (base->two_phase) {
        set_error("lpx_session_reoptimize: the base is a two-phase session (its slack layout is not the one "
                  "re-optimization reads); re-optimization is defined for Primal Simplex results");
        return nullptr;
    }
    if (kind == LPX_REOPT_ROW && payload[base->n] != 0.0 && payload[base->n] != 1.0) {
        set_error("lpx_session_reoptimize: the added row's rel must be 0 (<=) or 1 (>=)");
        return nullptr;
    }
    if (ensure_device() != LPX_OK) return nullptr;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    return session_reoptimize(base, kind, payload, opt);
}

int lpx_session_parametric(const lpx_session* base, int kind, const double* payload, int seg_cap,
                           const lpx_options* opt, int* end, int* n_segments, int* n_pivots, double* segments,
                           int* seg_pivots, int* basis, double* tableau) {
    if (!base || !payload || !end || (kind != LPX_PARAM_RHS && kind != LPX_PARAM_COST) || seg_cap < 1) {
        set_error("lpx_session_parametric: bad arguments (NULL base, payload or end, an unknown kind, or seg_cap < 1)");
        return LPX_E_BAD_ARGS;
    }
    if (base->two_phase) {
        set_error("lpx_session_parametric: the base is a two-phase session (its slack layout is not the one parametric "
                  "analysis reads); parametric analysis is defined for Primal Simplex results");
        return LPX_E_BAD_ARGS;
    }
    if (!(payload[lpx_param_payload_stride(kind, base->m_in, base->n) - 1] >= 0.0)) {
        set_error("lpx_session_parametric: theta_max must be >= 0 or +inf (not NaN)");
        return LPX_E_BAD_ARGS;
    }
    if (base->dual_model) {
        set_error("lpx_session_parametric: the base is a Dual Simplex session (its tableau treats '>=' rows as '<='); "
                  "parametric analysis is defined for Primal Simplex results");
        return LPX_E_BAD_ARGS;
    }
    if (!base->sens_ok) {
        set_error("lpx_session_parametric: not defined for the query session of an added row or column");
        return LPX_E_BAD_ARGS;
    }
    int rc = ensure_device();
    if (rc != LPX_OK) return rc;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    return session_parametric(base, kind, payload, seg_cap, opt, end, n_segments, n_pivots, segments, seg_pivots, basis,
                              tableau);
}

int lpx_session_step_async(lpx_session* s, int max_pivots) {
    if (!s || max_pivots < 0) {
        set_error("lpx_session_step_async: bad arguments");
        return LPX_E_BAD_ARGS;
    }
    if (s->pipe) {
        // No fence against the main stream here: the look-ahead only depends on the session's own
        // kernels (event chain below), so the first look-ahead of this call overlaps the last pass
        // of the previous call and the pipeline never drains between calls.
        return launch_pipe_blocks(s, max_pivots, false);
    }
    if (s->P.kblock > 0) {
        for (int left = max_pivots; left > 0; left -= s->P.kblock) {
            int rc = launch_block(s, std::min(left, s->P.kblock));
            if (rc != LPX_OK) return rc;
        }
        return LPX_OK;
    }
    for (int k = 0; k < max_pivots; k++) {
        int rc = launch_pair(s, 0);
        if (rc != LPX_OK) return rc;
    }
    return LPX_OK;
}

// Development aid: n pivots with CUDA events around each of the two kernels.  us[0] = mean
// prep/select time, us[1] = mean update time, us[2] = mean time per pivot including the gaps.
int lpx_session_profile(lpx_session* s, int n, double* us) {
    if (!s || n < 1 || !us) return LPX_E_BAD_ARGS;
    std::vector<cudaEvent_t> ev((size_t)3 * n);
    for (auto& e : ev) LPX_CUDA(cudaEventCreate(&e));
    for (int k = 0; k < n; k++) {
        LPX_CUDA(cudaEventRecord(ev[3 * k], s->stream));
        if (s->pipe) {
            const int par = (int)(s->blocks & 1);
            LPX_CUDA(cudaStreamWaitEvent(s->stream, s->evL[par ^ 1], 0));
            stream_lookahead_pipe_kernel<<<LPX_LA_CLUSTER, LPX_LA_THREADS, lookahead_cluster_smem(s->P), s->stream>>>(
                s->P, s->P.kblock, par, 1);
            LPX_CUDA(cudaEventRecord(s->evL[par], s->stream));
            LPX_CUDA(cudaEventRecord(ev[3 * k + 1], s->stream));
            stream_update_pipe_tma_kernel<LPX_PIPE_K><<<s->grid_pipe, 256, pipe_pass_smem(), s->stream>>>(s->P, s->rpc_pipe, par);
            LPX_CUDA(cudaEventRecord(s->evP[par], s->stream));
            LPX_CUDA(cudaEventRecord(ev[3 * k + 2], s->stream));
            s->blocks++;
            continue;
        }
        if (s->P.kblock > 0) {
            launch_lookahead(s, s->P.kblock);
            LPX_CUDA(cudaEventRecord(ev[3 * k + 1], s->stream));
            launch_block_pass(s);
            LPX_CUDA(cudaEventRecord(ev[3 * k + 2], s->stream));
            continue;
        }
        launch_select(s, 0);
        LPX_CUDA(cudaEventRecord(ev[3 * k + 1], s->stream));
        stream_update_kernel<4><<<s->grid_update, 256, 0, s->stream>>>(s->P);
        LPX_CUDA(cudaEventRecord(ev[3 * k + 2], s->stream));
    }
    LPX_CUDA(cudaStreamSynchronize(s->stream));
    double a = 0, b = 0;
    float ms = 0;
    for (int k = 0; k < n; k++) {
        cudaEventElapsedTime(&ms, ev[3 * k], ev[3 * k + 1]);
        a += ms;
        cudaEventElapsedTime(&ms, ev[3 * k + 1], ev[3 * k + 2]);
        b += ms;
    }
    cudaEventElapsedTime(&ms, ev[0], ev[3 * (n - 1) + 2]);
    us[0] = a * 1e3 / n;
    us[1] = b * 1e3 / n;
    us[2] = ms * 1e3 / n;
    for (auto& e : ev) cudaEventDestroy(e);
    return LPX_OK;
}

// Development aid: phase timestamps (ns) of the first step of the last look-ahead launch.
int lpx_session_debug_stamps(lpx_session* s, unsigned long long* out8) {
    if (!s || !out8 || !s->P.dbg) return LPX_E_BAD_ARGS;
    LPX_CUDA(cudaStreamSynchronize(s->stream));
    LPX_CUDA(cudaMemcpy(out8, s->P.dbg, 8 * 8, cudaMemcpyDeviceToHost));
    return LPX_OK;
}

int lpx_session_sync(lpx_session* s, int* status, int* pivots_total) {
    if (!s) {
        set_error("lpx_session_sync: null session");
        return LPX_E_BAD_ARGS;
    }
    // probe: resolves OPTIMAL / UNBOUNDED / ITER_LIMIT for the tableau as it stands, no pivot
    int rc = s->pipe ? launch_pipe_probe(s) : (s->P.kblock > 0 ? launch_block(s, 0) : launch_pair(s, 1));
    if (rc != LPX_OK) return rc;
    StreamCtl h;
    LPX_CUDA(cudaMemcpyAsync(&h, s->P.ctl, sizeof h, cudaMemcpyDeviceToHost, s->stream));
    LPX_CUDA(cudaStreamSynchronize(s->stream));
    if (status) *status = h.status;
    if (pivots_total) *pivots_total = h.pivots;
    return LPX_OK;
}

int lpx_session_step(lpx_session* s, int max_pivots, int* status, int* pivots_total) {
    int rc = lpx_session_step_async(s, max_pivots);
    if (rc != LPX_OK) return rc;
    return lpx_session_sync(s, status, pivots_total);
}

void* lpx_session_stream(lpx_session* s) { return s ? (void*)s->stream : nullptr; }

int lpx_session_dims(const lpx_session* s, int* rows, int* cols) {
    if (!s) return LPX_E_BAD_ARGS;
    if (rows) *rows = s->two_phase ? s->P.m + 1 : s->P.rows;  // two-phase: lpx_two_phase_dims
    if (cols) *cols = s->two_phase ? s->tp_ns + 1 : s->P.width;
    return LPX_OK;
}

int lpx_session_read_tableau(lpx_session* s, double* tableau) {
    if (!s || !tableau) return LPX_E_BAD_ARGS;
    const double* Tcur = s->P.T;
    if (s->pipe) {
        StreamCtl h;
        LPX_CUDA(cudaMemcpyAsync(&h, s->P.ctl, sizeof h, cudaMemcpyDeviceToHost, s->stream));
        LPX_CUDA(cudaStreamSynchronize(s->stream));
        if (pipe_current_buffer(s, h)) Tcur = s->P.T1;
    }
    if (s->two_phase) {
        // rows 0..m: the columns 0..n+s-1, then the RHS (column W - 1), compact
        const size_t oc = (size_t)s->tp_ns + 1, pitch = (size_t)s->P.ld * 8;
        LPX_CUDA(cudaMemcpy2DAsync(tableau, oc * 8, Tcur, pitch, (size_t)s->tp_ns * 8, s->P.m + 1,
                                   cudaMemcpyDeviceToHost, s->stream));
        LPX_CUDA(cudaMemcpy2DAsync(tableau + s->tp_ns, oc * 8, Tcur + s->P.width - 1, pitch, 8, s->P.m + 1,
                                   cudaMemcpyDeviceToHost, s->stream));
        LPX_CUDA(cudaStreamSynchronize(s->stream));
        return LPX_OK;
    }
    LPX_CUDA(cudaMemcpy2DAsync(tableau, (size_t)s->P.width * 8, Tcur, (size_t)s->P.ld * 8, (size_t)s->P.width * 8,
                               s->P.rows, cudaMemcpyDeviceToHost, s->stream));
    LPX_CUDA(cudaStreamSynchronize(s->stream));
    return LPX_OK;
}

int lpx_session_sensitivity(lpx_session* s, double* report) {
    if (!s || !report) {
        set_error("lpx_session_sensitivity: bad arguments");
        return LPX_E_BAD_ARGS;
    }
    if (s->two_phase) {
        set_error("lpx_session_sensitivity: not defined for a two-phase session (its slack layout is not the one the "
                  "report reads); the report is defined for Primal Simplex results");
        return LPX_E_BAD_ARGS;
    }
    if (s->dual_model) {
        set_error("lpx_session_sensitivity: not defined for a Dual Simplex session (its tableau treats '>=' rows as "
                  "'<='); the report is defined for Primal Simplex results");
        return LPX_E_BAD_ARGS;
    }
    if (!s->sens_ok) {
        set_error("lpx_session_sensitivity: not defined for the query session of an added row or column");
        return LPX_E_BAD_ARGS;
    }
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    const StreamParams& P = s->P;
    const size_t stride = lpx_sensitivity_stride(s->m_in, s->n);
    StreamCtl h;
    LPX_CUDA(cudaMemcpyAsync(&h, P.ctl, sizeof h, cudaMemcpyDeviceToHost, s->stream));
    LPX_CUDA(cudaStreamSynchronize(s->stream));
    if (h.status != LPX_OPTIMAL) {
        for (size_t e = 0; e < stride; e++) report[e] = std::numeric_limits<double>::quiet_NaN();
        return LPX_OK;
    }
    if (!s->sens_report) {
        s->sens_rowof = (int*)sess_alloc(s, (size_t)P.width * 4);
        s->sens_partial = sess_alloc(s, sens_session_partial_bytes(s->m_in, P.m));
        s->sens_report = (double*)sess_alloc(s, stride * 8);
        if (!s->sens_rowof || !s->sens_partial || !s->sens_report) {
            s->sens_report = nullptr;
            return LPX_E_CUDA;
        }
    }
    // the live tableau, as lpx_session_read_tableau finds it: z-row and RHS are kept in place in it
    const double* Tcur = (s->pipe && pipe_current_buffer(s, h)) ? P.T1 : P.T;
    int rc = sens_session_launch(s->m_in, s->n, P.m, (size_t)P.ld, s->sense, s->sens_rmap, s->sens_b, s->sens_c, P.basis,
                                 Tcur, s->sens_rowof, s->sens_partial, s->sens_report, s->stream);
    if (rc != LPX_OK) return rc;
    LPX_CUDA(cudaMemcpyAsync(report, s->sens_report, stride * 8, cudaMemcpyDeviceToHost, s->stream));
    LPX_CUDA(cudaStreamSynchronize(s->stream));
    return LPX_OK;
}

int lpx_session_two_phase_sensitivity(lpx_session* s, double* report) {
    if (!s || !report) {
        set_error("lpx_session_two_phase_sensitivity: bad arguments");
        return LPX_E_BAD_ARGS;
    }
    if (!s->two_phase) {
        set_error("lpx_session_two_phase_sensitivity: not a two-phase session (lpx_session_sensitivity reports on "
                  "Primal Simplex sessions)");
        return LPX_E_BAD_ARGS;
    }
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    const StreamParams& P = s->P;
    const size_t stride = lpx_sensitivity_stride(s->m_in, s->n);
    StreamCtl h;
    LPX_CUDA(cudaMemcpyAsync(&h, P.ctl, sizeof h, cudaMemcpyDeviceToHost, s->stream));
    LPX_CUDA(cudaStreamSynchronize(s->stream));
    if (h.status != LPX_OPTIMAL) {
        for (size_t e = 0; e < stride; e++) report[e] = std::numeric_limits<double>::quiet_NaN();
        return LPX_OK;
    }
    if (!s->sens_report) {
        s->sens_rowof = (int*)sess_alloc(s, (size_t)P.width * 4);
        s->sens_partial = sess_alloc(s, sens_session_partial_bytes(P.m, P.m));
        s->sens_report = (double*)sess_alloc(s, stride * 8);
        if (!s->sens_rowof || !s->sens_partial || !s->sens_report) {
            s->sens_report = nullptr;
            return LPX_E_CUDA;
        }
    }
    // a two-phase session runs the blocked protocol on one tableau; it is only read here
    int rc = tp_sens_session_launch(P.m, s->n, s->tp_ns, P.width, (size_t)P.ld, s->sense, s->tp_info, s->sens_b,
                                    s->sens_c, P.basis, P.T, s->sens_rowof, s->sens_partial, s->sens_report, s->stream);
    if (rc != LPX_OK) return rc;
    LPX_CUDA(cudaMemcpyAsync(report, s->sens_report, stride * 8, cudaMemcpyDeviceToHost, s->stream));
    LPX_CUDA(cudaStreamSynchronize(s->stream));
    return LPX_OK;
}

int lpx_session_read_solution(lpx_session* s, int* basis, double* x, double* z) {
    if (!s) return LPX_E_BAD_ARGS;
    const int m = s->P.m, n = s->P.n;
    std::vector<int> hb(m);
    std::vector<double> hr(s->P.rows);
    LPX_CUDA(cudaMemcpyAsync(hb.data(), s->P.basis, (size_t)m * 4, cudaMemcpyDeviceToHost, s->stream));
    LPX_CUDA(cudaMemcpyAsync(hr.data(), s->P.rhsbuf, (size_t)s->P.rows * 8, cudaMemcpyDeviceToHost, s->stream));
    LPX_CUDA(cudaStreamSynchronize(s->stream));
    if (basis) std::memcpy(basis, hb.data(), (size_t)m * 4);
    if (x) {
        for (int j = 0; j < n; j++) x[j] = 0.0;
        for (int i = 0; i < m; i++)
            if (hb[i] < n) x[hb[i]] = hr[i];
    }
    if (z) *z = hr[m];
    return LPX_OK;
}

int lpx_session_read_pivots(lpx_session* s, int* pivots, int pivots_cap) {
    if (!s || !pivots || pivots_cap < 0) return LPX_E_BAD_ARGS;
    StreamCtl h;
    LPX_CUDA(cudaMemcpyAsync(&h, s->P.ctl, sizeof h, cudaMemcpyDeviceToHost, s->stream));
    LPX_CUDA(cudaStreamSynchronize(s->stream));
    const int k = std::min(std::min(h.pivots, pivots_cap), s->P.pivlog_cap);
    if (k > 0) LPX_CUDA(cudaMemcpy(pivots, s->P.pivlog, (size_t)k * 8, cudaMemcpyDeviceToHost));
    return LPX_OK;
}

void lpx_session_close(lpx_session* s) { sess_free(s); }

}  // extern "C"
