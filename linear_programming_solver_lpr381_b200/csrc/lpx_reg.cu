// lpx_reg.cu — register-resident batched Primal Simplex (BASELINE config 2: 64 x 128).
//
// One CTA per tableau, the tableau lives in REGISTERS for the whole solve.  13 row warps: warp w
// owns constraint rows w*5 .. w*5+4, lane l the columns l, l+32, .. of those rows (30 doubles per
// thread).  One control warp owns what every decision needs — the objective row, the RHS column
// and the objective value — and makes the two decisions alone, so that the row warps neither
// repeat them nor compete with them for issue slots.  Per pivot only three small vectors cross
// shared memory: the entering column (= update factors), the raw leaving row and its quotients.
//
// A pivot is five short phases between block barriers (measured with ncu's PC sampling, cycles at
// one CTA per SM): row warps publish the entering column (~460) | control warp: ratios, two rows
// per lane, and the leaving row (~700) | the owner warp publishes the leaving row (~300) | 192
// threads divide it, one division each (~300) | rank-1 update, R*C unfused DMUL + DSUB per thread,
// while the control warp updates the objective row / RHS and picks the NEXT entering column (~840).
// The chain is latency, not throughput: FP64 pipe < 20 % busy, so two CTAs per SM are kept
// resident (CS = 2 of the 6 column slots move to shared memory to fit 72 registers, no spills)
// and one CTA's narrow phases hide behind the other's update.
//
// Same rules, same order, same rounding as the reference (R/Models/PrimalSimplex.cs:205-257):
// entering = most negative objective entry below -1e-9, lowest index on ties, as two REDUX minima
// over an order-preserving key plus one over the index; leaving = the sequential margin scan,
// answered by one REDUX min + one ballot when no other ratio lies within the margin of the minimum
// (warp_margin_scan64) and replayed exactly otherwise; pivot = true division then separate multiply
// and subtract, zero-factor rows included.
#include <cstdio>
#include <cstdlib>

#include "lpx_cta.cuh"
#include "lpx_stream.hpp"

namespace lpx {

struct RegBatch {
    const double* A;
    const double* b;
    const double* c;
    int m, n, sense, max_iter;
    int* status;
    int* n_pivots;
    int* basis;
    double* x;
    double* z;
    double* tableau;
    unsigned long long* total_pivots;
    long long* dbg;  // LPX_REG_STAMPS=1: per-phase clock64() sums of block 0 (8 slots)
};

// NW row warps + 1 control warp.  Row warp w owns constraint rows w*R .. w*R+R-1, lane l the columns
// l, l+32, .. of those rows.  The control warp (warp NW) owns what every decision needs: the
// objective row (C entries per lane), the RHS column (rows lane and lane+32) and the objective value.
// Column slots 0..CR-1 of every thread are registers, slots CR..CR+CS-1 live in shared memory
// (lane-interleaved, conflict-free): CS = 0 is the all-register build (one CTA per SM), CS = 2 leaves
// room for two CTAs per SM without spilling, so one CTA's narrow phases hide behind the other's update.
//
// COND = the CONDENSED tableau (see lpx_cta_cond.cuh for the argument): only the n non-basic columns are held
// and updated — the m basic columns are exact unit vectors (+0 / 1: every primal pivot element is positive)
// that no decision reads.  A pivot on (row l, slot e) hands slot e to the leaving variable, whose unit
// column goes through the same update as every other column (0 - f * (1 / piv), row l <- 1 / piv); ties of
// ChooseEntering go to the lowest VARIABLE index (s_nbvar).  A 64 x 128 problem then needs four column slots
// instead of six, which is what lets three CTAs share an SM; the full tableau the caller gets is put back
// together on the way out (non-basic columns scattered to their variables' places through a row buffer in
// shared memory, basic columns written as unit vectors), bit for bit what the full-width kernel holds.
template <int NW, int R, int CR, int CS, int OCC, bool DBG = false, bool COND = false>
__global__ void __launch_bounds__((NW + 1) * 32, OCC) reg_simplex_kernel(const RegBatch B) {
    constexpr int C = CR + CS;
    constexpr int ROWS = NW * R;   // padded constraint rows (>= m)
    constexpr int COLS = 32 * C;   // padded non-RHS columns (>= n + m; COND: >= n)
    constexpr int RBW = COND ? 32 * C + ((ROWS + 31) & ~31) + 32 : 0;  // COND: one full-width row per warp
    static_assert(!COND || COLS <= 256, "slot index packed into 8 bits");
    extern __shared__ __align__(16) double s_t[];  // (CS ? CS : 1) * (ROWS + 1) * 32: [slot][row][lane]; row ROWS = objective row
                                                   // COND: followed by (NW + 1) * RBW doubles of row buffers
    __shared__ int s_nbvar[COND ? COLS : 1];       // COND: the variable held by each column slot
    constexpr int NT = (NW + 1) * 32;
    static_assert(ROWS >= 64 && ROWS <= 96, "the control warp holds the RHS of rows lane and lane+32");
    __shared__ __align__(16) double s_f[ROWS];  // entering column = update factors
    __shared__ double s_rhs[ROWS + 1];
    __shared__ double s_p[COLS];     // normalised pivot row
    __shared__ double s_raw[COLS];   // the leaving row before normalisation
    __shared__ int s_basis[ROWS];
    __shared__ int s_ctl[4];

    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const bool ctl = w == NW;
    const int p = blockIdx.x;
    const int m = B.m, n = B.n, width = n + m + 1;
    const double* Ap = B.A + (size_t)p * m * n;
    const double* bp = B.b + (size_t)p * m;
    const double* cp = B.c + (size_t)p * n;

    // ---- BuildTableau straight into registers (PrimalSimplex.cs:179-203) ---------------------
    double t[R][CR];       // control warp: t[0][*] is the objective row
    const int row0 = ctl ? ROWS : w * R;  // first padded row of this warp in s_t
    // element (r, c) of this thread: a register for c < CR, shared memory otherwise
#define T_GET(r, c) ((c) < CR ? t[r][(c) < CR ? (c) : 0] : s_t[(((c) - CR) * (ROWS + 1) + row0 + (r)) * 32 + lane])
#define T_SET(r, c, v)                                                   \
    do {                                                                 \
        if ((c) < CR) t[r][(c) < CR ? (c) : 0] = (v);                    \
        else s_t[(((c) - CR) * (ROWS + 1) + row0 + (r)) * 32 + lane] = (v); \
    } while (0)
    // control-warp state lives in the row slots it does not use (t[1..][*]), so that it costs the
    // row warps no registers: RHS of rows lane / lane+32, objective value, and per-pivot scratch
    static_assert((R - 1) * CR >= 7, "control-warp aliases need seven slots in t[1..][*]");
#define CTL_ALIAS(k) t[1 + (k) / CR][(k) % CR]
    double &rhs0 = CTL_ALIAS(0), &rhs1 = CTL_ALIAS(1), &zrhs = CTL_ALIAS(2), &a0 = CTL_ALIAS(3), &a1 = CTL_ALIAS(4),
           &fz = CTL_ALIAS(5), &prhs = CTL_ALIAS(6);
#undef CTL_ALIAS
#pragma unroll
    for (int r = 0; r < R; r++) {
        const int i = w * R + r;
#pragma unroll
        for (int c = 0; c < C; c++) {
            const int j = lane + 32 * c;
            double v = 0.0;
            if (!ctl) {
                if (i < m) {
                    if (j < n) v = Ap[(size_t)i * n + j];
                    else if (!COND && j == n + i) v = 1.0;
                }
            } else if (r == 0 && j < n) {
                double cj = cp[j];
                if (B.sense == 1) cj = dneg(cj);
                v = dneg(cj);
            }
            if (!ctl || r == 0) T_SET(r, c, v);
            else if (c < CR) t[r][c < CR ? c : 0] = 0.0;
        }
    }
    if (ctl) {
        if (lane < m) rhs0 = bp[lane];
        if (lane + 32 < m) rhs1 = bp[lane + 32];
    }
    // the reference's up-front check (PrimalSimplex.cs:73-76); '>=' rows cannot occur here
    if (tid == 0) {
        s_ctl[1] = LPX_RUNNING;
        s_ctl[3] = 0;  // pivots done: kept here by lane 0 of the control warp, not in a register of every thread
    }
    for (int i = tid; i < m; i += NT) s_basis[i] = n + i;
    if (COND)
        for (int j = tid; j < COLS; j += NT) s_nbvar[j] = j;
    __syncthreads();
    if (ctl && (rhs0 < -1e-9 || rhs1 < -1e-9)) s_ctl[1] = LPX_S_NEG_RHS;
    __syncthreads();
    int status = s_ctl[1];
    int n_piv = 0;

    if (status == LPX_RUNNING) {
        // ChooseEntering on the objective row (control warp): most negative entry below -1e-9,
        // lowest column on ties, NaN never wins.  Two REDUX minima on the value key, one on the
        // column index.
        // The keys are computed twice rather than kept in an array: the control warp shares the register budget
        // with the row warps' tableau.
        auto choose_entering = [&]() {
            auto key = [&](int c) {
                const double zv = T_GET(0, c);
                return zv < -LPX_EPS ? dkey(zv) : ~0ULL;
            };
            unsigned long long kl = ~0ULL;
#pragma unroll
            for (int c = 0; c < C; c++) {
                const unsigned long long kc = key(c);
                kl = kc < kl ? kc : kl;
            }
            const unsigned long long K = warp_min_u64(kl);
            int ln;  // the lane index read afresh: held across the pivot loop it costs a register the row warps need
            asm volatile("mov.u32 %0, %%laneid;" : "=r"(ln));
            int jl = INT_MAX;
#pragma unroll
            for (int c = C - 1; c >= 0; c--)
                if (key(c) == K) {
                    if (COND) jl = min(jl, (s_nbvar[ln + 32 * c] << 8) | (ln + 32 * c));  // lowest VARIABLE wins
                    else jl = ln + 32 * c;
                }
            int j = __reduce_min_sync(0xffffffffu, jl);
            if (COND) j &= 255;
            // one word tells every warp how the next pass starts: the column, -1 = optimal, -2 = the
            // reference's iteration limit, which it tests BEFORE looking for an entering column
            if (lane == 0) s_ctl[0] = s_ctl[3] + 1 > B.max_iter ? -2 : (K == ~0ULL ? -1 : j);
        };
        if (ctl) choose_entering();

        // One pivot = five short phases separated by block barriers.  Latency, not throughput,
        // bounds it, so the narrow decisions (entering column, ratios, leaving row, RHS) run in the
        // control warp only — the row warps neither repeat them nor compete for issue slots — and
        // every division is done by a different thread.
        // DBG build: lane 0 of four warps records its ARRIVAL time at each barrier of pivots 4..7
        const int dslot = w == 0 ? 0 : w == 5 ? 1 : w == NW - 1 ? 2 : ctl ? 3 : -1;
        int dbg_piv = 0;
#define REG_STAMP(k)                                                                                  \
    if (DBG && B.dbg && p == 0 && lane == 0 && dslot >= 0 && dbg_piv >= 3 && dbg_piv < 7)             \
        B.dbg[((dbg_piv - 3) * 4 + dslot) * 8 + (k)] = clock64();
        while (true) {
            __syncthreads();  // (A) s_ctl[0] holds the entering column; all updates are done
            const int e = s_ctl[0];
            if (e < 0) {
                status = e == -2 ? LPX_S_ITER_LIMIT : LPX_OPTIMAL;
                break;
            }
            // ---- P2: the lanes that own the entering column publish it -----------------------------
            const int ce = e >> 5, le = e & 31;
            // A chain of warp-uniform branches: predicated-off stores still queue in the memory pipe
            // (30 slots per warp) and a jump table costs an indirect branch; the empty asm keeps the
            // compiler from if-converting the bodies.
            if (!ctl) {
#define REG_PUT(K)                                                                        \
    if (K < C && ce == K) {                                                               \
        asm volatile("" ::: "memory");                                                    \
        if (lane == le) {                                                                 \
            _Pragma("unroll") for (int r = 0; r < R; r++) s_f[w * R + r] = T_GET(r, K);   \
        }                                                                                 \
    }
                REG_PUT(0) else REG_PUT(1) else REG_PUT(2) else REG_PUT(3) else REG_PUT(4) else REG_PUT(5) else REG_PUT(6) else REG_PUT(7)
#undef REG_PUT
            } else {
                double v = 0.0;
#pragma unroll
                for (int c = 0; c < C; c++)
                    if (c == ce) v = T_GET(0, c);
                fz = __shfl_sync(0xffffffffu, v, le);
            }
            REG_STAMP(0)
            __syncthreads();  // (B)
            // ---- P3 (control warp): ratios, two rows per lane, and ChooseLeaving --------------------
            if (ctl) {
                a0 = s_f[lane];
                a1 = s_f[lane + 32];
                const double nan = __longlong_as_double(0x7ff8000000000000LL);  // = not eligible
                const double r0 = (lane < m && a0 > LPX_EPS) ? __ddiv_rn(rhs0, a0) : nan;
                const double r1 = (lane < m - 32 && a1 > LPX_EPS) ? __ddiv_rn(rhs1, a1) : nan;  // lane + 32 < m
                const int row = warp_margin_scan64(m, LPX_MARGIN_PRIMAL, r0, r1);
                if (lane == 0) s_ctl[2] = row;
            }
            REG_STAMP(1)
            __syncthreads();  // (C)
            const int lr = s_ctl[2];
            if (lr < 0) {
                status = LPX_UNBOUNDED;
                break;
            }
            const double piv = s_f[lr];
            // ---- P4: the owner of the leaving row publishes it; the control warp normalises its RHS ---
            const int wl = lr / R, rl = lr - wl * R;
            double f[R];  // this warp's update factors; the all-register build has room to fetch them
                          // while the pivot row is still being prepared
            if (CS == 0 && !ctl) {
#pragma unroll
                for (int r = 0; r < R; r++) f[r] = s_f[w * R + r];
            }
            if (w == wl) {
#pragma unroll
                for (int r = 0; r < R; r++) {
                    if (r == rl) {
#pragma unroll
                        for (int c = 0; c < C; c++) s_raw[lane + 32 * c] = T_GET(r, c);
                    }
                }
            }
            REG_STAMP(2)
            __syncthreads();  // (D)
            // ---- P5: one division per thread ------------------------------------------------------
            if (tid < COLS) {
                s_p[tid] = ddiv_by_pos((COND && tid == e) ? 1.0 : s_raw[tid], piv);  // COND: the leaving variable's unit column
            } else if (ctl) {
                const double rl_rhs = __shfl_sync(0xffffffffu, lr < 32 ? rhs0 : rhs1, lr & 31);
                prhs = ddiv_by_pos(rl_rhs, piv);
            }
            REG_STAMP(3)
            __syncthreads();  // (E)
            // ---- P1: rank-1 update in registers; the control warp updates the objective row and the
            // RHS column and picks the NEXT entering column meanwhile.  Only the warp that owns the
            // leaving row pays for the "this row becomes the pivot row" select.
            if (ctl) {
#pragma unroll
                for (int c = 0; c < C; c++) {
                    double cur = T_GET(0, c);
                    if (COND && c == ce && lane == le) cur = 0.0;
                    T_SET(0, c, __dsub_rn(cur, __dmul_rn(fz, s_p[lane + 32 * c])));
                }
                if (COND) {  // slot e now holds the leaving variable
                    if (lane == 0) {
                        const int ve = s_nbvar[e];
                        s_nbvar[e] = s_basis[lr];
                        s_basis[lr] = ve;
                    }
                    __syncwarp();
                }
                if (lane == 0) s_ctl[3]++;
                choose_entering();
                const double u0 = __dsub_rn(rhs0, __dmul_rn(a0, prhs)), u1 = __dsub_rn(rhs1, __dmul_rn(a1, prhs));
                rhs0 = lane == lr ? prhs : u0;
                rhs1 = lane == lr - 32 ? prhs : u1;
                zrhs = __dsub_rn(zrhs, __dmul_rn(fz, prhs));
                if (!COND && lane == 0) s_basis[lr] = e;
            } else {
                if (COND) {  // slot e enters the update as the leaving variable's unit column: zero outside row lr
#define REG_ZERO(K)                                                              \
    if (K < C && ce == K) {                                                      \
        asm volatile("" ::: "memory");                                           \
        if (lane == le) {                                                        \
            _Pragma("unroll") for (int r = 0; r < R; r++) T_SET(r, K, 0.0);      \
        }                                                                        \
    }
                    REG_ZERO(0) else REG_ZERO(1) else REG_ZERO(2) else REG_ZERO(3) else REG_ZERO(4) else REG_ZERO(5) else REG_ZERO(6) else REG_ZERO(7)
#undef REG_ZERO
                }
                // rows outside, slots inside: the C pivot-row entries stay in registers and each factor is
                // read where it is used (two rows per broadcast LDS.128), so that a 16-row warp never holds
                // all R factors at once; the shared-memory slot of a row is loaded and stored exactly once
                double pc[C];
#pragma unroll
                for (int c = 0; c < C; c++) pc[c] = s_p[lane + 32 * c];
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const double fr = CS == 0 ? f[r] : s_f[w * R + r];
#pragma unroll
                    for (int c = 0; c < C; c++) T_SET(r, c, __dsub_rn(T_GET(r, c), __dmul_rn(fr, pc[c])));
                }
                // the leaving row becomes the normalised pivot row; its index is read again rather than held
                // across barrier (E) in a register the update needs
                const int rlp = s_ctl[2] - w * R;
                if (rlp >= 0 && rlp < R) {
#pragma unroll
                    for (int r = 0; r < R; r++)
                        if (r == rlp) {
#pragma unroll
                            for (int c = 0; c < C; c++) T_SET(r, c, pc[c]);
                        }
                }
            }
            REG_STAMP(4)
            if (DBG) dbg_piv++;
        }
        __syncthreads();
#undef REG_STAMP
        n_piv = s_ctl[3];

        // ---- results ----------------------------------------------------------------------------
        if (ctl) {
            s_rhs[lane] = rhs0;
            s_rhs[lane + 32] = rhs1;
            if (lane == 0) s_rhs[ROWS] = zrhs;
        }
        if (B.tableau && COND) {
            // the full-width rows, put together in this warp's row buffer: zeros, the non-basic entries at their
            // variables' columns, the row's own basic variable = 1; then one coalesced copy
            double* To = B.tableau + (size_t)p * (m + 1) * width;
            double* rb = s_t + (size_t)(CS ? CS : 1) * (ROWS + 1) * 32 + (size_t)w * RBW;
            // zeroed once: every row of the warp scatters its non-basic entries to the same places (by the same
            // lane), so between rows only the unit of the row's basic variable has to be taken back out
            for (int k = lane; k < RBW; k += 32) rb[k] = 0.0;
            __syncwarp();
#pragma unroll
            for (int r = 0; r < R; r++) {
                const int i = ctl ? m : w * R + r;
                if (ctl ? r == 0 : i < m) {
#pragma unroll
                    for (int c = 0; c < C; c++) {
                        const int j = lane + 32 * c;
                        if (j < n) rb[s_nbvar[j]] = T_GET(r, c);
                    }
                    if (!ctl && lane == 0) rb[s_basis[i]] = 1.0;
                    __syncwarp();
                    for (int j = lane; j < width - 1; j += 32) To[(size_t)i * width + j] = rb[j];
                    __syncwarp();
                    if (!ctl && lane == 0) rb[s_basis[i]] = 0.0;
                }
            }
            if (ctl) {
                if (lane < m) To[(size_t)lane * width + width - 1] = rhs0;
                if (lane + 32 < m) To[(size_t)(lane + 32) * width + width - 1] = rhs1;
                if (lane == 0) To[(size_t)m * width + width - 1] = zrhs;
            }
        } else if (B.tableau) {
            double* To = B.tableau + (size_t)p * (m + 1) * width;
            if (!ctl) {
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const int i = w * R + r;
                    if (i < m) {
#pragma unroll
                        for (int c = 0; c < C; c++) {
                            const int j = lane + 32 * c;
                            if (j < width - 1) To[(size_t)i * width + j] = T_GET(r, c);
                        }
                    }
                }
            } else {
#pragma unroll
                for (int c = 0; c < C; c++) {
                    const int j = lane + 32 * c;
                    if (j < width - 1) To[(size_t)m * width + j] = T_GET(0, c);
                }
                if (lane < m) To[(size_t)lane * width + width - 1] = rhs0;
                if (lane + 32 < m) To[(size_t)(lane + 32) * width + width - 1] = rhs1;
                if (lane == 0) To[(size_t)m * width + width - 1] = zrhs;
            }
        }
        if (B.x) {
            double* xo = B.x + (size_t)p * n;
            for (int j = tid; j < n; j += NT) xo[j] = 0.0;
        }
        __syncthreads();
        if (B.basis)
            for (int i = tid; i < m; i += NT) B.basis[(size_t)p * m + i] = s_basis[i];
        if (B.x) {  // basic decision variables take their row's RHS (distinct rows, distinct targets)
            double* xo = B.x + (size_t)p * n;
            for (int i = tid; i < m; i += NT)
                if (s_basis[i] < n) xo[s_basis[i]] = s_rhs[i];
        }
        if (tid == 0 && B.z) B.z[p] = s_rhs[ROWS];
    } else {
        // rejected up front (negative RHS): no result; zero-fill so reused buffers carry no leftovers
        if (B.tableau) {
            double* To = B.tableau + (size_t)p * (m + 1) * width;
            for (int k = tid; k < (m + 1) * width; k += NT) To[k] = 0.0;
        }
        if (B.x)
            for (int j = tid; j < n; j += NT) B.x[(size_t)p * n + j] = 0.0;
        if (B.basis)
            for (int i = tid; i < m; i += NT) B.basis[(size_t)p * m + i] = 0;
        if (tid == 0 && B.z) B.z[p] = 0.0;
    }
#undef T_GET
#undef T_SET
    if (tid == 0) {
        B.status[p] = status;
        if (B.n_pivots) B.n_pivots[p] = n_piv;
        if (B.total_pivots && n_piv) atomicAdd(B.total_pivots, (unsigned long long)n_piv);
    }
}

// dynamic shared memory of an instance: the CS column slots kept out of the register file
static size_t reg_smem(int nw, int r, int cs) { return (size_t)(cs ? cs : 1) * (nw * r + 1) * 32 * 8; }

// Shapes served by the <13, 5, 6> instance: m + 1 <= 65 rows, n + m <= 192 columns, all '<='.
bool reg_kernel_supports(int m, int n, int m_expanded, bool has_rel) {
    if (has_rel || m_expanded != m) return false;
    return m + 1 <= 65 && n + m <= 192 && m >= 1 && n >= 1;
}

int reg_launch_batched(int count, int m, int n, int sense, const double* A, const double* b, const double* c,
                       const lpx_options& opt, int* status, int* n_pivots, int* basis, double* x, double* z,
                       double* tableau, unsigned long long* total_pivots, cudaStream_t stream) {
    if (!reg_kernel_supports(m, n, m, false)) {
        set_error("LPX_KERNEL_CTA_REG: no register-resident kernel is built for this shape (need m <= 64, n + m <= 192, "
                  "all '<=' rows)");
        return LPX_E_CAPACITY;
    }
    if (count <= 0) return LPX_OK;
    RegBatch B;
    B.A = A;
    B.b = b;
    B.c = c;
    B.m = m;
    B.n = n;
    B.sense = sense;
    B.max_iter = opt.max_iterations;
    B.status = status;
    B.n_pivots = n_pivots;
    B.basis = basis;
    B.x = x;
    B.z = z;
    B.tableau = tableau;
    B.total_pivots = total_pivots;
    // Builds: the condensed tableau at three CTAs per SM (reg_variant 4, the default for n <= 128, and 5); the full tableau
    // with all six column slots in registers, one CTA per SM (1), four in registers + two in shared memory, two CTAs
    // per SM (2: 1.04 ms per 4096-LP batch, against 1.34 for 1), or two + four at three CTAs per SM (3: 1.19 ms).
    B.dbg = nullptr;
    static const bool stamps = getenv("LPX_REG_STAMPS") != nullptr;  // measurement aid, prints to stderr
    if (stamps) {
        long long* d = nullptr;
        const int nslots = 4 * 4 * 8;
        LPX_CUDA(cudaMalloc(&d, nslots * sizeof(long long)));
        LPX_CUDA(cudaMemsetAsync(d, 0, nslots * sizeof(long long), stream));
        B.dbg = d;
        if (opt.reg_variant == 1) reg_simplex_kernel<13, 5, 6, 0, 1, true><<<count, 14 * 32, reg_smem(13, 5, 0), stream>>>(B);
        else reg_simplex_kernel<13, 5, 4, 2, 2, true><<<count, 14 * 32, reg_smem(13, 5, 2), stream>>>(B);
        long long h[nslots];
        LPX_CUDA(cudaMemcpyAsync(h, d, sizeof h, cudaMemcpyDeviceToHost, stream));
        LPX_CUDA(cudaStreamSynchronize(stream));
        cudaFree(d);
        // arrival times at barriers B, C, D, E, A(next), relative to the control warp's arrival at B
        static const char* wn[4] = {"warp0", "warp5", "warp12", "ctl"};
        for (int it = 0; it < 4; it++) {
            const long long t0 = h[(it * 4 + 3) * 8 + 0];
            for (int sl = 0; sl < 4; sl++) {
                fprintf(stderr, "[reg arrivals] pivot %d %-6s:", it + 4, wn[sl]);
                for (int k = 0; k < 5; k++) fprintf(stderr, " %c=%lld", "BCDEA"[k], h[(it * 4 + sl) * 8 + k] - t0);
                fprintf(stderr, "\n");
            }
        }
        count_launch();
        return LPX_OK;
    }
    // Default: the condensed build, three CTAs per SM (n <= 128 columns of A; wider problems keep the six-slot build).
    const int variant = opt.reg_variant ? opt.reg_variant : (n <= 128 ? 4 : 2);
    if ((variant == 4 || variant == 5) && n > 128) {
        set_error("LPX_KERNEL_CTA_REG, reg_variant 4 / 5: the condensed build holds n <= 128 non-basic columns");
        return LPX_E_CAPACITY;
    }
    if (variant == 5) {
        // 4 row warps x 16 rows, three of the four column slots in registers (128 registers, no spills) and one in
        // shared memory, + one row buffer per warp: half the update's shared-memory traffic of build 4, but at 15
        // warps per SM instead of 27 (0.780 ms per 4096-LP batch against 0.726 for build 4, DESIGN.md §9)
        constexpr size_t smem5 = (size_t)1 * (4 * 16 + 1) * 32 * 8 + (size_t)5 * (128 + 64 + 32) * 8;
        reg_simplex_kernel<4, 16, 3, 1, 3, false, true><<<count, 5 * 32, smem5, stream>>>(B);
    } else if (variant == 4) {
        // 8 row warps x 8 rows, four column slots (two in registers, two in shared memory) + one row buffer per warp;
        // 72 registers, no spills (11 warps x 6 rows at 56 registers: 0.806 ms against 0.782 per 4096-LP batch)
        constexpr size_t smem4 = (size_t)2 * (8 * 8 + 1) * 32 * 8 + (size_t)9 * (128 + 64 + 32) * 8;
        auto k4 = reg_simplex_kernel<8, 8, 2, 2, 3, false, true>;
        static const bool ok4 = cudaFuncSetAttribute(k4, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4) == cudaSuccess;
        if (!ok4) return cuda_fail(cudaGetLastError(), "cudaFuncSetAttribute(reg_simplex_kernel<8,8,2,2,3,cond>)", __FILE__, __LINE__);
        k4<<<count, 9 * 32, smem4, stream>>>(B);
    } else if (variant == 1) {
        reg_simplex_kernel<13, 5, 6, 0, 1><<<count, 14 * 32, reg_smem(13, 5, 0), stream>>>(B);
    } else if (variant == 3) {
        // three CTAs per SM: 11 row warps x 6 rows, two of the six column slots in registers (56 registers), four
        // in shared memory (67 KB per CTA)
        static const bool ok3 = cudaFuncSetAttribute(reg_simplex_kernel<11, 6, 2, 4, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                     (int)reg_smem(11, 6, 4)) == cudaSuccess;
        if (!ok3) return cuda_fail(cudaGetLastError(), "cudaFuncSetAttribute(reg_simplex_kernel<11,6,2,4,3>)", __FILE__, __LINE__);
        reg_simplex_kernel<11, 6, 2, 4, 3><<<count, 12 * 32, reg_smem(11, 6, 4), stream>>>(B);
    } else {
        reg_simplex_kernel<13, 5, 4, 2, 2><<<count, 14 * 32, reg_smem(13, 5, 2), stream>>>(B);
    }
    LPX_CUDA(cudaGetLastError());
    count_launch();
    return LPX_OK;
}

}  // namespace lpx
