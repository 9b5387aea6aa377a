// lpx_common.cuh — shared host/device helpers of liblpx (sm_100a only).
//
// Numerics contract (SURVEY.md F6/F7): every tableau operation is a separate IEEE binary64
// multiply, subtract or divide (__dmul_rn/__dsub_rn/__ddiv_rn are never contracted into FMA),
// evaluated in the order of the reference's C# loops:
//   ChooseEntering  R/Models/PrimalSimplex.cs:205-220
//   ChooseLeaving   R/Models/PrimalSimplex.cs:222-243   (sequential epsilon-margin scan)
//   Pivot           R/Models/PrimalSimplex.cs:245-257
#pragma once
#include <cuda_runtime.h>

#include <climits>
#include <cstdint>
#include <cstdio>
#include <string>

#include "../../include/lpx.h"

#define LPX_EPS 1e-9            // PrimalSimplex.Eps / DualSimplex.Eps
#define LPX_MARGIN_PRIMAL 1e-9  // PrimalSimplex.cs:235
#define LPX_MARGIN_DUAL 1e-12   // DualSimplex.cs:85,220
#define LPX_DUAL_MAX_ITER 10000  // DualSimplex.cs:39: a literal, independent of PrimalSimplex.MaxIterations
#define LPX_DUAL_SILENT_MAX 100  // DualSimplex.cs:195-228: ForceDualFeasibility's guard

namespace lpx {

// ---- host side error plumbing -------------------------------------------------------------------
void set_error(const std::string& msg);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);
void count_launch(int n = 1);

#define LPX_CUDA(expr)                                                        \
    do {                                                                      \
        cudaError_t _e = (expr);                                              \
        if (_e != cudaSuccess) return lpx::cuda_fail(_e, #expr, __FILE__, __LINE__); \
    } while (0)

int ensure_device();  // lazily initialises the library on the current device; LPX_OK or LPX_E_CUDA
int sm_count();
int max_smem_optin();

// ---- device helpers ---------------------------------------------------------------------------
struct ArgMin {
    double v;
    int i;
};

__device__ __forceinline__ ArgMin argmin_pick(ArgMin a, ArgMin b) {
    // smaller value wins; equal values -> lower index (what a left-to-right strict '<' scan keeps)
    return (b.v < a.v || (b.v == a.v && b.i < a.i)) ? b : a;
}

__device__ __forceinline__ ArgMin warp_argmin(ArgMin a) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        ArgMin o;
        o.v = __shfl_xor_sync(0xffffffffu, a.v, off);
        o.i = __shfl_xor_sync(0xffffffffu, a.i, off);
        a = argmin_pick(a, o);
    }
    return a;
}

// ---- 64-bit keys and REDUX-based warp minima ---------------------------------------------------
// Order-preserving key of a double: a < b (as doubles)  =>  dkey(a) < dkey(b).  -0.0 sorts just
// below +0.0 and NaN above +inf; callers that care about -0.0 == +0.0 re-check with a real compare.
__device__ __forceinline__ unsigned long long dkey(double x) {
    const long long b = __double_as_longlong(x);
    return (unsigned long long)(b ^ ((b >> 63) | (long long)0x8000000000000000ULL));
}
__device__ __forceinline__ double dkey_inv(unsigned long long k) {
    const long long b = (long long)k;
    return __longlong_as_double(b < 0 ? (b ^ (long long)0x8000000000000000ULL) : ~b);
}
// Warp minimum of a 64-bit key with two 32-bit REDUX instructions (no shuffle ladder).
__device__ __forceinline__ unsigned long long warp_min_u64(unsigned long long k) {
    const unsigned hi = (unsigned)(k >> 32), lo = (unsigned)k;
    const unsigned hmin = __reduce_min_sync(0xffffffffu, hi);
    const unsigned lmin = __reduce_min_sync(0xffffffffu, hi == hmin ? lo : 0xffffffffu);
    return ((unsigned long long)hmin << 32) | lmin;
}

// Block-wide "most negative entry below thresh, lowest index on ties" over load(0..n).
// Returns -1 when no entry is < thresh.  NaN entries never win (comparison is false).
// Per warp: REDUX minimum of the value keys, then of the indices that hold it; the per-warp partials
// meet in shared memory and EVERY warp reduces them itself, so one barrier publishes the answer
// (the second one only frees `red`, >= 33 ArgMin, for immediate reuse).
template <int THREADS, class Load>
__device__ __forceinline__ int block_argmin_core(int n, double thresh, ArgMin* red, Load load) {
    unsigned long long kl = ~0ULL;
    int il = INT_MAX;
    for (int j = threadIdx.x; j < n; j += THREADS) {
        const double z = load(j);
        if (z < thresh) {
            const unsigned long long k = dkey(z);
            if (k < kl) {
                kl = k;
                il = j;
            }
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
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
    const int idx = __reduce_min_sync(0xffffffffu, k2 == K2 ? i2 : INT_MAX);
    __syncthreads();
    return K2 == ~0ULL ? -1 : idx;
}
template <int THREADS>
__device__ __forceinline__ int block_argmin_below(const double* v, int n, double thresh, ArgMin* red) {
    return block_argmin_core<THREADS>(n, thresh, red, [&](int j) { return v[j]; });
}
// Same with a stride between consecutive entries (column scans of a row-major tableau).
template <int THREADS>
__device__ __forceinline__ int block_argmin_below_strided(const double* v, size_t stride, int n, double thresh,
                                                          ArgMin* red) {
    return block_argmin_core<THREADS>(n, thresh, red, [&](int j) { return v[(size_t)j * stride]; });
}

// The reference's ratio test is NOT an argmin (SURVEY.md F6):
//     if (ratio < bestRatio - margin) { bestRatio = ratio; bestRow = i; }     for i = 0, 1, 2, ...
// One warp reproduces the exact sequential outcome: 32 candidates per step; the first lane that
// beats the running best is accepted, lanes at or before it are retired (they were compared with
// the best of their own time), later lanes are re-tested against the new best.
// get(i, r) -> bool eligible, r = ratio.  Must be called by all 32 lanes of the warp.
template <class Get>
__device__ __forceinline__ int warp_margin_scan(int count, double margin, Get get) {
    const int lane = threadIdx.x & 31;
    double best = __longlong_as_double(0x7ff0000000000000LL);  // +inf
    int row = -1;
    for (int base = 0; base < count; base += 32) {
        const int i = base + lane;
        double r = 0.0;
        bool live = false;
        if (i < count) live = get(i, r);
        while (true) {
            const double thr = __dsub_rn(best, margin);
            const unsigned hit = __ballot_sync(0xffffffffu, live && (r < thr));
            if (hit == 0u) break;
            const int first = __ffs(hit) - 1;
            best = __shfl_sync(0xffffffffu, r, first);
            row = base + first;
            if (lane <= first) live = false;
        }
    }
    return row;
}

// num / den for a divisor that is a pivot element or an eligible ratio denominator (|den| > 1e-9,
// never NaN or zero).  Bit-identical to __ddiv_rn, but a ZERO numerator — tableau rows are full of
// them — no longer drags its whole warp through the division's slow path (a subroutine call that
// costs several times the inline sequence): zeros divide a stand-in and return the signed zero that
// IEEE division gives, sign(num) xor sign(den).
// Same for a divisor known to be positive (primal pivot elements and ratio denominators).
__device__ __forceinline__ double ddiv_by_pos(double num, double den) {
    double n = num != 0.0 ? num : 1.0;
    asm volatile("" : "+d"(n));
    const double q = __ddiv_rn(n, den);
    return num != 0.0 ? q : num;
}
__device__ __forceinline__ double ddiv_by_pivot(double num, double den) {
    double n = num != 0.0 ? num : 1.0;
    asm volatile("" : "+d"(n));  // opaque, or the compiler folds the stand-in away again
    const double q = __ddiv_rn(n, den);
    const double z = den < 0.0 ? __longlong_as_double(__double_as_longlong(num) ^ (long long)0x8000000000000000ULL) : num;
    return num != 0.0 ? q : z;
}

// Certified shortcut of the margin scan.  Let v be the minimum eligible ratio and i* its lowest row.
// If v is the ONLY eligible ratio with  !(v < r_j - margin)  (v itself always is one), then whatever
// record b precedes i*,  v < b - margin  (monotone in b), so i* is accepted, and nothing after it can
// be (r_k < v - margin <= v is impossible): the sequential answer is i*.  One REDUX minimum and a
// count decide that; ties, near-ties inside the margin and -0.0 / +0.0 pairs fail the certificate and
// take the exact replay.
//
// Up to 64 rows held two per lane (r0 = row lane, r1 = row lane + 32; NaN = not eligible).
__device__ __forceinline__ int warp_margin_scan64(int count, double margin, double r0, double r1) {
    const unsigned long long k0 = dkey(r0), k1 = dkey(r1);
    const double d0 = __dsub_rn(r0, margin), d1 = __dsub_rn(r1, margin);  // off the critical path
    const unsigned long long K = warp_min_u64(k1 < k0 ? k1 : k0);
    const double vmin = dkey_inv(K);
    if (vmin != vmin) return -1;  // no eligible row
    const unsigned b0 = __ballot_sync(0xffffffffu, k0 == K);
    const unsigned b1 = __ballot_sync(0xffffffffu, k1 == K);
    const unsigned c0 = __ballot_sync(0xffffffffu, (r0 == r0) && !(vmin < d0));
    const unsigned c1 = __ballot_sync(0xffffffffu, (r1 == r1) && !(vmin < d1));
    if (__popc(c0) + __popc(c1) == 1 && vmin < __longlong_as_double(0x7ff0000000000000LL))
        return b0 ? __ffs(b0) - 1 : 32 + __ffs(b1) - 1;
    return warp_margin_scan(count, margin, [&](int i, double& ratio) {
        ratio = i < 32 ? r0 : r1;
        return ratio == ratio;
    });
}

// Wider certificate for ties.  C = the eligible ratios r with !(vmin < r - margin) — the minimum, its exact
// ties, anything within the margin of it.  If every eligible ratio OUTSIDE C clears all of C by the margin,
//     max(C) < min over j not in C of (r_j - margin),
// the sequential answer is the FIRST row of C: whatever record b stands when that row c1 comes up (+inf, or a
// ratio outside C) has r_c1 < b - margin, so c1 is accepted; after it a row k would need
// r_k < r_c1 - margin <= vmin, which nothing satisfies.  B&B node LPs on integer data tie all the time (equal
// bound rows, zero right-hand sides); only a ratio strictly between "tied" and "clear" falls through to the
// replay.  Each lane passes the largest key of its C members (0 if none), the smallest key of r - margin over
// its other eligible rows (~0 if none) and its first row in C (INT_MAX if none); returns the row, or -1.
__device__ __forceinline__ int warp_tie_certificate(unsigned long long cmax_key, unsigned long long dmin_key, int first_in_c) {
    const unsigned long long CM = ~warp_min_u64(~cmax_key);
    const unsigned long long DM = warp_min_u64(dmin_key);
    const int first = __reduce_min_sync(0xffffffffu, first_in_c);
    if (DM == ~0ULL || dkey_inv(CM) < dkey_inv(DM)) return first;
    return -1;
}

// Any number of candidates, read through get(i, r) -> eligible (cheap, called up to three times per
// candidate).  Must be called by all 32 lanes of the warp.
template <class Get>
__device__ __forceinline__ int warp_margin_scan_cert(int count, double margin, Get get) {
    const int lane = threadIdx.x & 31;
    unsigned long long kl = ~0ULL;
    for (int i = lane; i < count; i += 32) {
        double r;
        if (get(i, r)) {
            const unsigned long long k = dkey(r);
            kl = k < kl ? k : kl;
        }
    }
    const unsigned long long K = warp_min_u64(kl);
    if (K == ~0ULL) return -1;
    const double vmin = dkey_inv(K);
    int il = INT_MAX, close = 0;
    for (int i = lane; i < count; i += 32) {
        double r;
        if (get(i, r)) {
            if (dkey(r) == K && i < il) il = i;
            if (!(vmin < __dsub_rn(r, margin))) close++;
        }
    }
    const int imin = __reduce_min_sync(0xffffffffu, il);
    const int nclose = __reduce_add_sync(0xffffffffu, close);
    if (nclose == 1 && vmin < __longlong_as_double(0x7ff0000000000000LL)) return imin;
    if (vmin < __longlong_as_double(0x7ff0000000000000LL)) {  // ties: the wider certificate
        unsigned long long cm = 0ULL, dm = ~0ULL;
        int ic = INT_MAX;
        for (int i = lane; i < count; i += 32) {
            double r;
            if (get(i, r)) {
                const double d = __dsub_rn(r, margin);
                if (!(vmin < d)) {
                    const unsigned long long k = dkey(r);
                    cm = k > cm ? k : cm;
                    if (i < ic) ic = i;
                } else {
                    const unsigned long long kd = dkey(d);
                    dm = kd < dm ? kd : dm;
                }
            }
        }
        const int first = warp_tie_certificate(cm, dm, ic);
        if (first >= 0) return first;
    }
    return warp_margin_scan(count, margin, get);
}

// The same certified scan over ratios staged in shared memory (NaN = not eligible), with the candidates
// of a lane (rows lane, lane + 32, ..) held in K registers: the loops of warp_margin_scan_cert become
// straight-line code with K independent chains instead of K dependent round trips to shared memory —
// on a lone control warp, where every dependent instruction costs its full latency, that is the
// difference between ~1500 and a few hundred cycles per pivot.  count <= 32 K.
template <int K>
__device__ __forceinline__ int warp_margin_scan_regs(int count, double margin, const double* ratio) {
    const int lane = threadIdx.x & 31;
    double r[K];
    unsigned long long k[K];
#pragma unroll
    for (int s = 0; s < K; s++) {
        const int i = lane + 32 * s;
        r[s] = i < count ? ratio[i] : __longlong_as_double(0x7ff8000000000000LL);
    }
    unsigned long long kl = ~0ULL;
#pragma unroll
    for (int s = 0; s < K; s++) {
        k[s] = (r[s] == r[s]) ? dkey(r[s]) : ~0ULL;
        kl = k[s] < kl ? k[s] : kl;
    }
    const unsigned long long KK = warp_min_u64(kl);
    if (KK == ~0ULL) return -1;
    const double vmin = dkey_inv(KK);
    int il = INT_MAX, close = 0;
#pragma unroll
    for (int s = K - 1; s >= 0; s--) {
        if (k[s] == KK) il = lane + 32 * s;
        if ((r[s] == r[s]) && !(vmin < __dsub_rn(r[s], margin))) close++;
    }
    const int imin = __reduce_min_sync(0xffffffffu, il);
    const int nclose = __reduce_add_sync(0xffffffffu, close);
    if (nclose == 1 && vmin < __longlong_as_double(0x7ff0000000000000LL)) return imin;
    if (vmin < __longlong_as_double(0x7ff0000000000000LL)) {  // ties: the wider certificate (see warp_tie_certificate)
        unsigned long long cm = 0ULL, dm = ~0ULL;
        int ic = INT_MAX;
#pragma unroll
        for (int s = K - 1; s >= 0; s--)
            if (r[s] == r[s]) {
                const double d = __dsub_rn(r[s], margin);
                if (!(vmin < d)) {
                    cm = k[s] > cm ? k[s] : cm;
                    ic = lane + 32 * s;
                } else {
                    const unsigned long long kd = dkey(d);
                    dm = kd < dm ? kd : dm;
                }
            }
        const int first = warp_tie_certificate(cm, dm, ic);
        if (first >= 0) return first;
    }
    return warp_margin_scan(count, margin, [&](int i, double& rr) {
        rr = ratio[i];
        return rr == rr;
    });
}
// Dispatch on the number of candidates (a B&B node of a 60 x 120 problem has up to 186 rows).
__device__ __forceinline__ int warp_margin_scan_staged(int count, double margin, const double* ratio) {
    if (count <= 64) return warp_margin_scan_regs<2>(count, margin, ratio);
    if (count <= 128) return warp_margin_scan_regs<4>(count, margin, ratio);
    if (count <= 192) return warp_margin_scan_regs<6>(count, margin, ratio);
    if (count <= 256) return warp_margin_scan_regs<8>(count, margin, ratio);
    return warp_margin_scan_cert(count, margin, [&](int i, double& rr) {
        rr = ratio[i];
        return rr == rr;
    });
}

__device__ __forceinline__ double neg_if(double v, bool flip) {
    // "v *= -1" of the reference (PrimalSimplex.cs:170-171, DualSimplex.cs:135,144-152)
    return flip ? __dmul_rn(v, -1.0) : v;
}

}  // namespace lpx
