// lpx_stream.hpp — internal cross-file declarations (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>

#include "../../include/lpx.h"

namespace lpx {

// whole-GPU streaming solver (lpx_stream.cu), host buffers in / host buffers out
int stream_solve_host(int m, int n, int sense, const double* A, const int* rel, const double* b, const double* c,
                      const lpx_options* opt, int* status, int* n_pivots, int* pivots, int pivots_cap, int* basis,
                      double* x, double* z, double* tableau, double* history, int history_cap);
// the same for the Dual Simplex (lpx_dual_session_open)
int stream_dual_solve_host(int m, int n, int sense, const double* A, const int* rel, const double* b, const double* c,
                           const lpx_options* opt, int* status, int* n_pivots, int* silent_pivots, int* pivots,
                           int pivots_cap, int* basis, double* x, double* z, double* tableau, double* history,
                           int history_cap);

// Revised Primal Simplex on the whole GPU (lpx_revised_stream.cuh), host buffers in / host buffers out; the caller
// holds the runtime lock and has checked the arguments and the reference's precondition
int revised_stream_solve(int m, int n, int sense, const double* A, const double* b, const double* c,
                         const lpx_options& o, int* status, int* n_iters, int* pivots, double* theta, int pivots_cap,
                         int* basis, int* nonbasic, double* xB, double* Binv, double* x, double* history,
                         int history_cap);

// register-resident batched kernel (lpx_reg.cu)
bool reg_kernel_supports(int m, int n, int m_expanded, bool has_rel);
int reg_launch_batched(int count, int m, int n, int sense, const double* A, const double* b, const double* c,
                       const lpx_options& opt, int* status, int* n_pivots, int* basis, double* x, double* z,
                       double* tableau, unsigned long long* total_pivots, cudaStream_t stream);

void set_bnb_instance(int k);

// sensitivity report kernels (lpx_sens.cu).  Batched: compact tableaux, b / c / basis strided per LP, rel shared.
int sens_launch_batched(int count, int m, int n, int mm, int sense, const int* rel, const double* b, const double* c,
                        const int* status, const int* basis, const double* tableau, double* report,
                        cudaStream_t stream);
// Session: one OPTIMAL tableau with rows ld doubles apart; rmap[i] = expanded row of constraint i's slack,
// -(row + 1) for an EQ constraint.  rowof: n + mm + 1 ints, partial: sens_session_partial_bytes(m, mm).
#define LPX_SENS_CHUNK_ROWS 32
size_t sens_session_partial_bytes(int m, int mm);
int sens_session_launch(int m, int n, int mm, size_t ld, int sense, const int* rmap, const double* b, const double* c,
                        const int* basis, const double* T, int* rowof, void* partial, double* report,
                        cudaStream_t stream);

}  // namespace lpx
