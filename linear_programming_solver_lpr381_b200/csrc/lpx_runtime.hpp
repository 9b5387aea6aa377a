// lpx_runtime.hpp — host-side runtime of liblpx: device selection, streams, cached device /
// pinned workspaces.  Nothing here is visible through the C ABI.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <mutex>
#include <vector>

namespace lpx {

// Grow-only cached buffers, keyed by a small slot id, so that repeated solves do not pay
// cudaMalloc / cudaHostAlloc every call.  Freed by lpx_shutdown().
#define LPX_BB_SETS 4
enum Slot {
    WS_A = 0, WS_B, WS_C, WS_REL, WS_STATUS, WS_NPIV, WS_SILENT, WS_PIVOTS, WS_BASIS, WS_X, WS_Z, WS_TABLEAU,
    WS_HISTORY, WS_NHIST, WS_SCRATCH, WS_TOTAL, WS_NODE_INST, WS_NODE_OFF, WS_NODE_CNT, WS_NODE_MODE, WS_EX_VAR,
    WS_EX_REL, WS_EX_RHS, WS_KN_ITEMS, WS_KN_ASSIGN, WS_KN_OUT, WS_KN_AUX, WS_KN_EXACT, WS_MISC0, WS_MISC1, WS_MISC2,
    WS_PL_IN, WS_PL_OUT, WS_PL_ALL,  // pooled-tree B&B: node descriptors, own results, everybody's results
    WS_SENS,  // sensitivity reports of lpx_primal_solve_sensitivity_batched
    WS_RO_REC, WS_RO_PAY, WS_RO_SRC, WS_RO_BASE_T, WS_RO_BASE_I,  // re-optimization: records, payloads, base
    WS_CUT_INT, WS_CUT_DBL, WS_CUT_STORE,  // cutting plane: integer / double outputs, the cut store without one
    WS_PM_INT, WS_PM_DBL,  // parametric analysis: integer / double inputs and outputs of lpx_parametric
    WS_TP_INT, WS_TP_DBL,  // two-phase Simplex: integer / double outputs of lpx_two_phase_solve_batched
    WS_BB_SET0,  // pipelined B&B: descriptors, results, scratch of each of LPX_BB_SETS evaluation sets
    WS_COUNT = WS_BB_SET0 + 3 * 4
};

struct Runtime {
    bool ready = false;
    int device = -1;
    int sms = 0;
    int smem_optin = 0;
    cudaStream_t stream = nullptr;      // compute
    cudaStream_t h2d = nullptr, d2h = nullptr;
    void* dev[WS_COUNT] = {};
    size_t dev_bytes[WS_COUNT] = {};
    void* pin[WS_COUNT] = {};
    size_t pin_bytes[WS_COUNT] = {};
    std::recursive_mutex mu;
};

Runtime& rt();
// Returns nullptr (and sets the error) on failure.
void* ws_dev(Slot s, size_t bytes);
void* ws_pin(Slot s, size_t bytes);
void knapsack_release_cache();  // lpx_knapsack.cu
void pooled_release_cache();    // lpx_pooled.cu
int comm_merge_u64(unsigned long long* dev, size_t words, cudaStream_t s);  // lpx_comm.cu
int comm_allgather_dev(const void* send, void* recv, size_t bytes, cudaStream_t s);  // lpx_comm.cu
int comm_world();
int comm_rank();

template <class T>
T* ws_dev_as(Slot s, size_t count) { return static_cast<T*>(ws_dev(s, count * sizeof(T))); }
template <class T>
T* ws_pin_as(Slot s, size_t count) { return static_cast<T*>(ws_pin(s, count * sizeof(T))); }

}  // namespace lpx
