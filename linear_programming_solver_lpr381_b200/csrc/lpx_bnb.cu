// lpx_bnb.cu — Branch & Bound over simplex relaxations: BranchAndBound.Solve / SolveNode,
// R/Models/Branch&Bound.cs:30-258.
//
// GPU node pool: every LP relaxation (the ~100 % hot spot, Branch&Bound.cs:57,148) is a node
// descriptor "base problem + unit rows"; all open nodes of all instances of a batch whose
// relaxations are not known yet are solved in ONE launch of the per-CTA kernels (lpx_cta.cuh; batches
// without a callback: the condensed-tableau kernel, lpx_cta_cond.cuh, a quarter of the instances per
// launch so that four rounds are in flight), primal and dual nodes mixed.  A relaxation is a pure function of its node, so nodes are
// evaluated speculatively (both children at once) and then COMMITTED ON THE HOST IN THE
// REFERENCE'S ORDER (depth-first, ceil child first), which keeps incumbents, pruning decisions
// and node numbering identical to the recursive C# code.
//
// Reference semantics kept on purpose (SURVEY.md F5): a child with a '>=' row is routed to Dual
// Simplex, whose result has no Solution/Tableau, so SolveNode rejects it ("Invalid Simplex
// result").  It is still solved (it is a _solver.Solve call and its tableaux are part of the
// iteration log) but never branches.
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>
#include <memory>
#include <vector>

#include "lpx_cta.cuh"
#include "lpx_runtime.hpp"
#include "lpx_stream.hpp"

namespace lpx {
namespace {

const double BB_EPS = 1e-6;  // BranchAndBound.EPS  (Branch&Bound.cs:24)
const int BB_MAX_DEPTH = 200;  // BranchAndBound.MaxDepth (Branch&Bound.cs:25)

struct Extra {
    int var, rel;
    double rhs;
};

struct Node {
    int inst = 0;
    int depth = 0;
    int parent_rec = -1;
    bool ceil_child = false;
    bool is_root_lp = false;
    std::vector<int> id_path;
    std::vector<Extra> extras;  // all unit rows from the root down to this node
    int mode = 0;               // 0 primal, 1 dual
    // evaluation
    bool evaluated = false;
    int lp_status = 0, n_pivots = 0, silent = 0;
    int flags = 0, branch = -1;  // node epilogue of the kernel: bit 0 IsFeasible, bit 1 IsIntegral; branching variable
    double z = 0;
    std::vector<double> x;
    const double* xp = nullptr;  // pipelined batches: x stays in the evaluation set's pinned result block
    int slot = -1;               // ... at this index
    std::vector<int> pivots;
    std::vector<double> history;
    int n_history = 0;
};

struct Instance {
    std::vector<std::unique_ptr<Node>> stack;  // back() is solved next
    int counter = 1;                           // _subProblemCounter
    double best = -std::numeric_limits<double>::infinity();
    bool have_best = false;
    std::vector<double> best_x;
    int records = 0;
    long long lp_pivots = 0;
    double lp_flops = 0;  // sum over node LPs of pivots x flops per pivot at that node's shape (SURVEY 8d)
    int root_status = 0;
    bool finished = false;
    std::vector<Node*> open;  // pipelined batches: this instance's nodes in the evaluation set in flight
};

// Math.Round(double): ties to even
inline double round_even(double v) { return std::nearbyint(v); }

struct BaseProblem {
    int m, n;
    const double* A;
    const int* rel;
    const double* b;
};

int choose_mode(const BaseProblem& bp, const std::vector<Extra>& extras) {
    for (int r = 0; r < bp.m; r++)
        if (bp.rel && (bp.rel[r] == 1 || bp.rel[r] == 2)) return 1;
    for (const Extra& e : extras)
        if (e.rel == 1 || e.rel == 2) return 1;
    return 0;
}

int expanded_rows(int m, const int* rel) {
    int mm = 0;
    for (int i = 0; i < m; i++) mm += (rel && rel[i] == 2) ? 2 : 1;
    return mm;
}

// host threads for the per-instance commit: LPX_HOST_THREADS, else min(8, half the cores)
inline int host_threads() {
    static const int n = [] {
        if (const char* e = getenv("LPX_HOST_THREADS")) return std::max(1, atoi(e));
        const unsigned hw = std::thread::hardware_concurrency();
        return (int)std::max(1u, std::min(8u, hw / 2));
    }();
    return n;
}

struct Driver {
    int count, m, n, sense, mm;
    const double *A, *rel_unused = nullptr, *b, *c;
    const int* rel;
    lpx_options opt;
    int flags;
    lpx_bnb_node_fn on_node;
    void* user;
    std::vector<Instance> inst;
    // device copies of the base problems
    double *dA = nullptr, *db = nullptr, *dc = nullptr;
    int* drel = nullptr;

    BaseProblem base(int k) const { return BaseProblem{m, n, A + (size_t)k * m * n, rel, b + (size_t)k * m}; }

    // ---- GPU evaluation of a list of nodes ---------------------------------------------------
    int evaluate(std::vector<Node*>& nodes, bool want_history) {
        if (nodes.empty()) return LPX_OK;
        Runtime& r = rt();
        // split by whether the node tableau fits in shared memory
        std::vector<Node*> group[2];
        for (Node* nd : nodes) {
            const int rows = mm + (int)nd->extras.size() + 1, width = n + rows;
            group[cta_fits_smem(rows, width) ? 0 : 1].push_back(nd);
        }
        for (int g = 0; g < 2; g++) {
            std::vector<Node*>& G = group[g];
            if (G.empty()) continue;
            const bool want_piv = on_node != nullptr;
            // every pivot of a node is logged: a primal node makes at most max_iterations, a dual node at most
            // 100 silent + LPX_DUAL_MAX_ITER (consumers index pivots[0 .. n_pivots), include/lpx.h)
            const int pivots_cap = want_piv ? std::max(opt.max_iterations, LPX_DUAL_MAX_ITER) + 100 : 0;
            if (!want_history) {
                int rc = launch_group(G, 0, G.size(), pivots_cap, 0);
                if (rc != LPX_OK) return rc;
            } else {
                // pass 1 sizes the histories, pass 2 re-solves in slices under a memory budget
                int rc = launch_group(G, 0, G.size(), pivots_cap, 0);
                if (rc != LPX_OK) return rc;
                const size_t budget = (size_t)1 << 30;
                size_t lo = 0;
                while (lo < G.size()) {
                    size_t hi = lo, bytes = 0;
                    int cap = 0, max_rows = 0;
                    while (hi < G.size()) {
                        const int rows = mm + (int)G[hi]->extras.size() + 1;
                        const int need = G[hi]->n_pivots - G[hi]->silent + 1;
                        const int ncap = std::max(cap, need), nrows = std::max(max_rows, rows);
                        const size_t nb = (size_t)(hi - lo + 1) * ncap * nrows * (n + nrows) * 8;
                        if (hi > lo && nb > budget) break;
                        cap = ncap;
                        max_rows = nrows;
                        bytes = nb;
                        hi++;
                    }
                    (void)bytes;
                    rc = launch_group(G, lo, hi, pivots_cap, cap);
                    if (rc != LPX_OK) return rc;
                    lo = hi;
                }
            }
        }
        (void)r;
        return LPX_OK;
    }

    // LPX_BNB_TRACE=1: wall time, launches, nodes and pivots per kernel kind, printed by run()
    double tr_time[2] = {0, 0};
    long tr_launch[2] = {0, 0}, tr_nodes[2] = {0, 0}, tr_piv[2] = {0, 0};

    int launch_group(std::vector<Node*>& G, size_t lo, size_t hi, int pivots_cap, int history_cap) {
        Runtime& r = rt();
        const auto tr_t0 = std::chrono::steady_clock::now();
        const int cnt = (int)(hi - lo);
        int max_extra = 0;
        size_t total_extra = 0;
        for (size_t k = lo; k < hi; k++) {
            max_extra = std::max(max_extra, (int)G[k]->extras.size());
            total_extra += G[k]->extras.size();
        }
        const int max_rows = mm + max_extra + 1, max_width = n + max_rows;
        const size_t tsize = (size_t)max_rows * max_width;

        // host staging of descriptors
        int* h_inst = ws_pin_as<int>(WS_NODE_INST, cnt);
        int* h_off = ws_pin_as<int>(WS_NODE_OFF, cnt);
        int* h_cnt = ws_pin_as<int>(WS_NODE_CNT, cnt);
        int* h_mode = ws_pin_as<int>(WS_NODE_MODE, cnt);
        int* h_var = ws_pin_as<int>(WS_EX_VAR, total_extra + 1);
        int* h_rel = ws_pin_as<int>(WS_EX_REL, total_extra + 1);
        double* h_rhs = ws_pin_as<double>(WS_EX_RHS, total_extra + 1);
        int* d_inst = ws_dev_as<int>(WS_NODE_INST, cnt);
        int* d_off = ws_dev_as<int>(WS_NODE_OFF, cnt);
        int* d_cnt = ws_dev_as<int>(WS_NODE_CNT, cnt);
        int* d_mode = ws_dev_as<int>(WS_NODE_MODE, cnt);
        int* d_var = ws_dev_as<int>(WS_EX_VAR, total_extra + 1);
        int* d_rel = ws_dev_as<int>(WS_EX_REL, total_extra + 1);
        double* d_rhs = ws_dev_as<double>(WS_EX_RHS, total_extra + 1);
        int* d_stat = ws_dev_as<int>(WS_STATUS, (size_t)cnt * 6);
        double* d_x = ws_dev_as<double>(WS_X, (size_t)cnt * n);
        double* d_z = ws_dev_as<double>(WS_Z, cnt);
        int* d_piv = pivots_cap ? ws_dev_as<int>(WS_PIVOTS, (size_t)cnt * pivots_cap * 2) : nullptr;
        double* d_hist = history_cap ? ws_dev_as<double>(WS_HISTORY, (size_t)cnt * history_cap * tsize) : nullptr;
        // a forced global-memory tableau needs working storage also where the tableau would fit shared memory
        const bool fits = cta_fits_smem(max_rows, max_width) && opt.kernel != LPX_KERNEL_CTA_GLOBAL;
        double* d_scratch = fits ? nullptr : ws_dev_as<double>(WS_SCRATCH, (size_t)cnt * tsize);
        int* h_stat = ws_pin_as<int>(WS_STATUS, (size_t)cnt * 6);
        double* h_x = ws_pin_as<double>(WS_X, (size_t)cnt * n);
        double* h_z = ws_pin_as<double>(WS_Z, cnt);
        if (!h_inst || !h_off || !h_cnt || !h_mode || !h_var || !h_rel || !h_rhs || !d_inst || !d_off || !d_cnt ||
            !d_mode || !d_var || !d_rel || !d_rhs || !d_stat || !d_x || !d_z || (pivots_cap && !d_piv) ||
            (history_cap && !d_hist) || (!fits && !d_scratch) || !h_stat || !h_x || !h_z)
            return LPX_E_CUDA;

        size_t off = 0;
        for (int k = 0; k < cnt; k++) {
            Node* nd = G[lo + k];
            h_inst[k] = nd->inst;
            h_off[k] = (int)off;
            h_cnt[k] = (int)nd->extras.size();
            h_mode[k] = nd->mode;
            for (const Extra& e : nd->extras) {
                h_var[off] = e.var;
                h_rel[off] = e.rel;
                h_rhs[off] = e.rhs;
                off++;
            }
        }
        cudaStream_t s = r.stream;
        LPX_CUDA(cudaMemcpyAsync(d_inst, h_inst, (size_t)cnt * 4, cudaMemcpyHostToDevice, s));
        LPX_CUDA(cudaMemcpyAsync(d_off, h_off, (size_t)cnt * 4, cudaMemcpyHostToDevice, s));
        LPX_CUDA(cudaMemcpyAsync(d_cnt, h_cnt, (size_t)cnt * 4, cudaMemcpyHostToDevice, s));
        LPX_CUDA(cudaMemcpyAsync(d_mode, h_mode, (size_t)cnt * 4, cudaMemcpyHostToDevice, s));
        if (total_extra) {
            LPX_CUDA(cudaMemcpyAsync(d_var, h_var, total_extra * 4, cudaMemcpyHostToDevice, s));
            LPX_CUDA(cudaMemcpyAsync(d_rel, h_rel, total_extra * 4, cudaMemcpyHostToDevice, s));
            LPX_CUDA(cudaMemcpyAsync(d_rhs, h_rhs, total_extra * 8, cudaMemcpyHostToDevice, s));
        }

        CtaBatch B;
        std::memset(&B, 0, sizeof B);
        B.A = dA;
        B.b = db;
        B.c = dc;
        B.rel = rel ? drel : nullptr;
        B.strideA = (long long)m * n;
        B.strideB = m;
        B.strideC = n;
        B.m_in = m;
        B.n = n;
        B.sense = sense;
        B.m_base = mm;
        B.node_inst = d_inst;
        B.node_extra_off = d_off;
        B.node_extra_cnt = d_cnt;
        B.node_mode = d_mode;
        B.ex_var = d_var;
        B.ex_rel = d_rel;
        B.ex_rhs = d_rhs;
        B.max_iter = opt.max_iterations;
        B.max_rows = max_rows;
        B.max_width = max_width;
        B.scratch = d_scratch;
        B.scratch_stride = (long long)tsize;
        B.status = d_stat;
        B.n_pivots = d_stat + cnt;
        B.silent = d_stat + 2 * cnt;
        B.n_history = d_stat + 3 * cnt;
        B.node_flags = d_stat + 4 * cnt;
        B.node_branch = d_stat + 5 * cnt;
        B.pivots = d_piv;
        B.pivots_cap = pivots_cap;
        B.x = d_x;
        B.z = d_z;
        B.history = d_hist;
        B.history_stride = (long long)((size_t)history_cap * tsize);
        B.history_cap = history_cap;
        int rc = cta_launch(B, cnt, opt.kernel == LPX_KERNEL_CTA_GLOBAL ? LPX_KERNEL_CTA_GLOBAL : LPX_KERNEL_AUTO,
                            opt.threads, s, nullptr);
        if (rc != LPX_OK) return rc;
        LPX_CUDA(cudaMemcpyAsync(h_stat, d_stat, (size_t)cnt * 24, cudaMemcpyDeviceToHost, s));
        LPX_CUDA(cudaMemcpyAsync(h_x, d_x, (size_t)cnt * n * 8, cudaMemcpyDeviceToHost, s));
        LPX_CUDA(cudaMemcpyAsync(h_z, d_z, (size_t)cnt * 8, cudaMemcpyDeviceToHost, s));
        LPX_CUDA(cudaStreamSynchronize(s));
        {
            const int kind = fits ? 0 : 1;
            tr_time[kind] += std::chrono::duration<double>(std::chrono::steady_clock::now() - tr_t0).count();
            tr_launch[kind]++;
            tr_nodes[kind] += cnt;
            for (int k = 0; k < cnt; k++) tr_piv[kind] += h_stat[cnt + k];
        }
        for (int k = 0; k < cnt; k++) {
            Node* nd = G[lo + k];
            nd->evaluated = true;
            nd->lp_status = h_stat[k];
            nd->n_pivots = h_stat[cnt + k];
            nd->silent = h_stat[2 * cnt + k];
            nd->flags = h_stat[4 * cnt + k];
            nd->branch = h_stat[5 * cnt + k];
            nd->z = h_z[k];
            nd->x.assign(h_x + (size_t)k * n, h_x + (size_t)(k + 1) * n);
            if (pivots_cap) {
                const int np = std::min(nd->n_pivots, pivots_cap);
                nd->pivots.resize((size_t)np * 2);
                if (np)
                    LPX_CUDA(cudaMemcpy(nd->pivots.data(), d_piv + (size_t)k * pivots_cap * 2, (size_t)np * 8,
                                        cudaMemcpyDeviceToHost));
            }
            if (history_cap) {
                const int rows = mm + (int)nd->extras.size() + 1, width = n + rows;
                const int nh = h_stat[3 * cnt + k];
                nd->n_history = nh;
                nd->history.resize((size_t)nh * rows * width);
                if (nh)
                    LPX_CUDA(cudaMemcpy(nd->history.data(), d_hist + (size_t)k * history_cap * tsize,
                                        nd->history.size() * 8, cudaMemcpyDeviceToHost));
            }
        }
        return LPX_OK;
    }

    // ---- pipelined evaluation (batches without a callback) ---------------------------------------
    // The batch is cut into 2-4 evaluation SETS of instances.  One round of a set = all its open nodes:
    // descriptors staged in one pinned blob, one upload, one launch per occupancy class, one download, one
    // event — on the set's own stream, so that the tail of one set's kernel overlaps the next set's.  While
    // the GPU solves the other sets the host commits this set's round (SolveNode bodies, independent per
    // instance) and stages its next one on a few persistent worker threads.
    struct HostPool {
        std::vector<std::thread> th;
        std::mutex mu;
        std::condition_variable cv;
        std::atomic<unsigned> gen{0};
        std::atomic<int> next{0}, pending{0};
        std::atomic<bool> stop{false};
        int hi = 0, chunk = 1;
        const std::function<void(int, int)>* fn = nullptr;

        explicit HostPool(int workers) {
            for (int t = 0; t < workers; t++) th.emplace_back([this] { loop(); });
        }
        ~HostPool() {
            {
                std::lock_guard<std::mutex> lk(mu);
                stop.store(true);
                gen.fetch_add(1, std::memory_order_release);
            }
            cv.notify_all();
            for (std::thread& t : th) t.join();
        }
        void work() {
            for (;;) {
                const int a = next.fetch_add(chunk);
                if (a >= hi) break;
                (*fn)(a, std::min(hi, a + chunk));
            }
        }
        void loop() {
            unsigned seen = 0;
            for (;;) {
                int spins = 0;
                while (gen.load(std::memory_order_acquire) == seen) {
                    if (++spins < 4000) {
                        std::this_thread::yield();
                        continue;
                    }
                    std::unique_lock<std::mutex> lk(mu);
                    cv.wait(lk, [&] { return gen.load(std::memory_order_acquire) != seen; });
                }
                if (stop.load()) return;
                seen = gen.load(std::memory_order_acquire);
                work();
                pending.fetch_sub(1, std::memory_order_release);
            }
        }
        // f(a, b) over [lo, hi_) in chunks, on the workers and the calling thread
        void run(int lo, int hi_, int chunk_, const std::function<void(int, int)>& f) {
            if (th.empty() || hi_ - lo <= chunk_) {
                if (hi_ > lo) f(lo, hi_);
                return;
            }
            fn = &f;
            hi = hi_;
            chunk = chunk_;
            next.store(lo);
            pending.store((int)th.size());
            {
                std::lock_guard<std::mutex> lk(mu);
                gen.fetch_add(1, std::memory_order_release);
            }
            cv.notify_all();
            work();
            while (pending.load(std::memory_order_acquire) != 0) std::this_thread::yield();
        }
    };

    bool use_condensed = true;  // run(): opt.kernel == AUTO and LPX_BNB_FULL_TABLEAU unset
    struct EvalSet {
        int lo = 0, hi = 0;         // instances [lo, hi)
        std::vector<Node*> nodes;   // occupancy class 0 first, then class 1
        std::vector<int> offs;      // first extra row of each node in the blob
        int total = 0;
        cudaStream_t stream = nullptr;
        cudaEvent_t done = nullptr, began = nullptr;
        bool active = false;
        int* h_stat = nullptr;
        double *h_x = nullptr, *h_z = nullptr;
    };
    std::vector<EvalSet> sets;
    bool trace_gpu = false;
    double gpu_ms = 0;
    long long* d_prof = nullptr;  // LPX_BNB_TRACE: phase cycles of the condensed kernel, two occupancy classes x 14 slots

    // stage and launch the open nodes (Instance::open) of set g
    int enqueue(int g, HostPool& pool) {
        EvalSet& E = sets[g];
        E.active = false;
        const auto tr_t0 = std::chrono::steady_clock::now();
        // no callback on this path, so nobody reads a node's tableau: when the deepest node's CONDENSED tableau
        // (non-basic columns + RHS, lpx_cta_cond.cuh) fits one SM, every node runs on the condensed kernel —
        // in two launches, so that the shallow nodes (two CTAs per SM) are not held to the occupancy of the
        // deepest one.  Otherwise: nodes that fit one SM's shared memory | cluster / global-memory nodes.
        int deepest = -1;
        for (int k = E.lo; k < E.hi; k++)
            for (Node* nd : inst[k].open) deepest = std::max(deepest, (int)nd->extras.size());
        if (deepest < 0) return LPX_OK;
        const bool cond = use_condensed && cta_condensed_fits(mm + deepest + 1, n);
        // evaluation classes, one launch each.  Condensed: 0 / 1 = two / one CTA per SM.  Otherwise: 0 = the
        // node's full tableau fits one SM's shared memory, 1 = cluster / global memory.
        std::vector<Node*> cls[2];
        int max_extra[2] = {0, 0};
        for (int k = E.lo; k < E.hi; k++)
            for (Node* nd : inst[k].open) {
                const int rows = mm + (int)nd->extras.size() + 1, width = n + rows;
                const int kind = (cond ? cta_condensed_ctas_per_sm(rows, n) >= 2 : cta_fits_smem(rows, width)) ? 0 : 1;
                cls[kind].push_back(nd);
                max_extra[kind] = std::max(max_extra[kind], (int)nd->extras.size());
            }
        E.nodes.clear();
        int first[3] = {0, 0, 0};
        for (int kind = 0; kind < 2; kind++) {
            E.nodes.insert(E.nodes.end(), cls[kind].begin(), cls[kind].end());
            first[kind + 1] = (int)E.nodes.size();
        }
        const int total = E.total = (int)E.nodes.size();
        E.offs.resize((size_t)total + 1);
        size_t total_extra = 0;
        for (int k = 0; k < total; k++) {
            E.offs[k] = (int)total_extra;
            total_extra += E.nodes[k]->extras.size();
        }
        // input blob: inst, off, cnt, mode (ints per node), var, rel (ints per extra), rhs (doubles per extra)
        const size_t in_ints = (size_t)4 * total + 2 * (total_extra + 1);
        const size_t in_bytes = ((in_ints * 4 + 7) & ~(size_t)7) + (total_extra + 1) * 8;
        // output blob: status, n_pivots, silent, n_history, flags, branch (ints), z, x (doubles)
        const size_t out_bytes = (size_t)total * 6 * 4 + (size_t)total * 8 + (size_t)total * n * 8;
        const Slot s_in = (Slot)(WS_BB_SET0 + 3 * g), s_out = (Slot)(WS_BB_SET0 + 3 * g + 1),
                   s_scr = (Slot)(WS_BB_SET0 + 3 * g + 2);
        unsigned char* h_in = (unsigned char*)ws_pin(s_in, in_bytes);
        unsigned char* d_in = (unsigned char*)ws_dev(s_in, in_bytes);
        unsigned char* h_out = (unsigned char*)ws_pin(s_out, out_bytes);
        unsigned char* d_out = (unsigned char*)ws_dev(s_out, out_bytes);
        if (!h_in || !d_in || !h_out || !d_out) return LPX_E_CUDA;
        int* hi = (int*)h_in;
        int *h_inst = hi, *h_off = hi + total, *h_cnt = hi + 2 * total, *h_mode = hi + 3 * total;
        int *h_var = hi + 4 * total, *h_rel = h_var + total_extra + 1;
        double* h_rhs = (double*)(h_in + ((in_ints * 4 + 7) & ~(size_t)7));
        pool.run(0, total, 32, [&](int a, int b) {
            for (int k = a; k < b; k++) {
                Node* nd = E.nodes[k];
                nd->slot = k;
                size_t off = (size_t)E.offs[k];
                h_inst[k] = nd->inst;
                h_off[k] = (int)off;
                h_cnt[k] = (int)nd->extras.size();
                h_mode[k] = nd->mode;
                for (const Extra& e : nd->extras) {
                    h_var[off] = e.var;
                    h_rel[off] = e.rel;
                    h_rhs[off] = e.rhs;
                    off++;
                }
            }
        });
        cudaStream_t s = E.stream;
        if (trace_gpu) LPX_CUDA(cudaEventRecord(E.began, s));
        LPX_CUDA(cudaMemcpyAsync(d_in, h_in, in_bytes, cudaMemcpyHostToDevice, s));
        int* di = (int*)d_in;
        int* d_stat = (int*)d_out;
        double* d_z = (double*)(d_out + (size_t)total * 24);
        double* d_x = d_z + total;
        for (int kind = 0; kind < 2; kind++) {
            const int lo = first[kind], cnt = first[kind + 1] - first[kind];
            if (cnt == 0) continue;
            const int max_rows = mm + max_extra[kind] + 1, max_width = n + max_rows;
            const size_t tsize = (size_t)max_rows * max_width;
            CtaBatch B;
            std::memset(&B, 0, sizeof B);
            B.A = dA;
            B.b = db;
            B.c = dc;
            B.rel = rel ? drel : nullptr;
            B.strideA = (long long)m * n;
            B.strideB = m;
            B.strideC = n;
            B.m_in = m;
            B.n = n;
            B.sense = sense;
            B.m_base = mm;
            B.node_inst = di + lo;
            B.node_extra_off = di + total + lo;
            B.node_extra_cnt = di + 2 * total + lo;
            B.node_mode = di + 3 * total + lo;
            B.ex_var = di + 4 * total;
            B.ex_rel = di + 4 * total + total_extra + 1;
            B.ex_rhs = (const double*)(d_in + ((in_ints * 4 + 7) & ~(size_t)7));
            B.max_iter = opt.max_iterations;
            B.max_rows = max_rows;
            B.max_width = max_width;
            // beyond a 4-CTA cluster, or a forced global-memory tableau (either kind of node)
            if (!cond && ((kind == 1 && cta_cluster_size_for(max_rows, max_width) == 0) ||
                          opt.kernel == LPX_KERNEL_CTA_GLOBAL)) {
                double* sc = (double*)ws_dev(s_scr, (size_t)cnt * tsize * 8);
                if (!sc) return LPX_E_CUDA;
                B.scratch = sc;
                B.scratch_stride = (long long)tsize;
            }
            B.status = d_stat + lo;
            B.n_pivots = d_stat + total + lo;
            B.silent = d_stat + 2 * total + lo;
            B.n_history = d_stat + 3 * total + lo;
            B.node_flags = d_stat + 4 * total + lo;
            B.node_branch = d_stat + 5 * total + lo;
            B.x = d_x + (size_t)lo * n;
            B.z = d_z + lo;
            if (d_prof) B.dbg = d_prof + 14 * kind;
            int rc = cond ? cta_condensed_launch(B, cnt, s)
                          : cta_launch(B, cnt, opt.kernel == LPX_KERNEL_CTA_GLOBAL ? LPX_KERNEL_CTA_GLOBAL : LPX_KERNEL_AUTO,
                                       opt.threads, s, nullptr);
            if (rc != LPX_OK) return rc;
            tr_launch[kind]++;
            tr_nodes[kind] += cnt;
        }
        LPX_CUDA(cudaMemcpyAsync(h_out, d_out, out_bytes, cudaMemcpyDeviceToHost, s));
        LPX_CUDA(cudaEventRecord(E.done, s));
        E.h_stat = (int*)h_out;
        E.h_z = (double*)(h_out + (size_t)total * 24);
        E.h_x = E.h_z + total;
        E.active = true;
        tr_time[1] += std::chrono::duration<double>(std::chrono::steady_clock::now() - tr_t0).count();
        return LPX_OK;
    }

    // results of set g's round -> its nodes, SolveNode bodies in the reference's order, next round's open nodes
    int finish_and_commit(int g, HostPool& pool) {
        EvalSet& E = sets[g];
        if (E.active) {
            const auto tr_t0 = std::chrono::steady_clock::now();
            LPX_CUDA(cudaEventSynchronize(E.done));
            tr_time[0] += std::chrono::duration<double>(std::chrono::steady_clock::now() - tr_t0).count();
            if (trace_gpu) {
                float ms = 0;
                cudaEventElapsedTime(&ms, E.began, E.done);
                gpu_ms += ms;
            }
        }
        const int total = E.total;
        pool.run(E.lo, E.hi, 4, [&](int a, int b) {
            for (int k = a; k < b; k++) {
                Instance& I = inst[k];
                for (Node* nd : I.open) {
                    const int q = nd->slot;
                    nd->evaluated = true;
                    nd->lp_status = E.h_stat[q];
                    nd->n_pivots = E.h_stat[total + q];
                    nd->silent = E.h_stat[2 * total + q];
                    nd->flags = E.h_stat[4 * total + q];
                    nd->branch = E.h_stat[5 * total + q];
                    nd->z = E.h_z[q];
                    nd->xp = E.h_x + (size_t)q * n;
                }
                I.open.clear();
                while (!I.finished && !I.stack.empty() && I.stack.back()->evaluated) {
                    std::unique_ptr<Node> nd = std::move(I.stack.back());
                    I.stack.pop_back();
                    if (nd->is_root_lp) commit_root_lp(I, std::move(nd));
                    else commit_node(I, std::move(nd));
                }
                if (I.stack.empty()) I.finished = true;
                if (!I.finished)  // the nodes without a relaxation yet are the top of the stack
                    for (size_t i = I.stack.size(); i-- > 0 && !I.stack[i]->evaluated;) I.open.push_back(I.stack[i].get());
            }
        });
        E.active = false;
        return LPX_OK;
    }

    int run_pipelined() {
        const int nsets = std::max(2, std::min(LPX_BB_SETS, count / 64));
        sets.resize(nsets);
        int rc = LPX_OK;
        LPX_CUDA(cudaStreamSynchronize(rt().stream));  // the base problems are on the device
        trace_gpu = getenv("LPX_BNB_TRACE") != nullptr;
        if (trace_gpu && cudaMalloc(&d_prof, 28 * 8) == cudaSuccess) cudaMemset(d_prof, 0, 28 * 8);
        for (int g = 0; g < nsets; g++) {
            EvalSet& E = sets[g];
            E.lo = (int)((long long)count * g / nsets);
            E.hi = (int)((long long)count * (g + 1) / nsets);
            if (cudaStreamCreateWithFlags(&E.stream, cudaStreamNonBlocking) != cudaSuccess ||
                cudaEventCreateWithFlags(&E.done, trace_gpu ? cudaEventDefault : cudaEventDisableTiming) != cudaSuccess ||
                cudaEventCreateWithFlags(&E.began, cudaEventDefault) != cudaSuccess)
                rc = LPX_E_CUDA;
        }
        if (rc == LPX_OK) {
            HostPool pool(host_threads() - 1);
            for (int g = 0; g < nsets && rc == LPX_OK; g++)
                if ((rc = finish_and_commit(g, pool)) == LPX_OK) rc = enqueue(g, pool);  // nothing to commit yet: the roots
            bool any = true;
            while (rc == LPX_OK && any) {
                any = false;
                for (int g = 0; g < nsets && rc == LPX_OK; g++) {
                    if (!sets[g].active) continue;
                    any = true;
                    if ((rc = finish_and_commit(g, pool)) == LPX_OK) rc = enqueue(g, pool);
                }
            }
        }
        for (EvalSet& E : sets) {
            if (E.stream) {
                cudaStreamSynchronize(E.stream);
                cudaStreamDestroy(E.stream);
            }
            if (E.done) cudaEventDestroy(E.done);
            if (E.began) cudaEventDestroy(E.began);
        }
        long long hp[28] = {0};
        if (d_prof) {
            cudaMemcpy(hp, d_prof, sizeof hp, cudaMemcpyDeviceToHost);
            cudaFree(d_prof);
            d_prof = nullptr;
        }
        if (rc != LPX_OK) {
            if (rc == LPX_E_CUDA) set_error("lpx_bnb_simplex: CUDA error in the pipelined node evaluation");
            return rc;
        }
        if (trace_gpu)
            for (int kind = 0; kind < 2; kind++) {
                const long long* h = hp + 14 * kind;
                if (!h[13]) continue;
                const double pp = (double)std::max(1LL, h[10]), dp = (double)std::max(1LL, h[11]), nc = (double)h[13];
                fprintf(stderr, "[bnb trace] condensed kernel, class %d: %lld nodes, %.0f cycles each (build %.0f, between/after "
                                "the loops %.0f); %lld primal pivots: ratios %.0f, scan %.0f, staging %.0f, update %.0f cycles; "
                                "%lld dual pivots: leaving %.0f, entering %.0f, staging %.0f, update %.0f\n",
                        kind, h[13], h[12] / nc, h[8] / nc, h[9] / nc, h[10], h[0] / pp, h[1] / pp, h[2] / pp, h[3] / pp,
                        h[11], h[4] / dp, h[5] / dp, h[6] / dp, h[7] / dp);
            }
        if (trace_gpu)
            fprintf(stderr, "[bnb trace] pipelined, %d sets: %.3f s waiting for the GPU, %.3f s staging + enqueueing, GPU busy "
                            "(sum over sets, upload to download) %.3f s; class 0: %ld launches / %ld nodes, class 1: %ld / %ld\n",
                    nsets, tr_time[0], tr_time[1], gpu_ms * 1e-3, tr_launch[0], tr_nodes[0], tr_launch[1], tr_nodes[1]);
        return LPX_OK;
    }

    // ---- commit logic -------------------------------------------------------------------------
    void emit(Instance& I, const Node& nd, int outcome, int branch_var, int floor_val, int ceil_val, int rec_index) {
        if (!on_node) return;
        lpx_bnb_node rec;
        std::memset(&rec, 0, sizeof rec);
        rec.index = rec_index;
        rec.depth = nd.depth;
        rec.parent = nd.parent_rec;
        rec.is_ceil_child = nd.ceil_child ? 1 : 0;
        rec.id_path_len = (int)nd.id_path.size();
        rec.id_path = nd.id_path.data();
        rec.bound_var = nd.extras.empty() || nd.is_root_lp ? -1 : nd.extras.back().var;
        rec.bound_val = nd.extras.empty() ? 0 : (int)nd.extras.back().rhs;
        rec.algo = nd.mode;
        rec.lp_status = nd.lp_status;
        rec.outcome = outcome;
        rec.n_pivots = nd.n_pivots;
        rec.silent_pivots = nd.silent;
        rec.pivots = nd.pivots.data();
        rec.rows = mm + (int)nd.extras.size() + 1;
        rec.cols = n + rec.rows;
        rec.z = nd.z;
        rec.x = nd.x.data();
        rec.branch_var = branch_var;
        rec.floor_val = floor_val;
        rec.ceil_val = ceil_val;
        rec.n_history = nd.n_history;
        rec.history = nd.history.data();
        set_bnb_instance(nd.inst);
        on_node(&rec, user);
        (void)I;
    }

    // 2 m (n+m+1) + (n+m+1) flops per pivot of an (m+1) x (n+m+1) tableau (SURVEY 8d), m = this node's rows
    double pivot_flops(const Node& nd) const {
        const double md = mm + (double)nd.extras.size(), w = n + md + 1;
        return (double)nd.n_pivots * (2.0 * md * w + w);
    }

    // One SolveNode body (Branch&Bound.cs:128-258) for an evaluated node.
    void commit_node(Instance& I, std::unique_ptr<Node> ndp) {
        Node& nd = *ndp;
        const int rec = I.records++;
        if (nd.depth > BB_MAX_DEPTH) {
            emit(I, nd, LPX_BNB_DEPTH, -1, 0, 0, rec);
            return;
        }
        I.lp_pivots += nd.n_pivots;
        I.lp_flops += pivot_flops(nd);
        if (nd.lp_status < 0) {  // the solve threw
            emit(I, nd, LPX_BNB_ERROR, -1, 0, 0, rec);
            return;
        }
        if (nd.mode == 1) {  // Dual Simplex returns no Solution/Tableau/Basis/VarNames
            emit(I, nd, LPX_BNB_INVALID, -1, 0, 0, rec);
            return;
        }
        const double* x = nd.xp ? nd.xp : nd.x.data();
        const double z = nd.z;
        const BaseProblem bp = base(nd.inst);
        // IsFeasible, IsIntegral and the branching variable were computed by the node's kernel (cta_node_epilogue)
        if (!(nd.flags & 1)) {
            emit(I, nd, LPX_BNB_INFEASIBLE, -1, 0, 0, rec);
            return;
        }
        if (z <= I.best + BB_EPS) {
            emit(I, nd, LPX_BNB_PRUNED, -1, 0, 0, rec);
            return;
        }
        if (nd.flags & 2) {
            I.best = z;
            I.have_best = true;
            I.best_x.resize(n);
            for (int i = 0; i < n; i++) I.best_x[i] = round_even(x[i]);
            emit(I, nd, LPX_BNB_INCUMBENT, -1, 0, 0, rec);
            return;
        }
        const int frac_index = nd.branch;
        if (frac_index == -1) {
            emit(I, nd, LPX_BNB_NOFRAC, -1, 0, 0, rec);
            return;
        }
        const int floor_val = (int)std::floor(x[frac_index]);
        const int ceil_val = (int)std::ceil(x[frac_index]);
        emit(I, nd, LPX_BNB_BRANCHED, frac_index, floor_val, ceil_val, rec);

        auto child = [&](bool ceil_side, int id) {
            std::unique_ptr<Node> ch(new Node());
            ch->inst = nd.inst;
            ch->depth = nd.depth + 1;
            ch->parent_rec = rec;
            ch->ceil_child = ceil_side;
            if (on_node) {  // only the callback's records carry the id path
                ch->id_path = nd.id_path;
                ch->id_path.push_back(id);
            }
            ch->extras = nd.extras;
            ch->extras.push_back(Extra{frac_index, ceil_side ? 1 : 0, (double)(ceil_side ? ceil_val : floor_val)});
            ch->mode = choose_mode(bp, ch->extras);
            if (ch->depth > BB_MAX_DEPTH) ch->evaluated = true;  // pruned without an LP
            return ch;
        };
        const int ceil_id = I.counter, floor_id = I.counter + 1;
        I.counter += 2;
        // SolveNode(right) then SolveNode(left): the stack pops the ceil child first
        I.stack.push_back(child(false, floor_id));
        I.stack.push_back(child(true, ceil_id));
    }

    // Root LP of BranchAndBound.Solve (Branch&Bound.cs:53-95).
    void commit_root_lp(Instance& I, std::unique_ptr<Node> ndp) {
        Node& nd = *ndp;
        const int rec = I.records++;
        I.lp_pivots += nd.n_pivots;
        I.lp_flops += pivot_flops(nd);
        I.root_status = nd.lp_status;
        if (nd.lp_status < 0) {
            emit(I, nd, LPX_BNB_ERROR, -1, 0, 0, rec);
            I.finished = true;
            return;
        }
        if (nd.mode == 1) {
            emit(I, nd, LPX_BNB_INVALID, -1, 0, 0, rec);
            I.finished = true;
            return;
        }
        const BaseProblem bp = base(nd.inst);
        if ((nd.flags & 3) == 3) {
            I.best = nd.z;
            I.have_best = true;
            I.best_x.resize(n);
            const double* xr = nd.xp ? nd.xp : nd.x.data();
            for (int i = 0; i < n; i++) I.best_x[i] = round_even(xr[i]);
            emit(I, nd, LPX_BNB_INCUMBENT, -1, 0, 0, rec);
            I.finished = true;
            return;
        }
        emit(I, nd, LPX_BNB_BRANCHED, -1, 0, 0, rec);
        // SolveNode(problem, "Root Problem", "", ..., 0): the root LP is solved a second time
        std::unique_ptr<Node> again(new Node());
        again->inst = nd.inst;
        again->depth = 0;
        again->parent_rec = rec;
        again->mode = nd.mode;
        I.stack.push_back(std::move(again));
    }

    int run() {
        Runtime& r = rt();
        // base problems to the device once
        dA = ws_dev_as<double>(WS_A, (size_t)count * m * n);
        db = ws_dev_as<double>(WS_B, (size_t)count * m);
        dc = ws_dev_as<double>(WS_C, (size_t)count * n);
        drel = ws_dev_as<int>(WS_REL, m);
        if (!dA || !db || !dc || !drel) return LPX_E_CUDA;
        LPX_CUDA(cudaMemcpyAsync(dA, A, (size_t)count * m * n * 8, cudaMemcpyHostToDevice, r.stream));
        LPX_CUDA(cudaMemcpyAsync(db, b, (size_t)count * m * 8, cudaMemcpyHostToDevice, r.stream));
        LPX_CUDA(cudaMemcpyAsync(dc, c, (size_t)count * n * 8, cudaMemcpyHostToDevice, r.stream));
        if (rel) LPX_CUDA(cudaMemcpyAsync(drel, rel, (size_t)m * 4, cudaMemcpyHostToDevice, r.stream));

        inst.resize(count);
        for (int k = 0; k < count; k++) {
            std::unique_ptr<Node> root(new Node());
            root->inst = k;
            root->is_root_lp = true;
            root->mode = choose_mode(base(k), root->extras);
            inst[k].stack.push_back(std::move(root));
        }
        const bool want_history = (flags & LPX_BNB_WANT_HISTORY) && on_node;
        use_condensed = opt.kernel == LPX_KERNEL_AUTO && !std::getenv("LPX_BNB_FULL_TABLEAU");
        if (!on_node) return run_pipelined();  // no callback: nobody needs a node's tableaux
        while (true) {
            std::vector<Node*> todo;
            for (Instance& I : inst)
                if (!I.finished)
                    for (auto& nd : I.stack)
                        if (!nd->evaluated) todo.push_back(nd.get());
            if (todo.empty()) {
                if (getenv("LPX_BNB_TRACE"))
                    for (int kind = 0; kind < 2; kind++)
                        fprintf(stderr, "[bnb trace] %s kernel: %.3f s, %ld launches, %ld nodes, %ld pivots\n",
                                kind ? "cluster / global-memory" : "shared-memory", tr_time[kind], tr_launch[kind], tr_nodes[kind],
                                tr_piv[kind]);
                break;
            }
            int rc = evaluate(todo, want_history);
            if (rc != LPX_OK) return rc;
            // SolveNode bodies of the evaluated nodes, on the calling thread: the callback's records must arrive in
            // the reference's order (calls without a callback take run_pipelined)
            for (Instance& I : inst) {
                while (!I.finished && !I.stack.empty() && I.stack.back()->evaluated) {
                    std::unique_ptr<Node> nd = std::move(I.stack.back());
                    I.stack.pop_back();
                    if (nd->is_root_lp) commit_root_lp(I, std::move(nd));
                    else commit_node(I, std::move(nd));
                }
                if (I.stack.empty()) I.finished = true;
            }
        }
        return LPX_OK;
    }
};

}  // namespace
}  // namespace lpx

using namespace lpx;

static thread_local double g_last_stats[4] = {0, 0, 0, 0};

extern "C" {

int lpx_bnb_last_stats(double* stats4) {
    if (!stats4) return LPX_E_BAD_ARGS;
    for (int k = 0; k < 4; k++) stats4[k] = g_last_stats[k];
    return LPX_OK;
}

int lpx_bnb_simplex_batched(int count, int m, int n, int sense, const double* A, const int* rel, const double* b,
                            const double* c, const lpx_options* opt, int flags, int* found, double* best_z,
                            double* best_x, int* n_nodes, long long* n_lp_pivots, int* root_status,
                            lpx_bnb_node_fn on_node, void* user) {
    if (count < 1 || m < 1 || n < 1 || !A || !b || !c || (sense != 0 && sense != 1)) {
        set_error("lpx_bnb_simplex: bad arguments");
        return LPX_E_BAD_ARGS;
    }
    if (rel)
        for (int i = 0; i < m; i++)
            if (rel[i] < 0 || rel[i] > 2) {
                set_error("lpx_bnb_simplex: rel[i] must be 0, 1 or 2");
                return LPX_E_BAD_ARGS;
            }
    int rc = ensure_device();
    if (rc != LPX_OK) return rc;
    std::lock_guard<std::recursive_mutex> lk(rt().mu);
    Driver d;
    d.count = count;
    d.m = m;
    d.n = n;
    d.sense = sense;
    d.mm = expanded_rows(m, rel);
    d.A = A;
    d.b = b;
    d.c = c;
    d.rel = rel;
    lpx_default_options(&d.opt);
    if (opt) d.opt = *opt;
    d.flags = flags;
    d.on_node = on_node;
    d.user = user;
    const auto t_run = std::chrono::steady_clock::now();
    rc = d.run();
    if (rc != LPX_OK) return rc;
    g_last_stats[0] = 0;
    g_last_stats[2] = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_run).count();
    // pipelined batches keep the GPU busy for the whole search: its seconds are the call's
    g_last_stats[1] = !on_node ? g_last_stats[2] : d.tr_time[0] + d.tr_time[1];
    g_last_stats[3] = (double)(d.tr_launch[0] + d.tr_launch[1]);
    for (int k = 0; k < count; k++) g_last_stats[0] += d.inst[k].lp_flops;
    for (int k = 0; k < count; k++) {
        const Instance& I = d.inst[k];
        if (found) found[k] = I.have_best ? 1 : 0;
        if (best_z) best_z[k] = I.best;
        if (best_x && I.have_best)
            for (int j = 0; j < n; j++) best_x[(size_t)k * n + j] = I.best_x[j];
        if (n_nodes) n_nodes[k] = I.records;
        if (n_lp_pivots) n_lp_pivots[k] = I.lp_pivots;
        if (root_status) root_status[k] = I.root_status;
    }
    return LPX_OK;
}

int lpx_bnb_simplex(int m, int n, int sense, const double* A, const int* rel, const double* b, const double* c,
                    const lpx_options* opt, int flags, int* found, double* best_z, double* best_x, int* n_nodes,
                    long long* n_lp_pivots, int* root_status, lpx_bnb_node_fn on_node, void* user) {
    return lpx_bnb_simplex_batched(1, m, n, sense, A, rel, b, c, opt, flags, found, best_z, best_x, n_nodes,
                                   n_lp_pivots, root_status, on_node, user);
}

}  // extern "C"
