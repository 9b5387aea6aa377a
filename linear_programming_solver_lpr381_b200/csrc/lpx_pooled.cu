// lpx_pooled.cu — Mode B, the "pooled tree": Branch & Bound over simplex relaxations with BOTH children
// honoured, warm-started from the parent's tableau, open nodes dealt over the GPUs of one box.
//
// NOT what the reference computes.  Its BranchAndBound sends every '>=' child to Dual Simplex and then
// rejects the result (SURVEY.md F5), so its tree is one floor path; lpx_bnb_simplex reproduces that
// bit for bit.  This file is the tree its doc comment describes (R/Models/Branch&Bound.cs:9-19:
// fractional part closest to 0.5, lowest subscript on ties, ceil branch first) and BASELINE.json's
// north_star asks for: a GPU node pool, relaxations warm-started from the parent's tableau, nodes
// sharded over the ranks, the incumbent shared every batch.  Its checker is oracle/orc_pooled.cpp
// (same search, same arithmetic, node for node) and an independent MILP solver for the optimum.
//
// The search (identical for any number of ranks):
//   root   Primal Simplex with the reference's rules; the final tableau stays in the node pool.
//   child  parent's final tableau + one row (x_k <= floor | x_k >= ceil, written in the parent's
//          non-basic variables) + one slack column, then the reference's Dual Simplex pivots
//          (R/Models/DualSimplex.cs:45-113): cta_simplex_kernel's warm path (lpx_cta.cuh).
//   round  the <= `batch` open nodes with the largest bound (parent's z, lower id on ties) that can
//          still beat the incumbent are evaluated, then committed in that order: infeasible |
//          z <= best + 1e-6 pruned | integral -> incumbent (z, x rounded) | branched (ceil child, then
//          floor child).
//
// Multi-GPU (one process per GPU, lpx_comm_init): every rank runs the same deterministic control
// loop — selection, commit, even every rank's pool allocator — so nothing about the tree is ever
// negotiated.  Node j of a round is evaluated by rank j mod world.  A node's final tableau stays in
// the pool of the rank that solved it; a child solved elsewhere reads its parent's tableau straight
// out of that rank's memory (CUDA IPC mapping, loads over NVLink inside the solve kernel) — no
// staging copy, no collective on the data path.  The exchange step of a round is one device-side
// NCCL all-gather of the small result records (status, pivots, flags, branching variable, z, x), from
// which every rank commits identically: the incumbent is global by construction.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <deque>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <queue>
#include <vector>

#include "lpx_cta.cuh"
#include "lpx_runtime.hpp"

namespace lpx {
namespace {

const double PL_EPS = 1e-6;  // BranchAndBound.EPS (Branch&Bound.cs:24)

struct PNode {
    int id = 0, parent = -1, var = -1, side = 0, bound_val = 0, depth = 0;
    double bound = 0;   // the parent's z
    int owner = 0;      // rank whose pool holds the final tableau
    long long slot = -1;  // byte offset of its slot in that pool
    int cls = 0;        // size class of the slot
    int rows = 0;       // rows of the final tableau
    int open_children = 0;
};

struct OpenRef {  // entry of the open-node queue: 16 bytes, no pointer chasing in the heap's compares
    double bound;
    int id;
};
struct ByBound {
    bool operator()(const OpenRef& a, const OpenRef& b) const {
        if (a.bound != b.bound) return a.bound < b.bound;
        return a.id > b.id;
    }
};

// One rank's node pool as EVERY rank simulates it (so that slot addresses never need to be communicated): a
// bump allocator with one free list per size class.  A node of `rows` tableau rows takes a slot of its class
// (rows rounded up to a multiple of 8): shallow nodes, the vast majority, cost a third of the deepest ones.
struct Pool {
    std::vector<std::vector<long long>> free_by_class;
    long long bump = 0, cap = 0;
    long long alloc(int cls, long long bytes) {
        if ((int)free_by_class.size() <= cls) free_by_class.resize(cls + 1);
        if (!free_by_class[cls].empty()) {
            const long long off = free_by_class[cls].back();
            free_by_class[cls].pop_back();
            return off;
        }
        if (bump + bytes > cap) return -1;
        const long long off = bump;
        bump += bytes;
        return off;
    }
    void release(int cls, long long off) { free_by_class[cls].push_back(off); }
};

// Pools stay allocated (and mapped into the peers) between calls: cudaMalloc / IPC open of gigabytes per call
// would cost more than a search.
struct PoolCache {
    unsigned char* base = nullptr;
    size_t bytes = 0;
    int world = 1;
    std::vector<unsigned char*> peer;  // per rank: base address of its pool in THIS process
} g_pool;

void release_pool() {
    for (size_t r = 0; r < g_pool.peer.size(); r++)
        if (g_pool.peer[r] && g_pool.peer[r] != g_pool.base) cudaIpcCloseMemHandle(g_pool.peer[r]);
    if (g_pool.base) cudaFree(g_pool.base);
    g_pool = PoolCache();
}

}  // namespace

void pooled_release_cache() { release_pool(); }

}  // namespace lpx

using namespace lpx;

extern "C" int lpx_bnb_pooled(int m, int n, int sense, const double* A, const int* rel, const double* b, const double* c,
                              const lpx_options* opt, int batch, int* found, double* best_z, double* best_x,
                              long long* n_nodes, long long* n_pivots, long long* n_rounds, long long node_cap,
                              int* node_id, int* node_outcome, int* node_pivots, double* node_z) {
    if (m < 1 || n < 1 || !A || !b || !c || (sense != 0 && sense != 1) || batch < 1) {
        set_error("lpx_bnb_pooled: bad arguments");
        return LPX_E_BAD_ARGS;
    }
    for (int i = 0; i < m; i++)
        if ((rel && rel[i] != 0) || b[i] < -1e-9) {
            set_error("lpx_bnb_pooled: all rows must be '<=' with a non-negative right-hand side");
            return LPX_E_BAD_ARGS;
        }
    int rc = ensure_device();
    if (rc != LPX_OK) return rc;
    Runtime& r = rt();
    std::lock_guard<std::recursive_mutex> lk(r.mu);
    lpx_options o;
    lpx_default_options(&o);
    if (opt) o = *opt;
    cudaStream_t s = r.stream;
    const int world = comm_world(), rank = comm_rank();

    // ---- node pool: slots of (tableau | basis), one size class per 8 tableau rows ------------------------------
    const int max_extra = 248;  // bound rows below the root a node may carry (the kernels' limit, not memory's)
    const int max_rows = m + max_extra + 1;
    auto class_of = [&](int rows) { return (rows - (m + 1) + 7) / 8; };
    auto class_rows = [&](int cls) { return m + 1 + 8 * cls; };
    auto class_tbytes = [&](int cls) { return (size_t)class_rows(cls) * (n + class_rows(cls)) * 8; };
    auto class_bytes = [&](int cls) { return (long long)((class_tbytes(cls) + (size_t)class_rows(cls) * 4 + 255) & ~(size_t)255); };
    if (g_pool.world != world || !g_pool.base) {
        release_pool();
        size_t free_b = 0, total_b = 0;
        LPX_CUDA(cudaMemGetInfo(&free_b, &total_b));
        // every branched node keeps its tableau until both children are solved: a hard instance has tens of
        // thousands of them alive at once (untouched memory costs nothing but address space)
        size_t budget = std::min(free_b / 2, (size_t)64 << 30);
        if (world > 1) {  // every rank simulates every allocator: all pools have the smallest rank's size
            std::vector<unsigned long long> all(world);
            unsigned long long mine_b = budget;
            if ((rc = lpx_comm_allgather(&mine_b, all.data(), sizeof mine_b)) != LPX_OK) return rc;
            for (int q = 0; q < world; q++) budget = std::min<size_t>(budget, all[q]);
        }
        LPX_CUDA(cudaMalloc((void**)&g_pool.base, budget));
        g_pool.bytes = budget;
        g_pool.world = world;
        g_pool.peer.assign(world, nullptr);
        g_pool.peer[rank] = g_pool.base;
        if (world > 1) {
            // every rank maps every other rank's pool: children read their parent's tableau over NVLink
            cudaIpcMemHandle_t mine;
            LPX_CUDA(cudaIpcGetMemHandle(&mine, g_pool.base));
            std::vector<cudaIpcMemHandle_t> all(world);
            if ((rc = lpx_comm_allgather(&mine, all.data(), sizeof mine)) != LPX_OK) return rc;
            for (int q = 0; q < world; q++) {
                if (q == rank) continue;
                void* p = nullptr;
                LPX_CUDA(cudaIpcOpenMemHandle(&p, all[q], cudaIpcMemLazyEnablePeerAccess));
                g_pool.peer[q] = (unsigned char*)p;
            }
        }
    }
    auto slot_T = [&](int owner, long long off) { return (double*)(g_pool.peer[owner] + off); };
    auto slot_basis = [&](int owner, long long off, int cls) { return (int*)(g_pool.peer[owner] + off + class_tbytes(cls)); };

    // ---- base problem on the device ----------------------------------------------------------------------
    double* dA = ws_dev_as<double>(WS_A, (size_t)m * n);
    double* db = ws_dev_as<double>(WS_B, m);
    double* dc = ws_dev_as<double>(WS_C, n);
    if (!dA || !db || !dc) return LPX_E_CUDA;
    LPX_CUDA(cudaMemcpyAsync(dA, A, (size_t)m * n * 8, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemcpyAsync(db, b, (size_t)m * 8, cudaMemcpyHostToDevice, s));
    LPX_CUDA(cudaMemcpyAsync(dc, c, (size_t)n * 8, cudaMemcpyHostToDevice, s));

    // result record of one node: 4 ints (status, pivots, flags, branching variable), z, x[n]
    const size_t rec_bytes = 16 + 8 + (size_t)n * 8;
    const int per_rank_max = (batch + world - 1) / world;
    unsigned char* d_own = (unsigned char*)ws_dev(WS_PL_OUT, (size_t)per_rank_max * rec_bytes + 64);
    unsigned char* d_all = (unsigned char*)ws_dev(WS_PL_ALL, (size_t)per_rank_max * rec_bytes * world + 64);
    unsigned char* h_all = (unsigned char*)ws_pin(WS_PL_ALL, (size_t)per_rank_max * rec_bytes * world + 64);
    WarmNode* h_warm = (WarmNode*)ws_pin(WS_PL_IN, (size_t)per_rank_max * sizeof(WarmNode) + 64);
    WarmNode* d_warm = (WarmNode*)ws_dev(WS_PL_IN, (size_t)per_rank_max * sizeof(WarmNode) + 64);
    // the kernels write status / pivots / flags / branch / z / x into separate arrays; a small pack kernel would
    // be one more launch, so the record layout is "structure of arrays" per rank instead:
    //   [status per_rank_max][pivots ..][flags ..][branch ..] ints, then z doubles, then x rows
    if (!d_own || !d_all || !h_all || !h_warm || !d_warm) return LPX_E_CUDA;
    const size_t ints_bytes = (size_t)per_rank_max * 16;
    auto own_int = [&](unsigned char* base, int which) { return (int*)(base + (size_t)which * per_rank_max * 4); };
    auto own_z = [&](unsigned char* base) { return (double*)(base + ints_bytes); };
    auto own_x = [&](unsigned char* base) { return (double*)(base + ints_bytes + (size_t)per_rank_max * 8); };
    const size_t rank_bytes = (size_t)per_rank_max * rec_bytes;

    auto base_batch = [&](CtaBatch& B) {
        std::memset(&B, 0, sizeof B);
        B.A = dA;
        B.b = db;
        B.c = dc;
        B.m_in = m;
        B.n = n;
        B.sense = sense;
        B.m_base = m;
        B.max_iter = o.max_iterations;
        B.scratch = (double*)g_pool.base;  // never used: warm nodes and the root work in their pool slots
        B.scratch_stride = 0;
    };

    std::deque<PNode> nodes;  // stable addresses, chunked allocation: no malloc per node
    std::vector<Pool> pools(world);
    std::priority_queue<OpenRef, std::vector<OpenRef>, ByBound> open;
    double best = -std::numeric_limits<double>::infinity();
    bool have_best = false;
    std::vector<double> bx(n, 0.0);
    long long evaluated = 0, pivots = 0, rounds = 0;

    auto release_parent = [&](int id) {
        if (id < 0) return;
        PNode& p = nodes[id];
        if (--p.open_children == 0 && p.slot >= 0 && p.parent >= 0) {  // the root keeps slot 0 of every pool
            pools[p.owner].release(p.cls, p.slot);
            p.slot = -1;
        }
    };
    // one SolveNode-like commit from a result record (status, pivots, flags, branch, z, x)
    auto commit = [&](PNode& nd, int status, int npiv, int flags, int branch, double z, const double* x) {
        int outcome;
        pivots += npiv;
        if (status != LPX_OPTIMAL) outcome = LPX_BNB_INFEASIBLE;
        else if (z <= best + PL_EPS) outcome = LPX_BNB_PRUNED;
        else if (flags & 2) {
            outcome = LPX_BNB_INCUMBENT;
            best = z;
            have_best = true;
            for (int j = 0; j < n; j++) bx[j] = std::nearbyint(x[j]);
        } else if (branch < 0) outcome = LPX_BNB_NOFRAC;
        else {
            outcome = LPX_BNB_BRANCHED;
            const int nd_id = nd.id, nd_depth = nd.depth;
            nd.open_children = 2;
            for (int side = 1; side >= 0; side--) {  // ceil child first
                PNode ch;
                ch.id = (int)nodes.size();
                ch.parent = nd_id;
                ch.var = branch;
                ch.side = side;
                ch.bound_val = (int)(side ? std::ceil(x[branch]) : std::floor(x[branch]));
                ch.depth = nd_depth + 1;
                ch.bound = z;
                open.push(OpenRef{z, ch.id});
                nodes.push_back(ch);  // (a deque never moves existing elements: `nd` stays valid)
            }
        }
        if (evaluated < node_cap) {
            if (node_id) node_id[evaluated] = nd.id;
            if (node_outcome) node_outcome[evaluated] = outcome;
            if (node_pivots) node_pivots[evaluated] = npiv;
            if (node_z) node_z[evaluated] = status == LPX_OPTIMAL ? z : 0.0;
        }
        evaluated++;
        if (outcome != LPX_BNB_BRANCHED && nd.slot >= 0 && nd.parent >= 0) {  // nobody will read this tableau
            pools[nd.owner].release(nd.cls, nd.slot);
            nd.slot = -1;
        }
    };

    // ---- root: every rank solves it into slot 0 of its own pool (replicated, deterministic) ----------------
    {
        nodes.emplace_back();
        PNode* root = &nodes[0];
        root->bound = std::numeric_limits<double>::infinity();
        root->rows = m + 1;
        for (int q = 0; q < world; q++) {
            pools[q].cap = (long long)g_pool.bytes;
            pools[q].alloc(0, class_bytes(0));  // offset 0 everywhere
        }
        root->owner = rank;  // each rank reads its own copy
        root->slot = 0;
        root->cls = 0;
        CtaBatch B;
        base_batch(B);
        B.max_rows = m + 1;
        B.max_width = n + m + 1;
        B.status = own_int(d_own, 0);
        B.n_pivots = own_int(d_own, 1);
        B.node_flags = own_int(d_own, 2);
        B.node_branch = own_int(d_own, 3);
        B.z = own_z(d_own);
        B.x = own_x(d_own);
        B.tableau = slot_T(rank, 0);
        B.tableau_stride = 0;
        B.basis = slot_basis(rank, 0, 0);
        B.basis_stride = 0;
        rc = cta_launch(B, 1, cta_fits_smem(B.max_rows, B.max_width) ? LPX_KERNEL_CTA_SMEM : LPX_KERNEL_CTA_GLOBAL, o.threads,
                        s, nullptr);
        if (rc != LPX_OK) return rc;
        LPX_CUDA(cudaMemcpyAsync(h_all, d_own, rank_bytes, cudaMemcpyDeviceToHost, s));
        LPX_CUDA(cudaStreamSynchronize(s));
        const int st = own_int(h_all, 0)[0];
        if (st == LPX_UNBOUNDED || st < 0) {
            // the relaxation is unbounded or threw: no tree (the caller sees found = 0 and one node)
            commit(nodes[0], LPX_INFEASIBLE, own_int(h_all, 1)[0], 0, -1, 0.0, own_x(h_all));
        } else {
            commit(nodes[0], st, own_int(h_all, 1)[0], own_int(h_all, 2)[0], own_int(h_all, 3)[0], own_z(h_all)[0],
                   own_x(h_all));
        }
        // the root is "owned" by everybody: children anywhere read their local copy
    }

    std::vector<PNode*> sel;
    long long rounds_big = 0, nodes_big = 0;
    int deepest_rows = 0;
    double tr[3] = {0, 0, 0};  // LPX_POOLED_TRACE=1: seconds selecting + staging | launch .. results on the host | committing
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto secs = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
        return std::chrono::duration<double>(b - a).count();
    };
    while (!open.empty()) {
        const auto t0 = now();
        sel.clear();
        while (!open.empty() && (int)sel.size() < batch) {
            const OpenRef top = open.top();
            open.pop();
            PNode* nd = &nodes[top.id];
            if (top.bound <= best + PL_EPS) {  // cannot beat the incumbent any more: no LP
                release_parent(nd->parent);
                continue;
            }
            sel.push_back(nd);
        }
        if (sel.empty()) break;
        rounds++;
        const int nsel = (int)sel.size();
        // deal the round: node j -> rank j mod world, position j / world; every rank advances every allocator
        int mine = 0, my_max_rows = 0;
        bool any_big = false;
        for (int j = 0; j < nsel; j++) {
            PNode* nd = sel[j];
            const PNode& par = nodes[nd->parent];
            nd->owner = j % world;
            nd->rows = par.rows + 1;
            if (nd->rows > max_rows) {
                set_error("lpx_bnb_pooled: tree deeper than 248 bound rows");
                return LPX_E_CAPACITY;
            }
            nd->cls = class_of(nd->rows);
            nd->slot = pools[nd->owner].alloc(nd->cls, class_bytes(nd->cls));
            if (nd->slot < 0) {
                set_error("lpx_bnb_pooled: node pool exhausted (every open node keeps its parent's tableau)");
                return LPX_E_CAPACITY;
            }
            if (nd->owner != rank) continue;
            WarmNode& w = h_warm[mine++];
            const int powner = par.parent < 0 ? rank : par.owner;  // the root lives in everybody's slot 0
            w.T = slot_T(powner, par.slot);
            w.basis = slot_basis(powner, par.slot, par.cls);
            w.out_T = slot_T(rank, nd->slot);
            w.out_basis = slot_basis(rank, nd->slot, nd->cls);
            w.val = (double)nd->bound_val;
            w.rows = par.rows;
            w.var = nd->var;
            w.side = nd->side;
            w.kind = WARM_BOUND;
            w.base_status = LPX_OPTIMAL;
            my_max_rows = std::max(my_max_rows, nd->rows);
            any_big = any_big || !cta_fits_smem(nd->rows, n + nd->rows);
        }
        if (any_big) {
            rounds_big++;
            nodes_big += mine;
        }
        deepest_rows = std::max(deepest_rows, my_max_rows);
        const auto t1 = now();
        if (mine > 0) {
            LPX_CUDA(cudaMemcpyAsync(d_warm, h_warm, (size_t)mine * sizeof(WarmNode), cudaMemcpyHostToDevice, s));
            CtaBatch B;
            base_batch(B);
            B.warm = d_warm;
            B.max_rows = my_max_rows;
            B.max_width = n + my_max_rows;
            B.status = own_int(d_own, 0);
            B.n_pivots = own_int(d_own, 1);
            B.node_flags = own_int(d_own, 2);
            B.node_branch = own_int(d_own, 3);
            B.z = own_z(d_own);
            B.x = own_x(d_own);
            // nodes that outgrow one SM's shared memory work directly in their pool slot (global memory)
            rc = cta_launch(B, mine, any_big ? LPX_KERNEL_CTA_GLOBAL : LPX_KERNEL_CTA_SMEM, o.threads, s, nullptr);
            if (rc != LPX_OK) return rc;
        }
        // the exchange step: everybody's result records, in rank order
        if ((rc = comm_allgather_dev(d_own, d_all, rank_bytes, s)) != LPX_OK) return rc;
        LPX_CUDA(cudaMemcpyAsync(h_all, d_all, rank_bytes * world, cudaMemcpyDeviceToHost, s));
        LPX_CUDA(cudaStreamSynchronize(s));
        const auto t2 = now();
        for (int j = 0; j < nsel; j++) {
            PNode* nd = sel[j];
            unsigned char* rb = h_all + (size_t)(j % world) * rank_bytes;
            const int q = j / world;
            commit(*nd, own_int(rb, 0)[q], own_int(rb, 1)[q], own_int(rb, 2)[q], own_int(rb, 3)[q], own_z(rb)[q],
                   own_x(rb) + (size_t)q * n);
            release_parent(nd->parent);
        }
        tr[0] += secs(t0, t1);
        tr[1] += secs(t1, t2);
        tr[2] += secs(t2, now());
    }
    if (getenv("LPX_POOLED_TRACE"))
        fprintf(stderr, "[pooled trace] rank %d of %d: %lld rounds, %lld nodes: select + stage %.3f s, launch .. results on the host "
                        "%.3f s, commit %.3f s; %lld rounds (%lld of this rank's nodes) on the global-memory kernel, deepest node %d rows\n", rank, world, rounds, evaluated, tr[0], tr[1], tr[2], rounds_big, nodes_big, deepest_rows);
    if (found) *found = have_best ? 1 : 0;
    if (best_z) *best_z = best;
    if (best_x && have_best)
        for (int j = 0; j < n; j++) best_x[j] = bx[j];
    if (n_nodes) *n_nodes = evaluated;
    if (n_pivots) *n_pivots = pivots;
    if (n_rounds) *n_rounds = rounds;
    return LPX_OK;
}
