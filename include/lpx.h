/* lpx — C ABI of the B200-native LP/IP solve engine (liblpx.so).
 *
 * Drop-in boundary for the solver seam of Jellyman750/Linear_Programming_Solver_LPR381
 * (R = Linear_Programming_Solver/ in that repository):
 *
 *     interface ILPAlgorithm { SimplexResult Solve(LPProblem, Action<string,bool[,]> updatePivot); }
 *                                                                    R/Models/IPLAlgorithm.cs:5-8
 *
 * The reference has no FFI of its own; a C# shim class per algorithm (see INTEGRATION.md and
 * linear_programming_solver_lpr381_b200/csharp/) flattens LPProblem into the arrays below and
 * P/Invokes these entry points.  Everything here is blittable: plain pointers, ints, doubles.
 * No torch types, no C++ types, no callbacks from device threads.
 *
 * Conventions
 *   sense : 0 = Max, 1 = Min                      (enum Sense, R/Models/PrimalSimplex.cs:8)
 *   rel   : 0 = LE, 1 = GE, 2 = EQ                (enum Rel,   R/Models/PrimalSimplex.cs:9)
 *   A     : row-major m x n (Constraints[i].A[j]), b[m], c[n]
 *   tableau: row-major rows x cols, rows = m' + 1, cols = n + m' + 1 where m' = m + #EQ rows;
 *            the z-row is the LAST row, the RHS the last column (R/Models/PrimalSimplex.cs:179-203)
 *   pivots: (entering column, leaving row) pairs, one per Pivot call
 *   All arithmetic is IEEE binary64 with separate multiply / subtract and true division, in the
 *   reference's evaluation order, so results are bit-identical to the C# loops.
 *
 * Return value of every int function: LPX_OK (0) or a negative LPX_E_* for failures of the call
 * itself (bad arguments, CUDA errors).  Solver outcomes, including the reference's exception
 * cases, are reported per problem in *status.
 *
 * There is NO CPU fallback: without a usable sm_100 device every solve entry point fails with
 * LPX_E_CUDA and lpx_last_error() says why.
 */
#ifndef LPX_H_
#define LPX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes (per problem) ------------------------------------------------------------- */
#define LPX_OPTIMAL            0   /* "OPTIMAL"    R/Models/PrimalSimplex.cs:126 */
#define LPX_UNBOUNDED          1   /* "UNBOUNDED"  R/Models/PrimalSimplex.cs:102-106 */
#define LPX_INFEASIBLE         2   /* "INFEASIBLE" R/Models/DualSimplex.cs:92-96 (dual simplex only) */
#define LPX_RUNNING            3   /* session not finished yet */
#define LPX_S_GE_ROW          -1   /* exception, R/Models/PrimalSimplex.cs:68-71 */
#define LPX_S_NEG_RHS         -2   /* exception, R/Models/PrimalSimplex.cs:73-76 */
#define LPX_S_ITER_LIMIT      -3   /* exception, R/Models/PrimalSimplex.cs:95-96, DualSimplex.cs:39, RevisedPrimalSimplex.cs:144 */
#define LPX_S_REV_UNSUPPORTED -10  /* exception, R/Models/RevisedPrimalSimplex.cs:19-21 (needs all <= rows, b >= -1e-9) */
#define LPX_S_SINGULAR        -11  /* exception, R/Models/RevisedPrimalSimplex.cs:433 "Singular basis encountered." */

/* ---- call-level error codes ----------------------------------------------------------------- */
#define LPX_OK                 0
#define LPX_E_BAD_ARGS        -4
#define LPX_E_CUDA            -5
#define LPX_E_CAPACITY        -8   /* problem too large for the selected kernel / buffer */
#define LPX_E_NCCL            -9

/* ---- options; zero-initialise then lpx_default_options() ------------------------------------ */
typedef struct lpx_options {
    int max_iterations;   /* PrimalSimplex.MaxIterations = 10000 (R/Models/PrimalSimplex.cs:54) */
    int kernel;           /* LPX_KERNEL_*: force a kernel family (tests/benchmarks); 0 = auto */
    int threads;          /* CTA size override for the per-tableau kernels; 0 = auto */
    int knap_spec_nodes;  /* knapsack B&B: heap nodes speculated per round (0 = default 16) */
    int knap_spec_depth;  /* knapsack B&B: look-ahead depth under the front runner (0 = default 2) */
    int stream_protocol;  /* streaming kernels: 0 auto (pipelined blocked look-ahead: the look-ahead of block
                             B+1 overlaps the HBM pass of block B), 1 single-CTA select per pivot, 2 multi-CTA
                             prep per pivot, 3 blocked with a one-CTA look-ahead, 4 blocked, not pipelined.
                             Dual Simplex sessions (lpx_dual_session_open, RHS / ROW re-optimization queries):
                             1 and 2 one pivot per HBM pass; 0, 3 and 4 the blocked dual look-ahead (one CTA
                             decides stream_block pivots, one HBM pass applies them; not pipelined), or one
                             pivot per pass when the look-ahead's shared-memory carve does not fit */
    int reg_variant;      /* register-resident kernel: 0 = default build (4 when n <= 128, else 2), 1 one CTA per SM
                             (all registers), 2 two CTAs per SM (two column slots in shared memory), 3 three CTAs per
                             SM (four slots), 4 condensed tableau (non-basic columns only), three CTAs per SM, 8 row
                             warps x 8 rows (two of four slots in shared memory), 5 the same with 4 row warps x 16
                             rows (one of four slots in shared memory); 4 and 5 need n <= 128 */
    int stream_block;     /* streaming kernels: pivots applied per HBM pass (0 = default, max 16) */
    int stream_pass_variant; /* blocked pass: 0 auto, 1 two doubles per thread, 2 one double per thread,
                                3 TMA-staged (cp.async.bulk + mbarrier pipeline) */
    int knap_ordered_sums; /* knapsack: 1 = always sum in the reference's order, even for exactly summable
                              integer data (which otherwise take the warp-parallel exact path) */
    int knap_shard_tree;   /* knapsack: 1 = ONE search tree evaluated by all ranks of lpx_comm_init: every rank
                              plans and commits identically, evaluates the speculative subtrees it owns
                              (round robin), and the relaxations are merged by an NCCL all-reduce per round */
    int knap_warps;        /* knapsack, warps per instance: 0 auto (2 = a main + helper pair when there are at most four
                              instances per SM, else 1), 1 or 2 to force */
    int reserved[4];
} lpx_options;

#define LPX_KERNEL_AUTO        0
#define LPX_KERNEL_CTA_SMEM    1   /* one CTA per tableau, tableau resident in shared memory */
#define LPX_KERNEL_CTA_GLOBAL  2   /* one CTA per tableau, tableau in global memory (L2/HBM) */
#define LPX_KERNEL_STREAM      3   /* one tableau over the whole GPU, HBM-streamed rank-1 pivots */
#define LPX_KERNEL_CTA_REG     4   /* one CTA per tableau, tableau resident in registers */
#define LPX_KERNEL_CTA_CLUSTER 5   /* one 2- or 4-CTA cluster per tableau, rows split over their shared memories */

void lpx_default_options(lpx_options* opt);

/* ---- library / device ------------------------------------------------------------------------ */
const char* lpx_version(void);
const char* lpx_last_error(void);              /* thread-local, never NULL */
const char* lpx_status_message(int status);    /* the reference's exception text for status < 0 */
int lpx_device_count(void);
int lpx_init(int device);                      /* device < 0: keep the current CUDA device */
void lpx_shutdown(void);
void* lpx_host_alloc(size_t bytes);            /* page-locked host memory for fast H2D/D2H */
void lpx_host_free(void* p);
/* rows/cols of the tableau after EQ expansion (R/Models/PrimalSimplex.cs:161-177). */
int lpx_tableau_dims(int m, int n, const int* rel, int* rows, int* cols);

/* ---- Primal Simplex: PrimalSimplex.Solve, R/Models/PrimalSimplex.cs:57-127 ------------------ */
/* One LP, host buffers.  Any output pointer may be NULL.  history (nullable) receives the
 * tableau after iteration 0..k, at most history_cap tableaux: what AppendTableau prints each
 * iteration (R/Models/PrimalSimplex.cs:88-90,113-114). */
int lpx_primal_solve(int m, int n, int sense, const double* A, const int* rel, const double* b, const double* c,
                     const lpx_options* opt, int* status, int* n_pivots, int* pivots, int pivots_cap, int* basis,
                     double* x, double* z, double* tableau, double* history, int history_cap);

/* `count` LPs of one shape (shared m, n, sense, rel pattern), host buffers, strided per problem:
 * A[count][m][n], b[count][m], c[count][n]; outputs status[count], n_pivots[count],
 * basis[count][m'], x[count][n], z[count], tableau[count][rows][cols] (nullable).
 * Copies are staged and overlapped with the solve; pass lpx_host_alloc memory for full speed. */
int lpx_primal_solve_batched(int count, int m, int n, int sense, const double* A, const int* rel, const double* b,
                             const double* c, const lpx_options* opt, int* status, int* n_pivots, int* basis,
                             double* x, double* z, double* tableau, long long* total_pivots);

/* Same, all pointers are DEVICE pointers (rel too), asynchronous on `stream` (a cudaStream_t;
 * NULL = default stream).  total_pivots is a device pointer to one 64-bit counter (nullable),
 * accumulated with atomicAdd — zero it first. */
int lpx_primal_solve_batched_dev(int count, int m, int n, int sense, const double* A, const int* rel,
                                 const double* b, const double* c, const lpx_options* opt, int* status,
                                 int* n_pivots, int* basis, double* x, double* z, double* tableau,
                                 unsigned long long* total_pivots, void* stream);

/* ---- Dual Simplex: DualSimplex.Solve, R/Models/DualSimplex.cs:15-114 ------------------------ */
/* pivots lists the *silent ForceDualFeasibility pivots first (R/Models/DualSimplex.cs:195-228);
 * history[0] is the tableau after them ("Iteration 0").  opt.kernel AUTO routes as lpx_primal_solve does (per-CTA
 * kernels while the tableau fits shared memory or has at most 96 K elements, else a Dual Simplex session on the whole
 * GPU; with history the per-CTA global-memory kernel); LPX_KERNEL_STREAM forces the session (history: E_CAPACITY). */
int lpx_dual_solve(int m, int n, int sense, const double* A, const int* rel, const double* b, const double* c,
                   const lpx_options* opt, int* status, int* n_pivots, int* silent_pivots, int* pivots,
                   int pivots_cap, int* basis, double* x, double* z, double* tableau, double* history,
                   int history_cap);

/* ---- Large single LP, stepwise (HBM-streamed pivots) ---------------------------------------- */
typedef struct lpx_session lpx_session;
/* Host buffers are copied to the device once; the tableau then lives in HBM for the session. */
lpx_session* lpx_session_open(int m, int n, int sense, const double* A, const int* rel, const double* b,
                              const double* c, const lpx_options* opt);
/* A, b, c are DEVICE pointers (rel stays a host pointer: it only shapes the tableau). */
lpx_session* lpx_session_open_dev(int m, int n, int sense, const double* A, const int* rel, const double* b,
                                  const double* c, const lpx_options* opt);
/* Run at most max_pivots more pivots (stops early at OPTIMAL / UNBOUNDED / ITER_LIMIT).
 * *status = LPX_RUNNING while unfinished.  *pivots_total = pivots performed since open. */
int lpx_session_step(lpx_session* s, int max_pivots, int* status, int* pivots_total);
/* Enqueue max_pivots pivots without waiting (for timing with caller-side CUDA events). */
int lpx_session_step_async(lpx_session* s, int max_pivots);
int lpx_session_sync(lpx_session* s, int* status, int* pivots_total);
void* lpx_session_stream(lpx_session* s);            /* the cudaStream_t the session launches on */
int lpx_session_dims(const lpx_session* s, int* rows, int* cols);
int lpx_session_read_tableau(lpx_session* s, double* tableau);          /* rows x cols, compact */
int lpx_session_read_solution(lpx_session* s, int* basis, double* x, double* z);
int lpx_session_read_pivots(lpx_session* s, int* pivots, int pivots_cap);
void lpx_session_close(lpx_session* s);
/* Dual Simplex (DualSimplex.Solve, R/Models/DualSimplex.cs:15-114) on a large LP whose tableau lives in HBM: the rules
 * of lpx_dual_solve, bit for bit.  Open prepares the rows (PrepareForTableau: Min costs negated; an EQ row as given,
 * then negated; a GE row negated unless -b < -1e-9; an LE row negated when b < -1e-9; no GE / negative-RHS
 * validation), builds the tableau and runs the silent ForceDualFeasibility phase (at most 100 Primal Simplex pivots,
 * ratio margin 1e-12) synchronously.  Silent pivots come first in the pivot log and count in pivots_total; step / sync
 * then run the Dual Simplex loop (OPTIMAL / INFEASIBLE, or LPX_S_ITER_LIMIT after 10000 Dual Simplex pivots,
 * independent of opt.max_iterations).  opt.stream_protocol / stream_block / stream_pass_variant choose the protocol
 * (see lpx_options).  Every other session call works on it; lpx_session_sensitivity returns LPX_E_BAD_ARGS and
 * lpx_session_reoptimize returns NULL for it.  NULL (lpx_last_error() says why) for bad arguments. */
lpx_session* lpx_dual_session_open(int m, int n, int sense, const double* A, const int* rel, const double* b,
                                   const double* c, const lpx_options* opt);
/* A, b, c are DEVICE pointers, rel a host pointer; b is read back once for the row signs. */
lpx_session* lpx_dual_session_open_dev(int m, int n, int sense, const double* A, const int* rel, const double* b,
                                       const double* c, const lpx_options* opt);
/* Silent ForceDualFeasibility pivots of a Dual Simplex session; 0 for every other session. */
int lpx_session_silent_pivots(const lpx_session* s, int* silent);

/* ---- Branch & Bound (simplex): BranchAndBound.Solve, R/Models/Branch&Bound.cs:30-123 -------- */
/* One record per LP relaxation the reference solves (root LP, then every SolveNode call), in the
 * reference's order, delivered from the host thread after the node is committed. */
typedef struct lpx_bnb_node {
    int index;            /* 0 = root LP (R/Models/Branch&Bound.cs:57), 1.. = SolveNode calls */
    int depth;
    int parent;           /* index of the parent record, -1 for the root */
    int is_ceil_child;    /* 1: "x_k >= ceil" child, 0: "x_k <= floor" child / root */
    int id_path_len;      /* hierarchical id, e.g. {2,4} = "Subproblem 2.4" */
    const int* id_path;
    int bound_var;        /* variable of the branching row that created this node, -1 for root */
    int bound_val;        /* its floor / ceil value */
    int algo;             /* 0 Primal Simplex, 1 Dual Simplex (ChooseAlgorithm, :262-266) */
    int lp_status;        /* LPX_OPTIMAL.. / LPX_S_* */
    int outcome;          /* LPX_BNB_* */
    int n_pivots, silent_pivots;
    const int* pivots;    /* n_pivots pairs */
    int rows, cols;       /* node tableau shape */
    double z;
    const double* x;      /* n values (primal nodes) */
    int branch_var, floor_val, ceil_val;   /* valid when outcome == LPX_BNB_BRANCHED */
    int n_history;        /* tableaux available in history (0 unless requested) */
    const double* history;
} lpx_bnb_node;
typedef void (*lpx_bnb_node_fn)(const lpx_bnb_node* node, void* user);

#define LPX_BNB_ERROR       0   /* LP threw (R/Models/Branch&Bound.cs:150-154) */
#define LPX_BNB_INVALID     1   /* "Invalid Simplex result": every Dual Simplex node (:157-161) */
#define LPX_BNB_INFEASIBLE  2   /* IsFeasible failed (:175-179) */
#define LPX_BNB_PRUNED      3   /* z <= best + 1e-6 (:182-186) */
#define LPX_BNB_INCUMBENT   4   /* integral: new incumbent (:189-195) */
#define LPX_BNB_BRANCHED    5
#define LPX_BNB_NOFRAC      6   /* (:215-219) */
#define LPX_BNB_DEPTH       7   /* depth > 200 (:132-136) */

#define LPX_BNB_WANT_HISTORY 1  /* flags: deliver per-iteration tableaux to the node callback */

/* `count` independent IPs of one shape; instance k's records are delivered with user data
 * `user` and node->index local to the instance (on_node receives instance via lpx_bnb_instance()).
 * Outputs: found[count], best_z[count], best_x[count][n], n_nodes[count], n_lp_pivots[count]. */
int lpx_bnb_simplex_batched(int count, int m, int n, int sense, const double* A, const int* rel, const double* b,
                            const double* c, const lpx_options* opt, int flags, int* found, double* best_z,
                            double* best_x, int* n_nodes, long long* n_lp_pivots, int* root_status,
                            lpx_bnb_node_fn on_node, void* user);
int lpx_bnb_simplex(int m, int n, int sense, const double* A, const int* rel, const double* b, const double* c,
                    const lpx_options* opt, int flags, int* found, double* best_z, double* best_x, int* n_nodes,
                    long long* n_lp_pivots, int* root_status, lpx_bnb_node_fn on_node, void* user);
int lpx_bnb_instance(void);  /* inside on_node: which instance of the batch the record belongs to */

/* ---- Mode B: the pooled tree — NOT the reference's tree ------------------------------------------------ */
/* The reference's BranchAndBound never explores a '>=' child (R/Models/Branch&Bound.cs:157-161 rejects every
 * Dual Simplex result), so the tree lpx_bnb_simplex reproduces is one floor path.  lpx_bnb_pooled is the tree
 * the class's doc comment describes (R/Models/Branch&Bound.cs:9-19) with both children honoured: children are
 * warm-started from the parent's final tableau (bound row + Dual Simplex pivots with the reference's rules),
 * each round evaluates the `batch` open nodes with the largest bound, and after lpx_comm_init the nodes of a
 * round are dealt over the ranks (every rank makes the same call and returns the same result; children read
 * their parent's tableau from the owning GPU's memory over NVLink).  All rows must be '<=' with b >= 0.
 * Per evaluated node, in commit order (node 0 = root): id, outcome (LPX_BNB_*), dual pivots, z.
 * Checked against oracle/orc_pooled.cpp node for node and against an independent MILP solver. */
int lpx_bnb_pooled(int m, int n, int sense, const double* A, const int* rel, const double* b, const double* c,
                   const lpx_options* opt, int batch, int* found, double* best_z, double* best_x,
                   long long* n_nodes, long long* n_pivots, long long* n_rounds, long long node_cap, int* node_id,
                   int* node_outcome, int* node_pivots, double* node_z);

/* ---- Branch & Bound Knapsack: BranchAndBoundKnapsack.Solve, R/Models/BranchAndBoundKnapsack.cs:58-407 */
typedef struct lpx_knap_eval {   /* one ComputeRelaxation of the root or of a child (:108,209,269) */
    int pop_index;        /* index of the expanded pop this evaluation belongs to, -1 = root */
    int child;            /* 0: x_k = 0 (left), 1: x_k = 1 (right) */
    int var;              /* original index of the fixed item */
    double bound, weight; /* relaxation profit (== bound) and weight */
    int frac_rank;        /* ratio rank of the fractional item, -1 if none */
    double frac;          /* its fraction */
    int break_rank;       /* first ratio rank not (fully) packed; n if all were */
    int decision;         /* LPX_KN_* */
    const signed char* assigned;  /* n entries: -1 undecided, 0, 1 */
} lpx_knap_eval;
typedef struct lpx_knap_pop {    /* one node taken from the heap and expanded or closed (:120-177) */
    int pop_index;
    int label_len;        /* hierarchical label, e.g. {1,2,1} = "1.2.1"; root = {0} */
    const int* label;
    lpx_knap_eval relax;  /* the recomputed relaxation of the popped node (:127) */
    int closed;           /* 0 expanded; 1 candidate/BEST CANDIDATE; 2 CANDIDATE (not better); 3 INFEASIBLE */
} lpx_knap_pop;
typedef void (*lpx_knap_pop_fn)(const lpx_knap_pop* pop, const lpx_knap_eval* left, const lpx_knap_eval* right,
                                void* user);

#define LPX_KN_ROOT          0
#define LPX_KN_INFEASIBLE    1
#define LPX_KN_CANDIDATE_INT 2   /* integral and feasible: incumbent candidate, not pushed */
#define LPX_KN_PUSHED        3
#define LPX_KN_DROPPED       4   /* bound <= best + 1e-9 */

/* rank_order (nullable, n ints) receives the ratio ordering (original index per rank, :75-79). */
int lpx_bnb_knapsack(int n, const double* profit, const double* weight, double capacity, const lpx_options* opt,
                     int* found, double* best_value, int* best_x, long long* n_evals, long long* n_pops,
                     int* rank_order, lpx_knap_pop_fn on_pop, void* user);
/* `count` independent instances, n items each: profit[count][n], weight[count][n], capacity[count]. */
int lpx_bnb_knapsack_batched(int count, int n, const double* profit, const double* weight, const double* capacity,
                             const lpx_options* opt, int* found, double* best_value, int* best_x,
                             long long* n_evals, long long* n_pops);

/* ---- multi-GPU incumbent sharing (one process per GPU) -------------------------------------- */
/* NCCL is loaded at run time (libnccl.so.2).  Rank 0 creates the id, the host application ships
 * the 128 bytes to every rank (any transport), every rank calls lpx_comm_init. */
int lpx_comm_unique_id(void* id128);
int lpx_comm_init(int world, int rank, const void* id128);
int lpx_comm_allreduce_max(double* values, int count);      /* host values, in place */
int lpx_comm_allgather(const void* send, void* recv, size_t bytes_per_rank);  /* host buffers */
void lpx_comm_destroy(void);
int lpx_comm_world(void);
int lpx_comm_rank(void);

/* ---- Revised Primal Simplex ------------------------------------------------------------------- */
/* RevisedPrimalSimplex.Solve (R/Models/RevisedPrimalSimplex.cs:17-145): price-out with the basis
 * inverse recomputed by Gauss-Jordan (partial pivoting) every iteration, left-to-right dot products,
 * ratio margin 1e-12.  status: LPX_OPTIMAL / LPX_UNBOUNDED / LPX_S_ITER_LIMIT / LPX_S_REV_UNSUPPORTED /
 * LPX_S_SINGULAR.  pivots: 2 ints per iteration (entering column, leaving ROW = basis position),
 * theta: the chosen ratio.  basis (m) = Bidx, nonbasic (n) = Nidx in the reference's list order,
 * xB (m), Binv (m x m, row-major), x (n) = basic decision variables mapped back.
 * history (nullable): history_cap records of lpx_revised_history_stride(m, n) doubles, one per
 * BuildIterationBlock call (:62, :134): [Binv m*m][x_B m][z][r_N n][d m][theta][Bidx m][Nidx n][entering],
 * integers stored as doubles; record 0 is the initial basis (r_N, d, theta unused, entering -1).  On
 * LPX_S_SINGULAR only status, n_iters and the records of the completed iterations are written.
 * opt.kernel: LPX_KERNEL_CTA_GLOBAL one CTA (the work vectors of 20n + 68m + 16 bytes in shared memory, else
 * LPX_E_CAPACITY); LPX_KERNEL_STREAM the whole GPU (blocked Gauss-Jordan inversion with opt.stream_block steps per
 * pass, 0 = 8, and the pass kernel of opt.stream_pass_variant; grid-wide pricing); any other value AUTO: one CTA
 * while the vectors fit and m <= 64, else the whole GPU.  Both give the same bits.  A history the device cannot
 * hold fails the whole-GPU call with LPX_E_CAPACITY and the reason in lpx_last_error(); nothing is written. */
int lpx_revised_solve(int m, int n, int sense, const double* A, const int* rel, const double* b, const double* c,
                      const lpx_options* opt, int* status, int* n_iters, int* pivots, double* theta, int pivots_cap,
                      int* basis, int* nonbasic, double* xB, double* Binv, double* x, double* history,
                      int history_cap);
size_t lpx_revised_history_stride(int m, int n);

/* ---- Sensitivity analysis of an optimal Primal Simplex result — NOT the reference's ---------------------- */
/* The reference's SensitivityAnalysis reads the objective row as tableau row 0, while its PrimalSimplex and this
 * engine put the z-row last, so this report is defined here and checked against oracle/orc_sensitivity.cpp bit for
 * bit and against an independent LP solver.  Input: the final tableau of a Primal Simplex solve with status
 * LPX_OPTIMAL (m' rows after EQ expansion, W = n + m' + 1 columns), its basis, and the model's sense, rel, b, c.
 * EPS = 1e-9.  The slack of constraint i is column n + i1 of its expanded row i1; an EQ row i expands to rows i1
 * (a.x <= b) and i2 = i1 + 1 (-a.x <= -b).  z = T[m'], beta_r = T[r][W-1]; "non-basic" = not listed in basis.
 *   shadow[i]  = T[m'][n+i1]  (EQ: T[m'][n+i1] - T[m'][n+i2]), negated for Min: d(objective as written)/d b_i.
 *                (z itself stays as the solve returns it, the maximum of -c.x for Min.)
 *   slack[i]   = beta_r if slack column n+i1 is basic in row r, else +0.
 *   rhs range  : g = column n+i1 (EQ: column n+i1 minus column n+i2), q_r = beta_r / g_r;
 *                lo = b_i + max{-q_r : g_r > EPS}, hi = b_i + min{-q_r : g_r < -EPS}; an empty side is -inf / +inf.
 *   reduced[j] = T[m'][j] (>= 0 at an optimum for both senses).
 *   cost range : non-basic j: Max (-inf, c_j + d_j], Min [c_j - d_j, +inf).  Basic j in row r, over non-basic
 *                columns k < W-1 with alpha = T[r][k]: dlo = max{-(d_k/alpha) : alpha > EPS},
 *                dhi = min{-(d_k/alpha) : alpha < -EPS}; Max [c_j + dlo, c_j + dhi], Min [c_j - dhi, c_j - dlo].
 * Ties in every max / min: -0.0 equals +0.0 and the lowest row / column index wins (its own value is used).
 * Instances whose status is not LPX_OPTIMAL get a record of NaNs.
 * Scope: results of the Primal Simplex entry points.  GE rows never reach OPTIMAL there; lpx_dual_solve results are
 * excluded, because that solver treats a.x >= b (b > 0) as a.x <= b and its tableau does not describe the model.
 * One record per LP, lpx_sensitivity_stride(m, n) = 4m + 3n doubles:
 *   shadow[m] | slack[m] | rhs_lo[m] | rhs_hi[m] | reduced[n] | cost_lo[n] | cost_hi[n]  */
size_t lpx_sensitivity_stride(int m, int n);
/* From final tableaux already on the device: the outputs of lpx_primal_solve_batched_dev, same pointer
 * conventions (all device pointers, rel included), asynchronous on `stream`.  report: count x stride. */
int lpx_sensitivity_batched_dev(int count, int m, int n, int sense, const int* rel, const double* b, const double* c,
                                const int* status, const int* basis, const double* tableau, double* report, void* stream);
/* Host buffers: lpx_primal_solve_batched plus the reports (count x stride); any output but status and report may
 * be NULL.  The tableaux stay on the device: nothing but status / n_pivots / basis / x / z / report crosses PCIe. */
int lpx_primal_solve_sensitivity_batched(int count, int m, int n, int sense, const double* A, const int* rel,
                                         const double* b, const double* c, const lpx_options* opt, int* status,
                                         int* n_pivots, int* basis, double* x, double* z, double* report,
                                         long long* total_pivots);
/* Large LP whose tableau lives in HBM; report is a host buffer of one stride (NaNs unless the session's status,
 * as of its last step / sync, is LPX_OPTIMAL). */
int lpx_session_sensitivity(lpx_session* s, double* report);

/* ---- Re-optimization of an optimal Primal Simplex result — NOT the reference's ---------------------------- */
/* What-if queries past the sensitivity ranges: change b, change c, add a constraint or add a variable, then re-solve
 * warm from the final tableau of a Primal Simplex solve with status LPX_OPTIMAL, instead of from the slack basis.
 * Checked against oracle/orc_reopt.cpp bit for bit and against an independent LP solver.  Notation as in the
 * sensitivity section: m' rows after EQ expansion, W = n + m' + 1, the slack of constraint i is s1 = n + i1 (an EQ
 * row also has s2 = n + i2), T[m'] is the z-row, the RHS the last column, max-form (Min costs negated as
 * BuildTableau does).  FP64 with separate multiply / add / subtract; a term whose payload coefficient is zero
 * (either sign) is SKIPPED, so an all-zero change returns the base's bits.  One call has one kind; each query has
 * its own payload (lpx_reopt_payload_stride doubles) and names its base.
 *   LPX_REOPT_RHS   payload db[m].  For i ascending with db_i != 0, on every row r (z-row included):
 *                   T[r][W-1] += db_i * T[r][s1]; an EQ row also T[r][W-1] -= db_i * T[r][s2].
 *                   Then Dual Simplex with the reference's rules (most negative RHS < -1e-9 leaves; min z_j / -a over
 *                   a < -1e-9 with the 1e-12 margin scan enters; limit 10000), no silent pivots.  Shape unchanged.
 *   LPX_REOPT_COST  payload dc[n], in the model's sense.  delta_j = dc_j (Max) or -dc_j (Min).  For j ascending with
 *                   dc_j != 0: if j is basic in row r, z[k] += delta_j * T[r][k] for all k < W (RHS included); then
 *                   z[j] -= delta_j.  Then Primal Simplex with the reference's rules (entering below -1e-9, ratio
 *                   margin 1e-9, opt.max_iterations).  Shape unchanged.
 *   LPX_REOPT_ROW   payload a[n], rel (0 LE / 1 GE, stored as a double), beta.  New row m' and new slack column
 *                   n + m': the old RHS position becomes the slack column, the RHS moves right (the layout of the
 *                   pooled tree's bound row).  Raw row: a, +0 in the old slack columns, beta; for GE every entry of it,
 *                   zeros included, is negated.  +1 in the new slack column.  Then for r = 0 .. m'-1 ascending with
 *                   j = basis[r] < n and a_j != 0: row[k] -= a~_j * T[r][k] over the old columns and the RHS (a~ = the
 *                   raw row's a).  The old rows and the z-row get +0 in the new column.  Dual Simplex as for RHS.
 *                   rows + 1, cols + 1; the new slack is basic in the new row.
 *   LPX_REOPT_COL   payload a[m], c_new in the model's sense.  New decision variable at column n: old columns >= n and
 *                   basis entries >= n shift by one.  Its entry starts at +0 in the constraint rows and at -c'_new in
 *                   the z-row (c' = c for Max, -c for Min, as BuildTableau writes it); then on every row, for i
 *                   ascending with a_i != 0: v += a_i * T[r][s1]; an EQ row also v -= a_i * T[r][s2].  Primal Simplex
 *                   as for COST.  cols + 1; x has n + 1 entries.
 * A query whose base is not LPX_OPTIMAL gets the base's status, 0 pivots and zeroed basis / x / z / tableau.
 * Outcomes: RHS / ROW: LPX_OPTIMAL, LPX_INFEASIBLE, LPX_S_ITER_LIMIT; COST / COL: LPX_OPTIMAL, LPX_UNBOUNDED,
 * LPX_S_ITER_LIMIT.  opt.kernel: AUTO (shared-memory tableau when it fits, else global memory), CTA_SMEM
 * (LPX_E_CAPACITY when it does not fit) or CTA_GLOBAL; any other kernel, an unknown kind or a ROW rel other than 0 / 1
 * is LPX_E_BAD_ARGS.  opt.threads is honoured. */
#define LPX_REOPT_RHS  1
#define LPX_REOPT_COST 2
#define LPX_REOPT_ROW  3
#define LPX_REOPT_COL  4
/* doubles per query payload: m (RHS), n (COST), n + 2 (ROW), m + 1 (COL); 0 for an unknown kind */
size_t lpx_reopt_payload_stride(int kind, int m, int n);
/* rows / cols of a query's result tableau (rel: the base model's, host pointer, nullable = all LE) */
int lpx_reopt_dims(int kind, int m, int n, const int* rel, int* rows, int* cols);
/* Device pointers throughout (rel included; the outputs of lpx_primal_solve_batched_dev serve as the bases),
 * asynchronous on `stream`.  base_status / base_basis / base_tableau: the bases, indexed by src[q] (nullable: query q
 * uses base q).  payload: count x stride.  Per query: status, n_pivots (nullable), pivots (nullable, pivots_cap pairs),
 * basis (nullable, rows - 1), x (nullable, n or n + 1 for COL), z (nullable), tableau (nullable, rows x cols as
 * lpx_reopt_dims gives them; must not overlap the bases).  total_pivots: as in lpx_primal_solve_batched_dev. */
int lpx_reoptimize_batched_dev(int kind, int count, int m, int n, int sense, const int* rel, const int* base_status,
                               const int* base_basis, const double* base_tableau, const int* src, const double* payload,
                               const lpx_options* opt, int* status, int* n_pivots, int* pivots, int pivots_cap,
                               int* basis, double* x, double* z, double* tableau, unsigned long long* total_pivots,
                               void* stream);
/* Host buffers: one GPU Primal Simplex solve of the base (A, rel, b, c; opt.max_iterations and opt.threads apply to it,
 * the kernel is chosen automatically) and `count` queries of one kind against its final tableau.  *base_status is
 * the base's status.  Any per-query output may be NULL. */
int lpx_reoptimize(int kind, int m, int n, int sense, const double* A, const int* rel, const double* b, const double* c,
                   const lpx_options* opt, int count, const double* payload, int* base_status, int* status,
                   int* n_pivots, int* pivots, int pivots_cap, int* basis, double* x, double* z, double* tableau);
/* A NEW session holding one what-if query against an optimal base session.  The base is not modified and may be
 * stepped, read or re-queried afterwards; several query sessions of one base may be open at once.  kind / payload
 * (host pointer, lpx_reopt_payload_stride(kind, m, n) doubles, m / n the base model's) are the definition above; the
 * edit is applied to the base's current tableau and basis, and the query's results equal oracle/orc_reopt.cpp on them
 * bit for bit.  RHS / ROW run the Dual Simplex rules (limit 10000) with opt's stream protocol (see lpx_options: the
 * blocked dual look-ahead or one pivot per HBM pass); COST / COL run the Primal Simplex rules with opt's max_iterations
 * and stream protocol, as lpx_session_open does.  opt NULL: the base's options.
 * NULL (lpx_last_error() says why) when the base's status, as of its last step / sync, is not LPX_OPTIMAL, for an
 * unknown kind, a ROW rel other than 0 / 1, or a NULL base / payload.  The query is read with the session calls:
 * step / sync run its loop, pivots count from 0, dims give its shape (ROW: rows + 1; ROW / COL: cols + 1),
 * read_solution's x has n + 1 entries for COL.  lpx_session_sensitivity reports on the modified model (b + db, or
 * c + dc) for RHS / COST queries and returns LPX_E_BAD_ARGS for ROW / COL queries.  Free with lpx_session_close. */
lpx_session* lpx_session_reoptimize(const lpx_session* base, int kind, const double* payload, const lpx_options* opt);

/* ---- Gomory cutting plane: CuttingPlane.Solve, R/Models/CuttingPlane.cs:13-164 ------------------------------ */
/* `count` IPs, one CTA each, all rounds on the device.  A round solves the model plus the cuts so far with Primal
 * Simplex (the rules and bits of lpx_primal_solve, opt.max_iterations), reads x (an UNBOUNDED round's too), finds the
 * first j with 1e-9 < x_j - floor(x_j) < 1 - 1e-9 and, if there is one, appends the cut read from tableau row
 * (x_j's basis position + 1) — the reference's quirk: the row below x_j's, the z-row when x_j is basic in the last
 * constraint row: a_k = f_k when f_k = T[row][k] - floor(T[row][k]) > 1e-9, else +0.0, over the n decision columns;
 * b = rhs - floor(rhs); relation '<='.  The loop ends at an integral x (INTEGER), when Primal Simplex throws
 * (GE row or negative RHS in round 1, the iteration limit in any round: LP_ERROR), or after 50 rounds (INCOMPLETE).
 * A round's tableau is built cold as PrimalSimplex.Solve builds it for the grown model: the base rows (EQ expanded),
 * then the cuts in order, each with +1 in its own slack column, then the z-row.
 *   Shape      one per call: m, n, sense and rel are shared; A[count][m][n], b[count][m], c[count][n] strided per IP.
 *   end        LPX_CUT_*; n_rounds = rounds run (PrimalSimplex calls), n_cuts = n_rounds for INCOMPLETE, else
 *              n_rounds - 1.
 *   Per round  [count][50]: lp_status = LPX_OPTIMAL, LPX_UNBOUNDED or the LPX_S_* of the round that threw; lp_pivots =
 *              pivots of that round (0 for GE / negative RHS, max_iterations for LPX_S_ITER_LIMIT); rounds not run:
 *              LPX_RUNNING and 0.
 *   Per cut    [count][50]: frac_var, cut_row (the tableau row read), cut_a [count][50][n], cut_b; cuts not made: -1,
 *              -1, +0.0, +0.0.
 *   Final LP   only for INTEGER: basis [count][m'+49], x [count][n], z [count], tableau [count][max_rows*max_cols]
 *              hold the last round's LP, the tableau compact (rows = m' + n_cuts + 1, cols = n + m' + n_cuts + 1) at
 *              the start of the slot; every other entry, and all of them for any other end, is zero.
 * Every output except `end` may be NULL.  opt.kernel: AUTO (the tableau in shared memory when the 50-round shape fits,
 * else in global memory), LPX_KERNEL_CTA_SMEM (LPX_E_CAPACITY when it does not fit) or LPX_KERNEL_CTA_GLOBAL; any other
 * value is LPX_E_BAD_ARGS, as are count < 1, m < 1, n < 1, a rel value outside 0..2 or a sense outside 0..1 (checked
 * before any device work).  opt.threads is honoured.  Bit-exact with oracle/orc_cut.cpp (numbers) and oracle/orc_cutting.cpp (text). */
#define LPX_CUT_INTEGER    0   /* all x_j integral: the final LP's outputs are written */
#define LPX_CUT_INCOMPLETE 1   /* 50 rounds, 50 cuts */
#define LPX_CUT_LP_ERROR   2   /* a round's PrimalSimplex threw: its lp_status says which */
#define LPX_CUT_NONBASIC   3   /* kept for the oracle's enum; unreachable for a basic fractional value */
#define LPX_CUT_MAX_ROUNDS 50
/* max_rows = m' + 50, max_cols = n + m' + 50: the output strides (rel: host pointer, nullable = all LE) */
int lpx_cutting_plane_dims(int m, int n, const int* rel, int* max_rows, int* max_cols);
/* Host buffers. */
int lpx_cutting_plane_batched(int count, int m, int n, int sense, const double* A, const int* rel, const double* b,
                              const double* c, const lpx_options* opt, int* end, int* n_rounds, int* n_cuts,
                              int* lp_status, int* lp_pivots, int* frac_var, int* cut_row, double* cut_a, double* cut_b,
                              int* basis, double* x, double* z, double* tableau, long long* total_pivots);
/* Same, all pointers are DEVICE pointers (rel too; it is read back once for the tableau shape and checked then),
 * asynchronous on `stream`.  total_pivots: as in lpx_primal_solve_batched_dev (zero it first).  cut_a / cut_b, when
 * given, are the cut store the rounds read back; without them, and for the global-memory build without a tableau,
 * the library uses scratch of its own. */
int lpx_cutting_plane_batched_dev(int count, int m, int n, int sense, const double* A, const int* rel, const double* b,
                                  const double* c, const lpx_options* opt, int* end, int* n_rounds, int* n_cuts,
                                  int* lp_status, int* lp_pivots, int* frac_var, int* cut_row, double* cut_a,
                                  double* cut_b, int* basis, double* x, double* z, double* tableau,
                                  unsigned long long* total_pivots, void* stream);

/* ---- measurement helpers (bench.py) --------------------------------------------------------- */
/* Unfused FP64 rate (separate DMUL and DADD, the only arithmetic the bit-exactness contract
 * allows) in TFLOP/s: the roofline denominator of the on-chip batched kernels. */
int lpx_measure_fp64_rate(double* tflops);
/* Dependent-chain latencies in SM cycles, one warp alone: cycles8[0..7] = DADD, DMUL, DDIV, REDUX.MIN,
 * SHFL, shared-memory store+load round trip, BAR.SYNC of 13 warps, DSETP+select.  These, not the
 * FP64 rate, bound one pivot of a per-tableau kernel (DESIGN.md 4.1). */
int lpx_measure_latencies(double* cycles8);
/* Session kernels timed separately with CUDA events on the session stream, run back to back
 * (no overlap): us[0] = mean look-ahead / select time, us[1] = mean HBM pass time, us[2] = mean time
 * per block (blocked protocols) or per pivot (per-pivot protocols), over n blocks / pivots. */
int lpx_session_profile(lpx_session* s, int n, double* us);
/* Development aid: phase timestamps (ns, %globaltimer) of one look-ahead step. */
int lpx_session_debug_stamps(lpx_session* s, unsigned long long* out8);

/* Work of this thread's last lpx_bnb_simplex(_batched) call: stats4[0] = floating-point operations of all
 * node LPs (sum of pivots x (2 m_d (n+m_d+1) + (n+m_d+1)), m_d = constraint rows of that node's tableau:
 * SURVEY.md 8d), [1] = seconds inside the GPU evaluation calls (upload, kernels, download, sync),
 * [2] = seconds of the whole search, [3] = evaluation rounds (kernel launch groups). */
int lpx_bnb_last_stats(double* stats4);

/* ---- counters (for benchmarks: "how many of my kernels launched") --------------------------- */
long long lpx_kernel_launches(void);   /* since lpx_init / last reset */
void lpx_reset_counters(void);

#ifdef __cplusplus
}
#endif
#endif /* LPX_H_ */
