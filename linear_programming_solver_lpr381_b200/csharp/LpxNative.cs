// P/Invoke declarations for liblpx.so (include/lpx.h).  Source only: this image has no .NET
// toolchain, so the file is not compiled here; the identical C ABI is exercised by the C++ host
// layer (../host) and by the ctypes harness (../_ffi.py).
using System;
using System.Runtime.InteropServices;

namespace Linear_Programming_Solver.Models
{
    [StructLayout(LayoutKind.Sequential)]
    internal struct LpxOptions
    {
        public int max_iterations, kernel, threads;
        public int knap_spec_nodes, knap_spec_depth, stream_protocol, reg_variant, stream_block, stream_pass_variant;
        public int knap_ordered_sums, knap_shard_tree, knap_warps;
        public int r0, r1, r2, r3;
    }

    [StructLayout(LayoutKind.Sequential)]
    internal struct LpxBnbNode
    {
        public int index, depth, parent, is_ceil_child, id_path_len;
        public IntPtr id_path;
        public int bound_var, bound_val, algo, lp_status, outcome, n_pivots, silent_pivots;
        public IntPtr pivots;
        public int rows, cols;
        public double z;
        public IntPtr x;
        public int branch_var, floor_val, ceil_val, n_history;
        public IntPtr history;
    }

    [UnmanagedFunctionPointer(CallingConvention.Cdecl)]
    internal delegate void LpxBnbNodeFn(ref LpxBnbNode node, IntPtr user);

    // lpx_knap_eval (include/lpx.h): one ComputeRelaxation of a child, or of the popped node itself.
    // Natural C layout: the two doubles after three ints force 4 bytes of padding, likewise before `frac`.
    [StructLayout(LayoutKind.Sequential)]
    internal struct LpxKnapEval
    {
        public int pop_index, child, var;
        public double bound, weight;
        public int frac_rank;
        public double frac;
        public int break_rank, decision;
        public IntPtr assigned;      // n signed bytes: -1 undecided, 0, 1
    }

    // lpx_knap_pop: one node taken from the heap (the embedded relax is an LpxKnapEval by value)
    [StructLayout(LayoutKind.Sequential)]
    internal struct LpxKnapPop
    {
        public int pop_index, label_len;
        public IntPtr label;         // label_len ints, e.g. {1,2,1} = "1.2.1"; root = {0}
        public LpxKnapEval relax;
        public int closed;           // 0 expanded; 1 BEST CANDIDATE; 2 CANDIDATE; 3 INFEASIBLE
    }

    // left / right are null (IntPtr.Zero) for a closed pop
    [UnmanagedFunctionPointer(CallingConvention.Cdecl)]
    internal delegate void LpxKnapPopFn(ref LpxKnapPop pop, IntPtr left, IntPtr right, IntPtr user);

    internal static class LpxNative
    {
        const string Lib = "lpx";   // liblpx.so on Linux

        [DllImport(Lib)] public static extern void lpx_default_options(ref LpxOptions opt);
        [DllImport(Lib)] public static extern IntPtr lpx_last_error();
        [DllImport(Lib)] public static extern IntPtr lpx_status_message(int status);
        [DllImport(Lib)] public static extern int lpx_init(int device);
        [DllImport(Lib)] public static extern int lpx_tableau_dims(int m, int n, int[] rel, out int rows, out int cols);

        [DllImport(Lib)]
        public static extern int lpx_primal_solve(int m, int n, int sense, double[] A, int[] rel, double[] b, double[] c,
            ref LpxOptions opt, out int status, out int n_pivots, int[] pivots, int pivots_cap, int[] basis,
            double[] x, out double z, double[] tableau, double[] history, int history_cap);

        [DllImport(Lib)]
        public static extern int lpx_dual_solve(int m, int n, int sense, double[] A, int[] rel, double[] b, double[] c,
            ref LpxOptions opt, out int status, out int n_pivots, out int silent_pivots, int[] pivots, int pivots_cap,
            int[] basis, double[] x, out double z, double[] tableau, double[] history, int history_cap);

        // RevisedPrimalSimplex (R/Models/RevisedPrimalSimplex.cs:17-145): pivots = (entering column, leaving row)
        // pairs; history = one record per BuildIterationBlock call, lpx_revised_history_stride doubles each
        [DllImport(Lib)]
        public static extern int lpx_revised_solve(int m, int n, int sense, double[] A, int[] rel, double[] b, double[] c,
            ref LpxOptions opt, out int status, out int n_iters, int[] pivots, double[] theta, int pivots_cap,
            int[] basis, int[] nonbasic, double[] xB, double[] Binv, double[] x, double[] history, int history_cap);
        [DllImport(Lib)] public static extern UIntPtr lpx_revised_history_stride(int m, int n);

        // Sensitivity report of optimal Primal Simplex results (include/lpx.h; not the reference's SensitivityAnalysis,
        // which reads the z-row from tableau row 0): lpx_sensitivity_stride doubles per LP,
        // shadow[m] | slack[m] | rhs_lo[m] | rhs_hi[m] | reduced[n] | cost_lo[n] | cost_hi[n], NaNs unless OPTIMAL.
        [DllImport(Lib)] public static extern UIntPtr lpx_sensitivity_stride(int m, int n);
        [DllImport(Lib)]
        public static extern int lpx_sensitivity_batched_dev(int count, int m, int n, int sense, IntPtr rel, IntPtr b,
            IntPtr c, IntPtr status, IntPtr basis, IntPtr tableau, IntPtr report, IntPtr stream);
        [DllImport(Lib)]
        public static extern int lpx_primal_solve_sensitivity_batched(int count, int m, int n, int sense, double[] A,
            int[] rel, double[] b, double[] c, ref LpxOptions opt, int[] status, int[] n_pivots, int[] basis,
            double[] x, double[] z, double[] report, out long total_pivots);
        [DllImport(Lib)] public static extern int lpx_session_sensitivity(IntPtr session, double[] report);

        // Re-optimization of optimal Primal Simplex results (include/lpx.h; not the reference's): what-if queries that
        // change b (kind 1) or c (2), add a constraint (3) or a variable (4), re-solved warm from the final tableau.
        [DllImport(Lib)] public static extern UIntPtr lpx_reopt_payload_stride(int kind, int m, int n);
        [DllImport(Lib)] public static extern int lpx_reopt_dims(int kind, int m, int n, int[] rel, out int rows, out int cols);
        [DllImport(Lib)]
        public static extern int lpx_reoptimize_batched_dev(int kind, int count, int m, int n, int sense, IntPtr rel,
            IntPtr base_status, IntPtr base_basis, IntPtr base_tableau, IntPtr src, IntPtr payload, ref LpxOptions opt,
            IntPtr status, IntPtr n_pivots, IntPtr pivots, int pivots_cap, IntPtr basis, IntPtr x, IntPtr z,
            IntPtr tableau, IntPtr total_pivots, IntPtr stream);
        [DllImport(Lib)]
        public static extern int lpx_reoptimize(int kind, int m, int n, int sense, double[] A, int[] rel, double[] b,
            double[] c, ref LpxOptions opt, int count, double[] payload, out int base_status, int[] status,
            int[] n_pivots, int[] pivots, int pivots_cap, int[] basis, double[] x, double[] z, double[] tableau);
        // One query against an OPTIMAL session: a new session (IntPtr.Zero on refusal); opt IntPtr.Zero = the base's options.
        [DllImport(Lib)]
        public static extern IntPtr lpx_session_reoptimize(IntPtr base_session, int kind, double[] payload, IntPtr opt);

        // Dual Simplex on a large LP in HBM (DualSimplex.Solve as lpx_dual_solve computes it); IntPtr.Zero on refusal.
        [DllImport(Lib)]
        public static extern IntPtr lpx_dual_session_open(int m, int n, int sense, double[] A, int[] rel, double[] b,
            double[] c, ref LpxOptions opt);
        [DllImport(Lib)]
        public static extern IntPtr lpx_dual_session_open_dev(int m, int n, int sense, IntPtr A, int[] rel, IntPtr b,
            IntPtr c, ref LpxOptions opt);
        [DllImport(Lib)] public static extern int lpx_session_silent_pivots(IntPtr session, out int silent);

        // Gomory cutting plane (CuttingPlane.Solve, all rounds on the GPU, one CTA per IP; include/lpx.h).  No
        // ILPAlgorithm shim: the reference's CuttingPlane text prints every round's iteration tableaux, which stay on
        // the host path.  end: 0 integer, 1 incomplete (50 rounds), 2 LP error; any other output may be null.
        public const int LPX_CUT_MAX_ROUNDS = 50;
        [DllImport(Lib)] public static extern int lpx_cutting_plane_dims(int m, int n, int[] rel, out int max_rows, out int max_cols);
        [DllImport(Lib)]
        public static extern int lpx_cutting_plane_batched(int count, int m, int n, int sense, double[] A, int[] rel,
            double[] b, double[] c, ref LpxOptions opt, int[] end, int[] n_rounds, int[] n_cuts, int[] lp_status,
            int[] lp_pivots, int[] frac_var, int[] cut_row, double[] cut_a, double[] cut_b, int[] basis, double[] x,
            double[] z, double[] tableau, out long total_pivots);
        [DllImport(Lib)]
        public static extern int lpx_cutting_plane_batched_dev(int count, int m, int n, int sense, IntPtr A, IntPtr rel,
            IntPtr b, IntPtr c, ref LpxOptions opt, IntPtr end, IntPtr n_rounds, IntPtr n_cuts, IntPtr lp_status,
            IntPtr lp_pivots, IntPtr frac_var, IntPtr cut_row, IntPtr cut_a, IntPtr cut_b, IntPtr basis, IntPtr x,
            IntPtr z, IntPtr tableau, IntPtr total_pivots, IntPtr stream);

        // Parametric analysis (include/lpx.h): z*(theta) along b + theta d or c + theta d from an optimal Primal
        // Simplex result, one CTA per query.  payload per query: d, then theta_max; segment records of
        // lpx_param_segment_stride(n) = 4 + 2n doubles.  Every output except end may be null.
        public const int LPX_PARAM_RHS = 1, LPX_PARAM_COST = 2;
        public const int LPX_PARAM_REACHED = 0, LPX_PARAM_UNBOUNDED = 1, LPX_PARAM_INFEASIBLE = 2,
            LPX_PARAM_SEG_LIMIT = 3, LPX_PARAM_NO_BASE = 4;
        [DllImport(Lib)] public static extern UIntPtr lpx_param_payload_stride(int kind, int m, int n);
        [DllImport(Lib)] public static extern UIntPtr lpx_param_segment_stride(int n);
        [DllImport(Lib)] public static extern int lpx_parametric_dims(int kind, int m, int n, int[] rel, out int rows, out int cols);
        [DllImport(Lib)]
        public static extern int lpx_parametric(int kind, int m, int n, int sense, double[] A, int[] rel, double[] b,
            double[] c, ref LpxOptions opt, int count, double[] payload, int seg_cap, out int base_status, int[] end,
            int[] n_segments, int[] n_pivots, double[] segments, int[] seg_pivots, int[] basis, double[] tableau);
        [DllImport(Lib)]
        public static extern int lpx_parametric_batched_dev(int kind, int count, int m, int n, int sense, IntPtr rel,
            IntPtr base_status, IntPtr base_basis, IntPtr base_tableau, IntPtr src, IntPtr payload, int seg_cap,
            ref LpxOptions opt, IntPtr end, IntPtr n_segments, IntPtr n_pivots, IntPtr segments, IntPtr seg_pivots,
            IntPtr basis, IntPtr tableau, IntPtr total_pivots, IntPtr stream);

        // Two-phase Simplex (include/lpx.h; not the reference's): '>=' rows, '=' rows and negative right-hand sides,
        // one CTA per LP.  Output tableau (m + 1) x (n + s + 1), s = non-'=' rows; pivots past the last are (-1, -1).
        // Every output except status may be null.
        [DllImport(Lib)] public static extern int lpx_two_phase_dims(int m, int n, int[] rel, out int rows, out int cols);
        [DllImport(Lib)]
        public static extern int lpx_two_phase_solve_batched(int count, int m, int n, int sense, double[] A, int[] rel,
            double[] b, double[] c, ref LpxOptions opt, int[] status, int[] phase1_pivots, int[] n_pivots, int[] pivots,
            int pivots_cap, int[] basis, double[] x, double[] z, double[] tableau, out long total_pivots);
        [DllImport(Lib)]
        public static extern int lpx_two_phase_solve_batched_dev(int count, int m, int n, int sense, IntPtr A,
            IntPtr rel, IntPtr b, IntPtr c, ref LpxOptions opt, IntPtr status, IntPtr phase1_pivots, IntPtr n_pivots,
            IntPtr pivots, int pivots_cap, IntPtr basis, IntPtr x, IntPtr z, IntPtr tableau, IntPtr total_pivots,
            IntPtr stream);
        // Two-phase session: one LP whose two-phase tableau lives in HBM, stepped with the lpx_session_* calls.
        [DllImport(Lib)]
        public static extern IntPtr lpx_two_phase_session_open(int m, int n, int sense, double[] A, int[] rel,
            double[] b, double[] c, ref LpxOptions opt);
        [DllImport(Lib)]
        public static extern IntPtr lpx_two_phase_session_open_dev(int m, int n, int sense, IntPtr A, int[] rel,
            IntPtr b, IntPtr c, ref LpxOptions opt);
        [DllImport(Lib)]
        public static extern int lpx_session_two_phase_info(IntPtr s, out int phase, out int phase1_pivots);
        // Sensitivity of two-phase results (include/lpx.h; not the reference's): lpx_sensitivity_stride doubles per
        // LP, NaNs unless OPTIMAL.  Every output except status and report may be null.
        [DllImport(Lib)]
        public static extern int lpx_two_phase_solve_sensitivity_batched(int count, int m, int n, int sense,
            double[] A, int[] rel, double[] b, double[] c, ref LpxOptions opt, int[] status, int[] phase1_pivots,
            int[] n_pivots, int[] basis, double[] x, double[] z, double[] report, out long total_pivots);
        [DllImport(Lib)]
        public static extern int lpx_two_phase_solve_sensitivity_batched_dev(int count, int m, int n, int sense,
            IntPtr A, IntPtr rel, IntPtr b, IntPtr c, ref LpxOptions opt, IntPtr status, IntPtr phase1_pivots,
            IntPtr n_pivots, IntPtr basis, IntPtr x, IntPtr z, IntPtr report, IntPtr total_pivots, IntPtr stream);
        [DllImport(Lib)] public static extern int lpx_session_two_phase_sensitivity(IntPtr s, double[] report);
        // One query against an OPTIMAL session, on the whole GPU (host buffers, synchronous; the base is only read);
        // opt IntPtr.Zero = the base's options (stream_block: breakpoints per HBM pass).  Any output but end may be null.
        [DllImport(Lib)]
        public static extern int lpx_session_parametric(IntPtr base_session, int kind, double[] payload, int seg_cap,
            IntPtr opt, out int end, out int n_segments, out int n_pivots, double[] segments, int[] seg_pivots,
            int[] basis, double[] tableau);

        [DllImport(Lib)]
        public static extern int lpx_primal_solve_batched(int count, int m, int n, int sense, double[] A, int[] rel,
            double[] b, double[] c, ref LpxOptions opt, int[] status, int[] n_pivots, int[] basis, double[] x,
            double[] z, double[] tableau, out long total_pivots);

        [DllImport(Lib)]
        public static extern int lpx_bnb_simplex(int m, int n, int sense, double[] A, int[] rel, double[] b, double[] c,
            ref LpxOptions opt, int flags, out int found, out double best_z, double[] best_x, out int n_nodes,
            out long n_lp_pivots, out int root_status, LpxBnbNodeFn on_node, IntPtr user);

        [DllImport(Lib)]
        public static extern int lpx_bnb_knapsack(int n, double[] profit, double[] weight, double capacity,
            ref LpxOptions opt, out int found, out double best_value, int[] best_x, out long n_evals, out long n_pops,
            int[] rank_order, LpxKnapPopFn on_pop, IntPtr user);

        public static string LastError() => Marshal.PtrToStringUTF8(lpx_last_error()) ?? "";
        public static string StatusMessage(int s) => Marshal.PtrToStringUTF8(lpx_status_message(s)) ?? "";
    }
}
