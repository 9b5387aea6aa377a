// Drop-in ILPAlgorithm for "Revised Primal Simplex": same contract as RevisedPrimalSimplex.Solve
// (Models/RevisedPrimalSimplex.cs:17-145), arithmetic on the GPU through liblpx.so (lpx_revised_solve).
// It reuses the reference's own printing code, which must be made `internal static`
// (BuildIterationBlock, BuildFinalSummary); LPSolver.cs then maps "revised primal simplex" /
// "revised primal" to this class, and CuttingPlaneRevised.cs:16 constructs it instead of the CPU solver.
// Default options: a small model runs on one CTA, a large one (m past the crossover, or work vectors past shared
// memory) on the whole GPU, with the same results (include/lpx.h).
// Source only (no .NET toolchain in this image); host/revised_host.cpp is the compiled twin.
using System;
using System.Collections.Generic;
using System.Linq;

namespace Linear_Programming_Solver.Models
{
    internal class GpuRevisedPrimalSimplex : ILPAlgorithm
    {
        public SimplexResult Solve(LPProblem original, Action<string, bool[,]> updatePivot = null)
        {
            int m = original.Constraints.Count, n = original.NumVars;
            var A = new double[m * n];
            var rel = new int[m];
            var b = new double[m];
            for (int i = 0; i < m; i++)
            {
                Array.Copy(original.Constraints[i].A, 0, A, i * n, n);
                rel[i] = (int)original.Constraints[i].Relation;
                b[i] = original.Constraints[i].B;
            }
            var opt = new LpxOptions();
            LpxNative.lpx_default_options(ref opt);
            var basis = new int[m];
            var nonbasic = new int[n];
            var xB = new double[m];
            var x = new double[n];
            // first pass: status and iteration count; second pass: one record per BuildIterationBlock call
            int rc = LpxNative.lpx_revised_solve(m, n, (int)original.ObjectiveSense, A, rel, b, original.C, ref opt,
                out int status, out int iters, null, null, 0, basis, nonbasic, xB, null, x, null, 0);
            if (rc != 0) throw new Exception(LpxNative.LastError());
            if (status == -10) throw new Exception(LpxNative.StatusMessage(status));   // unsupported model, same text
            var names = Enumerable.Range(0, n).Select(j => $"x{j + 1}")
                .Concat(Enumerable.Range(0, m).Select(j => $"c{j + 1}")).ToArray();
            if (updatePivot != null && (status >= 0 || status == -3))
            {
                int stride = (int)LpxNative.lpx_revised_history_stride(m, n);
                var hist = new double[(long)stride * (iters + 1)];
                rc = LpxNative.lpx_revised_solve(m, n, (int)original.ObjectiveSense, A, rel, b, original.C, ref opt,
                    out status, out iters, null, null, 0, basis, nonbasic, xB, null, x, hist, iters + 1);
                if (rc != 0) throw new Exception(LpxNative.LastError());
                for (int k = 0; k <= iters; k++)
                {
                    // record layout (include/lpx.h): [Binv m*m][x_B m][z][r_N n][d m][theta][Bidx m][Nidx n][entering]
                    int o = k * stride;
                    var Binv = new double[m, m];
                    Buffer.BlockCopy(hist, o * 8, Binv, 0, m * m * 8);
                    o += m * m;
                    var xBk = hist.Skip(o).Take(m).ToArray(); o += m;
                    double z = hist[o++];
                    var rN = hist.Skip(o).Take(n).ToArray(); o += n;
                    var d = hist.Skip(o).Take(m).ToArray(); o += m;
                    double theta = hist[o++];
                    var Bidx = hist.Skip(o).Take(m).Select(v => (int)v).ToArray(); o += m;
                    var Nidx = hist.Skip(o).Take(n).Select(v => (int)v).ToList(); o += n;
                    int entering = (int)hist[o];
                    bool[,] hl = null;
                    if (k > 0)
                    {
                        hl = new bool[m, 4];
                        int leaveRow = Array.IndexOf(Bidx, entering);
                        for (int j = 0; j < 4; j++) hl[leaveRow, j] = true;
                    }
                    updatePivot(k == 0
                        ? RevisedPrimalSimplex.BuildIterationBlock(0, Bidx, Nidx, names, Binv, xBk, z, null, null, null, null)
                        : RevisedPrimalSimplex.BuildIterationBlock(k, Bidx, Nidx, names, Binv, xBk, z, rN, entering, d, theta), hl);
                }
            }
            if (status == -11) throw new Exception(LpxNative.StatusMessage(status));
            if (status == -3) throw new Exception("Iteration limit exceeded in Revised Primal Simplex.");
            return RevisedPrimalSimplex.BuildFinalSummary(original, basis, names, xB, status == 1 ? "UNBOUNDED" : "OPTIMAL");
        }
    }
}
