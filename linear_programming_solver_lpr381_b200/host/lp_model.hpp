// Host layer (C++) above the C ABI: a mirror of the reference's solver interface — same type and
// member names, same argument meaning, same exception messages — standing in for the C# host
// (no .NET toolchain in this image).  Arithmetic never happens here: every Solve() marshals the
// model into flat arrays and calls liblpx.so (include/lpx.h); this layer owns only the text.
//
//   Sense, Rel, Constraint, LPProblem, SimplexResult   R/Models/PrimalSimplex.cs:8-49
//   ILPAlgorithm                                       R/Models/IPLAlgorithm.cs:5-8
//   LPParser.ParseFromText                             R/Models/LPParser.cs:9-59
//   LPSolver.Solve / NormalizeAlgorithmKey             R/Models/LPSolver.cs:16-76
//   LPController.SolvePrimalSimplex                    R/Controllers/LPController.cs:13-17
//   CuttingPlane.Solve                                 R/Models/CuttingPlane.cs:13-164
#pragma once
#include <functional>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

namespace lpr381 {

enum class Sense { Max = 0, Min = 1 };
enum class Rel { LE = 0, GE = 1, EQ = 2 };

struct Constraint {
    std::vector<double> A;
    Rel Relation = Rel::LE;
    double B = 0;
};

struct LPProblem {
    Sense ObjectiveSense = Sense::Max;
    std::vector<double> C;
    std::vector<Constraint> Constraints;
    int NumVars() const { return (int)C.size(); }
    LPProblem Clone() const { return *this; }
};

// double[,]
struct Matrix {
    int rows = 0, cols = 0;
    std::vector<double> v;
    double& at(int i, int j) { return v[(size_t)i * cols + j]; }
    double at(int i, int j) const { return v[(size_t)i * cols + j]; }
    bool is_null() const { return rows == 0; }
};

// bool[,] (null when rows == 0)
struct Highlight {
    int rows = 0, cols = 0;
    std::vector<unsigned char> v;
};

struct SimplexResult {
    std::string Report, Summary;
    double OptimalValue = 0;
    bool HasSolution = false;  // Solution != null
    std::vector<double> Solution;
    Matrix Tableau;            // null when is_null()
    std::vector<int> Basis;
    std::vector<std::string> VarNames;
};

// Action<string, bool[,]> updatePivot
using UpdatePivot = std::function<void(const std::string&, const Highlight&)>;

// System.Exception with the reference's message
struct LpException : std::runtime_error {
    int code;
    explicit LpException(const std::string& m, int c = 0) : std::runtime_error(m), code(c) {}
};

struct ILPAlgorithm {
    virtual ~ILPAlgorithm() = default;
    virtual SimplexResult Solve(const LPProblem& problem, UpdatePivot updatePivot = nullptr) = 0;
};

struct LPParser {
    static LPProblem ParseFromText(const std::string& input);
};

struct PrimalSimplex : ILPAlgorithm {
    SimplexResult Solve(const LPProblem& original, UpdatePivot updatePivot = nullptr) override;
};
// R/Models/RevisedPrimalSimplex.cs:13-145 (LPSolver keys "revised primal simplex", "revised primal")
struct RevisedPrimalSimplex : ILPAlgorithm {
    SimplexResult Solve(const LPProblem& original, UpdatePivot updatePivot = nullptr) override;
};
struct DualSimplex : ILPAlgorithm {
    SimplexResult Solve(const LPProblem& original, UpdatePivot updatePivot = nullptr) override;
};
struct BranchAndBound : ILPAlgorithm {
    double BestObjective = 0;
    std::vector<double> BestSolution;
    bool HasBest = false;
    SimplexResult Solve(const LPProblem& problem, UpdatePivot updatePivot = nullptr) override;
};
struct BranchAndBoundKnapsack : ILPAlgorithm {
    SimplexResult Solve(const LPProblem& problem, UpdatePivot updatePivot = nullptr) override;
};

// R/Models/CuttingPlane.cs:9-165 — constructed directly by the GUI (Form1.cs:249-254), no LPSolver key
struct CuttingPlane : ILPAlgorithm {
    std::vector<Constraint> Cuts;  // the Gomory cuts added, in order (not kept upstream; for inspection)
    SimplexResult Solve(const LPProblem& problem, UpdatePivot updatePivot = nullptr) override;
};

// R/Models/CuttingPlaneRevised.cs:9-111 — GUI entry "Revised Cutting Plane" (Form1.cs:256-261)
struct CuttingPlaneRevised : ILPAlgorithm {
    std::vector<Constraint> Cuts;
    SimplexResult Solve(const LPProblem& problem, UpdatePivot updatePivot = nullptr) override;
};

struct LPSolver {
    Matrix FinalTableau;
    SimplexResult Solve(const LPProblem& problem, const std::string& algorithm, UpdatePivot updatePivot = nullptr);
    static std::string NormalizeAlgorithmKey(const std::string& algorithm);
};

struct LPController {
    static SimplexResult SolvePrimalSimplex(const LPProblem& problem);
};

// `lpr381 --sensitivity`: this project's sensitivity block for an optimal Primal Simplex result (sensitivity_host.cpp);
// the status message instead when the solve does not end OPTIMAL.  Not the reference's SensitivityAnalysis text.
std::string SensitivityText(const LPProblem& problem);
// `lpr381 --what-if`: re-optimization queries against the optimal Primal Simplex result (whatif_host.cpp)
std::string WhatIfText(const LPProblem& problem, const std::vector<std::string>& specs);

// Environment.NewLine of the host ("\n"; the reference's Windows build uses "\r\n")
std::string& NewLine();

}  // namespace lpr381
