// lpr381 — headless front end of the host layer: what Form1.btnSolve_Click / BtnExport_Click do
// (R/Form1.cs:231-279, 298-324) without the window.
//
//   lpr381 "<algorithm>" [input.txt]        algorithm: Primal Simplex | Revised Primal Simplex | Dual Simplex |
//                                           Branch and Bound | Cutting Plane | Revised Cutting Plane | BranchAndBoundKnapsack | ...
//   lpr381 --export "<algorithm>" [input]   the export file layout ("Linear Program:" / "Iterations:")
//   lpr381 --crlf ...                       Environment.NewLine = "\r\n" (where the reference runs)
//   lpr381 --sensitivity "Primal Simplex" [input]   appends this project's "Sensitivity Analysis" block (shadow
//                                           prices, slacks, RHS / cost ranges; not the reference's text)
//   lpr381 --what-if "<spec>" "Primal Simplex" [input]   repeatable: appends a "What-if" block, the optimum after
//                                           each change, re-solved warm (whatif_host.cpp; not the reference's)
//   lpr381 --parametric "<spec>" "Primal Simplex" [input]   repeatable: appends a "Parametric" block, the optimal
//                                           value along a RHS or cost direction (parametric_host.cpp; not the reference's)
//   lpr381 --two-phase [input]               this project's "Two-Phase Simplex" block: models with '>=' rows, '=' rows
//                                           and negative right-hand sides (two_phase_host.cpp; not the reference's)
//   lpr381 --two-phase-sensitivity [input]   the "Two-Phase Simplex" block, then this project's "Two-Phase Sensitivity
//                                           Analysis" block (shadow prices, slacks, ranges, b.y; sensitivity_host.cpp)
#include <cstdio>
#include <fstream>
#include <iostream>
#include <sstream>
#include <vector>

#include "lp_model.hpp"

using namespace lpr381;

int main(int argc, char** argv) {
    int arg = 1;
    bool as_export = false, sensitivity = false, bad_what_if = false, two_phase = false, two_phase_sens = false;
    std::vector<std::string> what_if, parametric;
    for (; arg < argc; arg++) {
        const std::string a = argv[arg];
        if (a == "--export") as_export = true;
        else if (a == "--crlf") NewLine() = "\r\n";
        else if (a == "--sensitivity") sensitivity = true;
        else if (a == "--two-phase") two_phase = true;
        else if (a == "--two-phase-sensitivity") two_phase_sens = true;
        else if (a == "--what-if") {
            if (++arg < argc) what_if.push_back(argv[arg]);
            else bad_what_if = true;
        } else if (a == "--parametric") {
            if (++arg < argc) parametric.push_back(argv[arg]);
            else bad_what_if = true;
        } else break;
    }
    if (two_phase || two_phase_sens) {
        if (sensitivity || !what_if.empty() || !parametric.empty() || bad_what_if || as_export || argc - arg > 1 ||
            (two_phase && two_phase_sens)) {
            std::fprintf(stderr, "usage: lpr381 [--crlf] --two-phase [input.txt]  (no algorithm, no other analysis)\n"
                                 "       lpr381 [--crlf] --two-phase-sensitivity [input.txt]\n");
            return 2;
        }
        std::stringstream in;
        if (arg < argc) {
            std::ifstream f(argv[arg]);
            if (!f) {
                std::fprintf(stderr, "Error reading file: %s\n", argv[arg]);
                return 2;
            }
            in << f.rdbuf();
        } else {
            in << std::cin.rdbuf();
        }
        try {
            const LPProblem problem = LPParser::ParseFromText(in.str());
            std::string out = TwoPhaseText(problem);
            if (two_phase_sens) out += NewLine() + TwoPhaseSensitivityText(problem);
            std::cout << out;
        } catch (const LpException& e) {
            std::fprintf(stderr, "Error: %s\n", e.what());
            return 1;
        }
        return 0;
    }
    if (arg >= argc || bad_what_if) {
        std::fprintf(stderr, "usage: lpr381 [--export] [--crlf] [--sensitivity] [--what-if \"<spec>\"]... \"<algorithm>\" "
                             "[input.txt]\n"
                             "       lpr381 [--crlf] --two-phase [input.txt]\n"
                             "       lpr381 [--crlf] --two-phase-sensitivity [input.txt]\n"
                             "  --sensitivity (\"Primal Simplex\" only): this project's sensitivity report, not the "
                             "reference's\n"
                             "  --what-if (\"Primal Simplex\" only): rhs <i> <b_i> | cost <j> <c_j> | row <constraint> | "
                             "col <c> <a_1> .. <a_m>\n"
                             "  --parametric (\"Primal Simplex\" only): rhs <d_1> .. <d_m> [to <theta_max>] | "
                             "cost <d_1> .. <d_n> [to <theta_max>]\n");
        return 2;
    }
    const std::string algorithm = argv[arg++];
    if ((sensitivity || !what_if.empty()) && algorithm != "Primal Simplex") {
        std::fprintf(stderr, "--sensitivity / --what-if: only \"Primal Simplex\" results are analysed\n");
        return 2;
    }
    if (!parametric.empty() && algorithm != "Primal Simplex") {
        std::fprintf(stderr, "--parametric: only \"Primal Simplex\" results are analysed\n");
        return 2;
    }
    std::stringstream in;
    if (arg < argc) {
        std::ifstream f(argv[arg]);
        if (!f) {
            std::fprintf(stderr, "Error reading file: %s\n", argv[arg]);
            return 2;
        }
        in << f.rdbuf();
    } else {
        in << std::cin.rdbuf();
    }
    const std::string input = in.str();
    std::string box;  // iterationOutputTextBox
    UpdatePivot append = [&](const std::string& text, const Highlight&) { box += text; };
    std::string sens_block;
    try {
        LPProblem problem = LPParser::ParseFromText(input);
        if (sensitivity) sens_block = "\n\n" + SensitivityText(problem);
        if (!what_if.empty()) sens_block += "\n\n" + WhatIfText(problem, what_if);
        if (!parametric.empty()) sens_block += "\n\n" + ParametricText(problem, parametric);
        SimplexResult result;
        // the dropdown routes "Branch and Bound Knapsack" to plain BranchAndBound upstream
        // (Form1.cs:263-270); the knapsack solver itself is reachable here under its class name
        if (algorithm == "BranchAndBoundKnapsack" || algorithm == "knapsack")
            result = BranchAndBoundKnapsack().Solve(problem, append);
        else if (algorithm == "Revised Cutting Plane")  // Form1.cs:256-261
            result = CuttingPlaneRevised().Solve(problem, append);
        else if (algorithm == "Cutting Plane")  // Form1.cs:249-254
            result = CuttingPlane().Solve(problem, append);
        else if (algorithm == "Branch and Bound" || algorithm == "Revised Branch and Bound" ||
                 algorithm == "Branch and Bound Knapsack")
            result = BranchAndBound().Solve(problem, append);
        else
            result = LPSolver().Solve(problem, algorithm, append);
        box += "\n\nFinal Report:\n" + result.Report;
        box += "\n\nSummary:\n" + result.Summary;
        box += sens_block;
    } catch (const LpException& e) {
        // a model the solve rejects (e.g. a '>=' row) still gets its sensitivity / what-if blocks: the status message
        if (!sens_block.empty()) std::cout << sens_block.substr(2);
        std::fprintf(stderr, "Error: %s\n", e.what());
        return 1;
    }
    // BtnExport_Click (Form1.cs:310-314): five StreamWriter.WriteLine calls, each ending in Environment.NewLine
    const std::string& nl = NewLine();
    if (as_export) std::cout << "Linear Program:" << nl << input << nl << nl << "Iterations:" << nl << box << nl;
    else std::cout << box;
    return 0;
}
