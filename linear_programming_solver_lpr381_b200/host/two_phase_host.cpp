// "Two-Phase Simplex" block of `lpr381 --two-phase [input]`: the model solved by lpx_two_phase_solve_batched
// (include/lpx.h, "Two-phase Simplex"), which accepts '>=' rows, '=' rows and negative right-hand sides.  This
// project's own text, not the reference's: the status, z as the solve returns it (for Min the maximum of -c.x, as in
// every other report), x, and the pivots of each phase.  Columns are named x<j> (decision variables), s<i> (the slack
// of constraint i) and a<i> (the artificial of constraint i); rows are numbered from 1.
#include <string>
#include <vector>

#include "../../include/lpx.h"
#include "dotnet_text.hpp"
#include "host_util.hpp"

namespace lpr381 {

namespace {

const char* status_text(int status) {
    switch (status) {
    case LPX_OPTIMAL: return "OPTIMAL";
    case LPX_UNBOUNDED: return "UNBOUNDED";
    case LPX_INFEASIBLE: return "INFEASIBLE";
    default: return lpx_status_message(status);
    }
}

}  // namespace

std::string TwoPhaseText(const LPProblem& problem) {
    Flat f = flatten(problem);
    const std::string& nl = NewLine();
    lpx_options opt;
    lpx_default_options(&opt);
    const int cap = opt.max_iterations + f.m;  // drive-out pivots come on top of the limit

    // column names in the definition's numbering: decision variables, slacks, artificials (b_i < 0 flips the row)
    std::vector<std::string> names;
    for (int j = 0; j < f.n; j++) names.push_back("x" + std::to_string(j + 1));
    for (int i = 0; i < f.m; i++)
        if (f.rel[i] != 2) names.push_back("s" + std::to_string(i + 1));
    for (int i = 0; i < f.m; i++) {
        const int rn = (f.b[i] < 0.0 && f.rel[i] != 2) ? 1 - f.rel[i] : f.rel[i];
        if (rn != 0) names.push_back("a" + std::to_string(i + 1));
    }

    int status = 0, phase1 = 0, npiv = 0;
    std::vector<int> pivots((size_t)cap * 2), basis(f.m);
    std::vector<double> x(f.n);
    double z = 0.0;
    long long total = 0;
    throw_on(lpx_two_phase_solve_batched(1, f.m, f.n, f.sense, f.A.data(), f.rel.data(), f.b.data(), f.c.data(), &opt,
                                         &status, &phase1, &npiv, pivots.data(), cap, basis.data(), x.data(), &z,
                                         nullptr, &total));
    std::string out = "Two-Phase Simplex:" + nl;
    out += "Status: " + std::string(status_text(status)) + nl;
    out += "z* = " + text::custom_hash(z) + nl;
    out += "x* = [";
    for (int j = 0; j < f.n; j++) out += (j ? ", " : "") + text::custom_hash(x[j]);
    out += "]" + nl;
    const int logged = npiv < cap ? npiv : cap;
    for (int ph = 1; ph <= 2; ph++) {
        const int lo = ph == 1 ? 0 : phase1, hi = ph == 1 ? phase1 : npiv;
        out += std::string(ph == 1 ? "Phase I" : "Phase II") + ": " + std::to_string(hi - lo) + " pivots" + nl;
        for (int k = lo; k < hi && k < logged; k++)
            out += "  " + names[pivots[2 * k]] + " enters in row " + std::to_string(pivots[2 * k + 1] + 1) + nl;
    }
    return out;
}

}  // namespace lpr381
