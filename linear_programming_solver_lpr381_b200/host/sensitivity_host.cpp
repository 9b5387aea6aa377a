// Sensitivity block of `lpr381 --sensitivity "Primal Simplex"`: this project's report (include/lpx.h, "Sensitivity
// analysis of an optimal Primal Simplex result"), not the text of the reference's SensitivityAnalysis, which reads
// the z-row from tableau row 0 where its PrimalSimplex keeps it last.  One lpx_primal_solve_sensitivity_batched call
// with count 1; only status, basis and the report come back from the device.
// The "Two-Phase Sensitivity Analysis" block of `lpr381 --two-phase-sensitivity` prints the two-phase report
// (lpx_two_phase_solve_sensitivity_batched) in the same line formats, then b.y and the objective as written.
#include <cmath>
#include <string>
#include <vector>

#include "../../include/lpx.h"
#include "dotnet_text.hpp"
#include "host_util.hpp"

namespace lpr381 {

static std::string num(double v) {
    if (std::isinf(v)) return v < 0 ? "-inf" : "inf";
    return text::custom_hash(v);
}

// Per variable: reduced cost and cost range; per constraint: shadow price, slack and RHS range.
static std::string report_lines(const double* rep, int m, int n) {
    const std::string& nl = NewLine();
    const double* shadow = rep;
    const double *slack = shadow + m, *rlo = slack + m, *rhi = rlo + m;
    const double *red = rhi + m, *clo = red + n, *chi = clo + n;
    std::string out;
    for (int j = 0; j < n; j++)
        out += "x" + std::to_string(j + 1) + ": reduced cost " + num(red[j]) + ", cost range [" + num(clo[j]) + ", " +
               num(chi[j]) + "]" + nl;
    for (int i = 0; i < m; i++)
        out += "Constraint " + std::to_string(i + 1) + ": shadow price " + num(shadow[i]) + ", slack " + num(slack[i]) +
               ", RHS range [" + num(rlo[i]) + ", " + num(rhi[i]) + "]" + nl;
    return out;
}

std::string SensitivityText(const LPProblem& problem) {
    Flat f = flatten(problem);
    int rows = 0, cols = 0;
    throw_on(lpx_tableau_dims(f.m, f.n, f.rel.data(), &rows, &cols));
    lpx_options opt;
    lpx_default_options(&opt);
    int status = 0;
    std::vector<double> rep(lpx_sensitivity_stride(f.m, f.n));
    throw_on(lpx_primal_solve_sensitivity_batched(1, f.m, f.n, f.sense, f.A.data(), f.rel.data(), f.b.data(),
                                                  f.c.data(), &opt, &status, nullptr, nullptr, nullptr, nullptr,
                                                  rep.data(), nullptr));
    const std::string& nl = NewLine();
    std::string out = "Sensitivity Analysis:" + nl;
    if (status != LPX_OPTIMAL) return out + lpx_status_message(status) + nl;
    return out + report_lines(rep.data(), f.m, f.n);
}

std::string TwoPhaseSensitivityText(const LPProblem& problem) {
    Flat f = flatten(problem);
    lpx_options opt;
    lpx_default_options(&opt);
    int status = 0;
    double z = 0.0;
    std::vector<double> rep(lpx_sensitivity_stride(f.m, f.n));
    throw_on(lpx_two_phase_solve_sensitivity_batched(1, f.m, f.n, f.sense, f.A.data(), f.rel.data(), f.b.data(),
                                                     f.c.data(), &opt, &status, nullptr, nullptr, nullptr, nullptr, &z,
                                                     rep.data(), nullptr));
    const std::string& nl = NewLine();
    std::string out = "Two-Phase Sensitivity Analysis:" + nl;
    if (status != LPX_OPTIMAL) return out + lpx_status_message(status) + nl;
    double by = 0.0;  // strong duality: b.y in row order from +0 against the objective as written
    for (int i = 0; i < f.m; i++) by += f.b[i] * rep[i];
    out += report_lines(rep.data(), f.m, f.n);
    out += "Dual objective b.y = " + num(by) + nl;
    out += "Objective as written = " + num(f.sense == 1 ? -z : z) + nl;
    return out;
}

}  // namespace lpr381
