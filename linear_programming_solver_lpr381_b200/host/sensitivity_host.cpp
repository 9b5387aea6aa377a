// Sensitivity block of `lpr381 --sensitivity "Primal Simplex"`: this project's report (include/lpx.h, "Sensitivity
// analysis of an optimal Primal Simplex result"), not the text of the reference's SensitivityAnalysis, which reads
// the z-row from tableau row 0 where its PrimalSimplex keeps it last.  One lpx_primal_solve_sensitivity_batched call
// with count 1; only status, basis and the report come back from the device.
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
    const int m = f.m, n = f.n;
    const double* shadow = rep.data();
    const double *slack = shadow + m, *rlo = slack + m, *rhi = rlo + m;
    const double *red = rhi + m, *clo = red + n, *chi = clo + n;
    for (int j = 0; j < n; j++)
        out += "x" + std::to_string(j + 1) + ": reduced cost " + num(red[j]) + ", cost range [" + num(clo[j]) + ", " +
               num(chi[j]) + "]" + nl;
    for (int i = 0; i < m; i++)
        out += "Constraint " + std::to_string(i + 1) + ": shadow price " + num(shadow[i]) + ", slack " + num(slack[i]) +
               ", RHS range [" + num(rlo[i]) + ", " + num(rhi[i]) + "]" + nl;
    return out;
}

}  // namespace lpr381
