// Parametric block of `lpr381 --parametric "<spec>" "Primal Simplex"`: the optimal value along b + theta d or
// c + theta d (include/lpx.h, "Parametric analysis") from the model's optimal Primal Simplex result, one
// lpx_parametric call per spec.  Specs (d in the model's constraint / variable order, c in the model's sense):
//   rhs <d_1> ... <d_m> [to <theta_max>]      cost <d_1> ... <d_n> [to <theta_max>]
// theta_max defaults to +inf.  Each spec prints one line per segment: the theta range, z at both ends (as the solve
// returns it: the maximum of -c.x for Min), the slope, and the pivot that ends the segment; then how the analysis ended.
#include <cmath>
#include <cstdlib>
#include <sstream>
#include <string>
#include <vector>

#include "../../include/lpx.h"
#include "dotnet_text.hpp"
#include "host_util.hpp"

namespace lpr381 {

namespace {

std::string trim(const std::string& s) {
    const size_t a = s.find_first_not_of(" \t\r\n"), b = s.find_last_not_of(" \t\r\n");
    return a == std::string::npos ? "" : s.substr(a, b - a + 1);
}

[[noreturn]] void bad(const std::string& spec) { throw LpException("Parametric spec incorrect: " + spec); }

double number(const std::string& t, const std::string& spec) {
    char* end = nullptr;
    const double v = std::strtod(t.c_str(), &end);
    if (t.empty() || end != t.c_str() + t.size()) bad(spec);
    return v;
}

// custom_hash for finite values, "inf" / "-inf" otherwise
std::string num(double v) {
    if (std::isinf(v)) return v > 0 ? "inf" : "-inf";
    return text::custom_hash(v);
}

const char* end_text(int end) {
    switch (end) {
    case LPX_PARAM_REACHED: return "theta_max reached";
    case LPX_PARAM_UNBOUNDED: return "unbounded beyond the last breakpoint";
    case LPX_PARAM_INFEASIBLE: return "infeasible beyond the last breakpoint";
    default: return "segment limit reached";
    }
}

}  // namespace

std::string ParametricText(const LPProblem& problem, const std::vector<std::string>& specs) {
    Flat f = flatten(problem);
    const std::string& nl = NewLine();
    const int seg_cap = 256;
    int mm = 0;
    for (int i = 0; i < f.m; i++) mm += f.rel[i] == 2 ? 2 : 1;
    const std::vector<std::string> names = var_names(f.n, mm);
    lpx_options opt;
    lpx_default_options(&opt);
    std::string out = "Parametric:" + nl;
    for (const std::string& raw : specs) {
        const std::string spec = trim(raw);
        std::istringstream in(spec);
        std::string word, t;
        in >> word;
        if (word != "rhs" && word != "cost") bad(spec);
        const int kind = word == "rhs" ? LPX_PARAM_RHS : LPX_PARAM_COST;
        const int k = kind == LPX_PARAM_RHS ? f.m : f.n;
        std::vector<double> pay;
        for (int i = 0; i < k; i++) {
            if (!(in >> t)) bad(spec);
            pay.push_back(number(t, spec));
        }
        double tmax = INFINITY;
        if (in >> t) {
            if (t != "to" || !(in >> t)) bad(spec);
            tmax = number(t, spec);
            if (!(tmax >= 0.0)) bad(spec);
        }
        if (in >> t) bad(spec);
        pay.push_back(tmax);

        const size_t sstride = lpx_param_segment_stride(f.n);
        std::vector<double> seg((size_t)seg_cap * sstride);
        std::vector<int> spv((size_t)seg_cap * 2);
        int base_status = LPX_OPTIMAL, end = 0, nseg = 0;
        throw_on(lpx_parametric(kind, f.m, f.n, f.sense, f.A.data(), f.rel.data(), f.b.data(), f.c.data(), &opt, 1,
                                pay.data(), seg_cap, &base_status, &end, &nseg, nullptr, seg.data(), spv.data(),
                                nullptr, nullptr));
        if (base_status != LPX_OPTIMAL) return out + lpx_status_message(base_status) + nl;
        out += spec + ": " + std::to_string(nseg) + " segments" + nl;
        for (int s = 0; s < nseg; s++) {
            const double* r = seg.data() + (size_t)s * sstride;
            const double lo = r[0], hi = r[1], z0 = r[2], dz = r[3];
            const double zlo = z0 + lo * dz, zhi = dz == 0.0 ? z0 : z0 + hi * dz;
            out += "  theta [" + num(lo) + ", " + num(hi) + "]: z " + num(zlo) + " -> " + num(zhi) + ", slope " +
                   num(dz);
            if (spv[2 * s] >= 0)
                out += ", then " + names[spv[2 * s + 1]] + " enters in row " + std::to_string(spv[2 * s] + 1);
            out += nl;
        }
        out += "  end: " + std::string(end_text(end)) + nl;
    }
    return out;
}

}  // namespace lpr381
