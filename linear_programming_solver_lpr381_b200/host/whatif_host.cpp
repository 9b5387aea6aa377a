// What-if block of `lpr381 --what-if "<spec>" "Primal Simplex"`: re-optimization queries (include/lpx.h,
// "Re-optimization") against the model's optimal Primal Simplex result, one lpx_reoptimize call per kind.  Specs
// (indices 1-based, as the report names x1 and Constraint 1):
//   rhs <i> <new b_i>            cost <j> <new c_j>
//   row <a constraint line>      the input format's constraint grammar, '<=' / '>=' only
//   col <c> <a_1> ... <a_m>      a new variable with objective coefficient c and column a
// Each query prints its spec, status, pivot count, z (as the solve returns it: the maximum of -c.x for Min) and x.
#include <cstdlib>
#include <sstream>
#include <string>
#include <vector>

#include "../../include/lpx.h"
#include "dotnet_text.hpp"
#include "host_util.hpp"

namespace lpr381 {

namespace {

struct Query {
    std::string spec;
    int kind = 0;
    std::vector<double> payload;
    int status = 0, pivots = 0;
    double z = 0;
    std::vector<double> x;
};

std::string trim(const std::string& s) {
    const size_t a = s.find_first_not_of(" \t\r\n"), b = s.find_last_not_of(" \t\r\n");
    return a == std::string::npos ? "" : s.substr(a, b - a + 1);
}

bool parse_double(const std::string& t, double& v) {
    char* end = nullptr;
    v = std::strtod(t.c_str(), &end);
    return !t.empty() && end == t.c_str() + t.size();
}

[[noreturn]] void bad(const std::string& spec) { throw LpException("What-if spec incorrect: " + spec); }

Query parse_spec(const std::string& spec, const Flat& f, const LPProblem& problem) {
    Query q;
    q.spec = trim(spec);
    std::istringstream in(q.spec);
    std::string word;
    in >> word;
    auto number = [&](double& v) {
        std::string t;
        if (!(in >> t) || !parse_double(t, v)) bad(q.spec);
    };
    auto index = [&](int limit) {
        double v;
        number(v);
        if (v != (int)v || v < 1 || v > limit) bad(q.spec);
        return (int)v - 1;
    };
    if (word == "rhs" || word == "cost") {
        const bool rhs = word == "rhs";
        const int k = index(rhs ? f.m : f.n);
        double v;
        number(v);
        q.kind = rhs ? LPX_REOPT_RHS : LPX_REOPT_COST;
        q.payload.assign(rhs ? f.m : f.n, 0.0);
        q.payload[k] = v - (rhs ? f.b[k] : f.c[k]);
    } else if (word == "row") {
        std::string line;
        std::getline(in, line);
        // the constraint grammar of LPParser, under a placeholder objective
        LPProblem one = LPParser::ParseFromText(std::string(problem.ObjectiveSense == Sense::Max ? "Max" : "Min") +
                                                ": 1x1\n" + trim(line));
        const Constraint& cons = one.Constraints.at(0);
        if (cons.Relation == Rel::EQ || (int)cons.A.size() > f.n) bad(q.spec);
        q.kind = LPX_REOPT_ROW;
        q.payload.assign(f.n + 2, 0.0);
        for (size_t j = 0; j < cons.A.size(); j++) q.payload[j] = cons.A[j];
        q.payload[f.n] = cons.Relation == Rel::GE ? 1.0 : 0.0;
        q.payload[f.n + 1] = cons.B;
    } else if (word == "col") {
        double c;
        number(c);
        q.kind = LPX_REOPT_COL;
        q.payload.assign(f.m + 1, 0.0);
        for (int i = 0; i < f.m; i++) number(q.payload[i]);
        q.payload[f.m] = c;
    } else {
        bad(q.spec);
    }
    std::string extra;
    if (in >> extra && word != "row") bad(q.spec);
    return q;
}

std::string status_name(int s) {
    if (s == LPX_OPTIMAL) return "OPTIMAL";
    if (s == LPX_UNBOUNDED) return "UNBOUNDED";
    if (s == LPX_INFEASIBLE) return "INFEASIBLE";
    return lpx_status_message(s);
}

}  // namespace

std::string WhatIfText(const LPProblem& problem, const std::vector<std::string>& specs) {
    Flat f = flatten(problem);
    std::vector<Query> qs;
    for (const std::string& s : specs) qs.push_back(parse_spec(s, f, problem));
    lpx_options opt;
    lpx_default_options(&opt);
    int base_status = LPX_OPTIMAL;
    for (int kind = LPX_REOPT_RHS; kind <= LPX_REOPT_COL; kind++) {
        std::vector<int> idx;
        for (int k = 0; k < (int)qs.size(); k++)
            if (qs[k].kind == kind) idx.push_back(k);
        if (idx.empty()) continue;
        const int count = (int)idx.size(), stride = (int)lpx_reopt_payload_stride(kind, f.m, f.n);
        const int nx = kind == LPX_REOPT_COL ? f.n + 1 : f.n;
        std::vector<double> pay((size_t)count * stride), x((size_t)count * nx), z(count);
        std::vector<int> status(count), piv(count);
        for (int k = 0; k < count; k++)
            std::copy(qs[idx[k]].payload.begin(), qs[idx[k]].payload.end(), pay.begin() + (size_t)k * stride);
        throw_on(lpx_reoptimize(kind, f.m, f.n, f.sense, f.A.data(), f.rel.data(), f.b.data(), f.c.data(), &opt, count,
                                pay.data(), &base_status, status.data(), piv.data(), nullptr, 0, nullptr, x.data(),
                                z.data(), nullptr));
        for (int k = 0; k < count; k++) {
            Query& q = qs[idx[k]];
            q.status = status[k];
            q.pivots = piv[k];
            q.z = z[k];
            q.x.assign(x.begin() + (size_t)k * nx, x.begin() + (size_t)(k + 1) * nx);
        }
    }
    const std::string& nl = NewLine();
    std::string out = "What-if:" + nl;
    if (base_status != LPX_OPTIMAL) return out + lpx_status_message(base_status) + nl;
    for (const Query& q : qs) {
        out += q.spec + ": " + status_name(q.status) + ", " + std::to_string(q.pivots) + " pivots";
        if (q.status == LPX_OPTIMAL) {
            out += ", z " + text::custom_hash(q.z) + ", x (";
            for (size_t j = 0; j < q.x.size(); j++) out += (j ? ", " : "") + text::custom_hash(q.x[j]);
            out += ")";
        }
        out += nl;
    }
    return out;
}

}  // namespace lpr381
