"""Deterministic synthetic workloads for the five BASELINE.json configs (SURVEY.md §8d).

Plain numpy; no torch, no CUDA.  Every generator is a pure function of its seed so that the
oracle, the CUDA path, the tests and bench.py all see identical inputs.
"""
import numpy as np

WYNDOR_TEXT = "Max: 3x1 + 5x2\n1x1 + 0x2 <= 4\n0x1 + 2x2 <= 12\n3x1 + 2x2 <= 18\n"


def _rng(seed):
    return np.random.Generator(np.random.PCG64(int(seed)))


def lp_integer(m, n, seed, a_hi=9, c_hi=9, b_lo_mul=2, b_hi_mul=6):
    """All-<= Max LP with small integer data: A U{1..a_hi}, b U{b_lo_mul*n .. b_hi_mul*n-1}, c U{1..c_hi}.
    Exactly representable, bounded, feasible at x = 0 (C2 / C3 generator)."""
    r = _rng(seed)
    A = r.integers(1, a_hi + 1, size=(m, n)).astype(np.float64)
    b = r.integers(b_lo_mul * n, b_hi_mul * n, size=m).astype(np.float64)
    c = r.integers(1, c_hi + 1, size=n).astype(np.float64)
    return A, b, c


def lp_decimal(m, n, seed):
    """Tie-free variant: 3-decimal U(0,1) for A and c, b 3-decimal U(n/8, n/4)."""
    r = _rng(seed)
    A = np.round(r.random((m, n)), 3)
    A[A == 0] = 0.001
    c = np.round(r.random(n), 3)
    b = np.round(n / 8 + r.random(m) * (n / 8), 3)
    return A, b, c


def batch_c2(count=4096, m=64, n=128, seed=1, kind="integer"):
    """C2: `count` independent LPs; instance k uses seed*4096 + k."""
    gen = lp_integer if kind == "integer" else lp_decimal
    A = np.empty((count, m, n))
    b = np.empty((count, m))
    c = np.empty((count, n))
    for k in range(count):
        A[k], b[k], c[k] = gen(m, n, seed * 4096 + k)
    return A, b, c


def large_c3(m=4096, n=8192, seed=7):
    """C3: one large dense LP, same integer generator."""
    return lp_integer(m, n, seed)


def large_dual(m_eq=2048, n=8192, seed=17):
    """Dual Simplex workload of C3's tableau shape: Min c.x subject to A x = b, x >= 0, every row an equality.
    A U{1..9}, c U{1..9}; b = A x0 for a random sparse integer x0 >= 0 (about n/64 entries U{1..4}), so the LP is
    feasible by construction and bounded (c > 0).  2 m_eq + 1 rows after the EQ expansion: 4097 x 12289 by default.
    Returns (A, b, c, rel, sense) with sense = 1 (Min); smaller m_eq, n for tests."""
    r = _rng(seed)
    A = r.integers(1, 10, size=(m_eq, n)).astype(np.float64)
    c = r.integers(1, 10, size=n).astype(np.float64)
    x0 = np.zeros(n)
    k = max(1, n // 64)
    x0[r.choice(n, size=k, replace=False)] = r.integers(1, 5, size=k)
    b = A @ x0
    return A, b, c, np.full(m_eq, 2, dtype=np.int32), 1


def ip_c4(m=60, n=120, seed=11):
    """C4: general IP, A U{1..19}, b U{5n..15n-1}, c U{1..29}."""
    r = _rng(seed)
    A = r.integers(1, 20, size=(m, n)).astype(np.float64)
    b = r.integers(5 * n, 15 * n, size=m).astype(np.float64)
    c = r.integers(1, 30, size=n).astype(np.float64)
    return A, b, c


def knapsack_c5(n=2000, seed=13, kind="uncorrelated"):
    """C5: weights U{1..1000}; profits uncorrelated / weakly (w +- 100) / strongly (w + 100)
    correlated; capacity floor(sum(w) / 2).  `kind="fractional"` gives non-integer data so that
    the ordered-summation path is exercised."""
    r = _rng(seed)
    w = r.integers(1, 1001, size=n).astype(np.float64)
    if kind == "uncorrelated":
        p = r.integers(1, 1001, size=n).astype(np.float64)
    elif kind == "weak":
        p = np.maximum(1.0, w + r.integers(-100, 101, size=n))
    elif kind == "strong":
        p = w + 100.0
    elif kind == "fractional":
        w = np.round(w / 7.0, 3)
        p = np.round(r.random(n) * 100.0 + 0.001, 3)
    else:
        raise ValueError(kind)
    cap = float(np.floor(w.sum() / 2.0))
    return p, w, cap


def lp_to_text(A, b, c, rel=None, sense=0):
    """Render a problem in the reference's text format (R/Models/LPParser.cs)."""
    def term(v, j):
        return f"{repr(float(v))}x{j + 1}" if v != int(v) else f"{int(v)}x{j + 1}"
    def expr(row):
        s = " + ".join(term(v, j) for j, v in enumerate(row))
        return s.replace("+ -", "- ")
    lines = [("Max: " if sense == 0 else "Min: ") + expr(c)]
    sym = {0: "<=", 1: ">=", 2: "="}
    for i in range(A.shape[0]):
        rv = b[i]
        rs = str(int(rv)) if rv == int(rv) else repr(float(rv))
        lines.append(f"{expr(A[i])} {sym[0 if rel is None else int(rel[i])]} {rs}")
    return "\n".join(lines) + "\n"
