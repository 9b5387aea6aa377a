"""Random small IPs for the cutting-plane parity tests (tests/test_cutting_plane_cpu.py, tests/test_gpu_cutting_plane.py).

One batch shares m, n, sense and rel; per instance the data takes one of three forms, so that one batch ends in
different ways: fractional data (the reference's cut never removes the vertex, so these usually run all 50 rounds),
box rows a unit vector each with integer bounds (an integral root, or an UNBOUNDED round when a column is left
uncovered), and fractional data with one column made non-positive (an unbounded direction)."""
import numpy as np


def random_ips(count, m, n, seed, box=0.25, unbounded=0.2):
    rng = np.random.default_rng(seed)
    A = rng.integers(0, 9, (count, m, n)) / rng.choice([1.0, 2.0, 3.0, 4.0, 7.0], (count, m, 1))
    b = rng.integers(4, 40, (count, m)) / rng.choice([1.0, 2.0, 3.0], (count, m))
    c = rng.integers(1, 12, (count, n)).astype(np.float64)
    for k in range(count):
        u = rng.random()
        if u < box:
            A[k] = 0.0
            for i in range(m):
                A[k, i, rng.integers(n)] = 1.0
            b[k] = rng.integers(1, 9, m)
        elif u < box + unbounded:
            A[k, :, rng.integers(n)] = -rng.integers(0, 3, m)
    return A, b, c
