"""Sturm counts and bisection of secedo_b200/csrc/sturm.hpp (the eigenvalues of the tridiagonal matrix that the device
computes one index per thread) compiled for the host (tests/sturm_host_check.cpp) against LAPACK's tridiagonal
eigenvalues (scipy.linalg.eigvalsh_tridiagonal)."""
import os
import struct
import subprocess

import numpy as np
import pytest
from scipy.linalg import eigvalsh_tridiagonal

from conftest import ROOT


@pytest.fixture(scope="module")
def sturm_check(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("sturm") / "sturm_host_check")
    subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-Wextra", "-o", exe, os.path.join(ROOT, "tests", "sturm_host_check.cpp")],
                   check=True)
    return exe


def write(path, d, e):
    with open(path, "wb") as f:
        f.write(struct.pack("<I", len(d)))
        f.write(np.ascontiguousarray(d, np.float64).tobytes())
        f.write(np.ascontiguousarray(e, np.float64).tobytes())


def bisect_all(exe, tmp_path, d, e):
    fin, fout = str(tmp_path / "t.bin"), str(tmp_path / "w.bin")
    write(fin, d, e)
    subprocess.run([exe, fin, fout], check=True)
    return np.frombuffer(open(fout, "rb").read())


def wilkinson_plus(m=10):
    """W_{2m+1}^+: d = |m - i|, e = 1; its largest eigenvalues come in pairs that agree to many digits"""
    return np.abs(np.arange(2 * m + 1) - m).astype(np.float64), np.ones(2 * m)


def graded(n, seed):
    rng = np.random.default_rng(seed)
    g = 10.0 ** -np.linspace(0, 12, n)
    return g * rng.uniform(0.5, 1.5, n), g[:-1] * rng.uniform(0.1, 1.0, n - 1)


def split(n, seed):
    rng = np.random.default_rng(seed)
    d, e = rng.normal(size=n), rng.normal(size=n - 1)
    e[rng.choice(n - 1, n // 5, replace=False)] = 0.0  # independent blocks
    d[: n // 3] = 0.25  # and repeated eigenvalues across them
    e[: n // 3] = 0.0
    return d, e


CASES = {
    "random_7": lambda: (np.random.default_rng(1).normal(size=7), np.random.default_rng(2).normal(size=6)),
    "random_300": lambda: (np.random.default_rng(3).normal(size=300), np.random.default_rng(4).normal(size=299)),
    "random_2000_scaled": lambda: (1e3 * np.random.default_rng(5).normal(size=2000), 1e3 * np.random.default_rng(6).normal(size=1999)),
    "graded_200": lambda: graded(200, 7),
    "split_500": lambda: split(500, 8),
    "diagonal_only": lambda: (np.random.default_rng(9).normal(size=64), np.zeros(63)),
    "zero": lambda: (np.zeros(33), np.zeros(32)),
    "wilkinson_21": lambda: wilkinson_plus(10),
    "one": lambda: (np.array([0.3]), np.zeros(0)),
    "two": lambda: (np.array([1.0, -1.0]), np.array([1e-3])),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_bisection_against_lapack(sturm_check, tmp_path, case):
    d, e = CASES[case]()
    w = bisect_all(sturm_check, tmp_path, d, e)
    ref = eigvalsh_tridiagonal(d, e) if len(d) > 1 else d.copy()
    scale = max(np.abs(d).max() + (2 * np.abs(e).max() if len(e) else 0.0), np.finfo(float).tiny)
    assert np.all(np.diff(w) >= 0), "sorted by construction"
    tol = max(8 * np.finfo(float).eps * scale * max(1.0, np.log2(len(d))), 8 * np.finfo(float).tiny)
    assert np.abs(w - ref).max() <= tol, (w - ref)
    if case == "zero":
        assert np.all(1.0 - w == 1.0)  # T = 0: within a few pivmin of 0, so the Laplacian's eigenvalues are exactly 1


def test_wilkinson_pairs_resolved(sturm_check, tmp_path):
    """the two largest eigenvalues of W21+ differ by ~1e-14 relative; both must be found, in order"""
    d, e = wilkinson_plus(10)
    w = bisect_all(sturm_check, tmp_path, d, e)
    ref = eigvalsh_tridiagonal(d, e)
    assert ref[-1] - ref[-2] < 1e-12
    assert np.abs(w[-2:] - ref[-2:]).max() <= 4e-15 * ref[-1]


def test_sturm_count(sturm_check, tmp_path):
    rng = np.random.default_rng(11)
    d, e = rng.normal(size=50), rng.normal(size=49)
    fin = str(tmp_path / "c.bin")
    write(fin, d, e)
    ref = eigvalsh_tridiagonal(d, e)
    for x in (-100.0, ref[0] - 1e-9, ref[0] + 1e-9, 0.0, ref[25] + 1e-9, ref[-1] + 1e-9, 100.0):
        c = int(subprocess.run([sturm_check, "--count", fin, repr(float(x)), "-"], check=True, capture_output=True, text=True).stdout)
        assert c == int((ref < x).sum()), x
