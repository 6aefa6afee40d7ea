"""All eigenvalues of the Laplacian on the GPU (sgpu_laplacian_eigenvalues / sgpu_similarity_finalize_eigenvalues: the
sim_mat_eigenvalues CSV of spectral_clustering.cpp:127-143) against LAPACK (numpy.linalg.eigvalsh of the oracle's
restated laplacian(), the dsyevd that arma::eig_sym runs), against closed forms at full size, and for determinism.
||L||_2 <= 2, so the bounds are absolute: 1e-10 against LAPACK, 1e-9 for the closed forms at 8 000 and 20 000 cells."""
import numpy as np
import pytest

from oracle import pyoracle as po
from secedo_b200 import api
from secedo_b200.synth import SynthConfig, make_pileup
from spectral_cases import noisy_clusters, reference_two_clusters

pytestmark = pytest.mark.gpu


def symmetric(a):
    a = np.array(a, dtype=np.float64)
    a = (a + a.T) / 2
    np.fill_diagonal(a, 0)
    return a


def isolated(a, cells):
    a = a.copy()
    a[cells, :] = 0
    a[:, cells] = 0
    return a


# the matrix families of test_gpu_spectral.py
FAMILIES = {
    "reference_two_clusters": lambda: reference_two_clusters(100),
    "reference_three_clusters_99": lambda: reference_two_clusters(99, seed=4),
    "one_cluster_noise": lambda: 1.0 + np.random.default_rng(1243).uniform(-1e-3, 1e-3, (100, 100)),
    "noise_700": lambda: noisy_clusters(700, 1, 0.0, seed=3),
    "weak_clusters_1500": lambda: noisy_clusters(1500, 3, 0.15, seed=5),
    "strong_clusters_2000": lambda: noisy_clusters(2000, 4, 5.0, seed=9),
    "isolated_cells": lambda: isolated(symmetric(noisy_clusters(300, 2, 2.0, seed=11)), [5, 77]),
    "two_components": lambda: np.kron(np.eye(2), np.ones((150, 150))) * noisy_clusters(300, 1, 0.0, seed=13),
}


def lapack(a):
    return np.linalg.eigvalsh(po.laplacian(a))


@pytest.mark.parametrize("name", sorted(FAMILIES))
def test_families_against_lapack(gpu_ctx, name):
    a = symmetric(FAMILIES[name]())
    ev = api.laplacian_eigenvalues(a, ctx=gpu_ctx)
    assert np.abs(ev - lapack(a)).max() <= 1e-10
    assert np.all(np.diff(ev) >= 0)


# block edges of panels of 32 and 64 columns and of the 64-row tiles
@pytest.mark.parametrize("n", [1, 2, 3, 31, 32, 33, 63, 64, 65, 127, 128, 129, 257, 1000, 2100, 4097])
def test_sizes_against_lapack(gpu_ctx, n):
    a = symmetric(noisy_clusters(n, 3, 1.0, seed=n))
    ev, st = api.laplacian_eigenvalues(a, ctx=gpu_ctx, return_stats=True)
    assert np.abs(ev - lapack(a)).max() <= 1e-10
    assert np.all(np.diff(ev) >= 0)
    m = n - 1
    assert st["bytes_matvec"] == int(8.0 * m * (m + 1) * (m + 2) / 6)
    if a.any():
        assert 0 < st["launches"] <= 8 * n + 8


def complete(n):
    return np.ones((n, n)) - np.eye(n)


def cycle(n):
    a = np.zeros((n, n))
    i = np.arange(n)
    a[i, (i + 1) % n] = 1
    a[(i + 1) % n, i] = 1
    return a


@pytest.mark.parametrize("n", [8000, 20000])
def test_closed_forms_full_size(gpu_ctx, n):
    # complete graph: 0 once, n / (n - 1) n - 1 times (a fully degenerate spectrum)
    ev = api.laplacian_eigenvalues(complete(n), ctx=gpu_ctx)
    want = np.full(n, n / (n - 1))
    want[0] = 0
    assert np.abs(ev - want).max() <= 1e-9
    # cycle: 1 - cos(2 pi k / n), in pairs
    ev = api.laplacian_eigenvalues(cycle(n), ctx=gpu_ctx)
    want = np.sort(1 - np.cos(2 * np.pi * np.arange(n) / n))
    assert np.abs(ev - want).max() <= 1e-9
    # c complete graphs: 0 exactly c times, m / (m - 1) for the rest
    c = 5 if n == 8000 else 4
    m = n // c
    ev = api.laplacian_eigenvalues(np.kron(np.eye(c), complete(m)), ctx=gpu_ctx)
    want = np.full(n, m / (m - 1))
    want[:c] = 0
    assert np.abs(ev - want).max() <= 1e-9
    assert ev[c] > 0.5


def synth_counts(ctx, cfg):
    ident = np.arange(cfg.n_cells, dtype=np.uint32)
    f, _ = api.Filter(0.01, 4, ctx).filter(make_pileup(cfg), ident, "", 1)
    c = api.Counts(ctx, cfg.n_cells)
    c.accumulate(f, 1000, ident, 0.01, 0.5, 0.01, 8, "gemm")
    return c


def test_cfg3_matrix(gpu_ctx):
    """8 000 cells (cfg3): trace and Frobenius norm of L, the range [0, 2] and the 7 smallest against the eigenpair
    solver"""
    n = 8000
    dev = gpu_ctx.synth_pileup(n, 0.5, 1, 2048, n_clones=4, theta=0.001, p_multi=0.005, p_mate=0.01, seed=5)
    ident = np.arange(n, dtype=np.uint32)
    fdev, _ = api.Filter(0.001, 4, gpu_ctx).filter_device(dev, ident)
    c = api.Counts(gpu_ctx, n)
    c.accumulate(fdev, 1000, ident, 0.01, 0.15, 0.001, 8, "gemm")
    ev, st, m = c.finalize_eigenvalues(1000, 0.01, 0.15, 0.001, "ADD_MIN", want_matrix=True)
    ev7, _, _, _ = c.finalize_spectral(1000, 0.01, 0.15, 0.001, "ADD_MIN", k=7, tol=1e-10)
    c.free()
    s = 1 / np.sqrt(m.sum(1))
    lap = np.eye(n) - m * s[:, None] * s[None, :]
    assert abs(ev.sum() - np.trace(lap)) <= 1e-9 * n
    fro = np.square(lap).sum()
    assert abs(np.square(ev).sum() - fro) <= 1e-9 * fro
    assert ev.min() >= -1e-12 and ev.max() <= 2 + 1e-12
    assert np.abs(ev[:7] - ev7).max() <= 1e-9
    print("eigenvalue stats at 8000 cells:", st)


def test_finalize_consistency_and_determinism(gpu_ctx):
    cfg = SynthConfig(n_cells=700, coverage=0.4, n_loci=3000, n_chr=2, n_clones=3, p_multi=0.1, p_mate=0.05, theta=0.01, seed=21)
    c = synth_counts(gpu_ctx, cfg)
    m = c.finalize(1000, 0.01, 0.5, 0.01, "ADD_MIN")
    ev, st, m2 = c.finalize_eigenvalues(1000, 0.01, 0.5, 0.01, "ADD_MIN", want_matrix=True)
    assert np.array_equal(m, m2)
    assert np.array_equal(ev, api.laplacian_eigenvalues(m, ctx=gpu_ctx))
    ev2, _, none = c.finalize_eigenvalues(1000, 0.01, 0.5, 0.01, "ADD_MIN")
    assert none is None and np.array_equal(ev, ev2)
    assert np.abs(ev - lapack(m)).max() <= 1e-10
    assert st["ms_tridiagonal"] > 0 and st["ms_epilogue"] > 0
    c.free()


def test_edge_cases_and_refusals(gpu_ctx):
    assert np.array_equal(api.laplacian_eigenvalues(np.zeros((99, 99)), ctx=gpu_ctx), np.ones(99))
    a = symmetric(noisy_clusters(200, 2, 1.0, seed=2))
    cells = [0, 17, 64, 199]
    ev = api.laplacian_eigenvalues(isolated(a, cells), ctx=gpu_ctx)
    ref = lapack(isolated(a, cells))
    assert np.abs(ev - ref).max() <= 1e-10
    assert (np.abs(ev - 1) <= 1e-12).sum() >= len(cells)
    with pytest.raises(api.SgpuError):
        api.laplacian_eigenvalues(-a, ctx=gpu_ctx)  # negative degrees
    with pytest.raises(api.SgpuError):
        api.laplacian_eigenvalues(np.zeros((0, 0)), ctx=gpu_ctx)
    nan = a.copy()
    nan[3, 4] = nan[4, 3] = np.nan
    with pytest.raises(api.SgpuError):
        api.laplacian_eigenvalues(nan, ctx=gpu_ctx)
