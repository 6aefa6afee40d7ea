"""Read pairs that overlap at many loci, planted one class at a time, up to the limits of the log-likelihood tables.

The multi-locus correction records every read pair with x_s + x_d >= 2 by its overlap class: order 2 in the int32
planes (2,0) (1,1) (0,2), order 3 in the planes (3,0) .. (0,3) (planes 5..8 of the count buffer) and order >= 4 as
sum G(x_s, x_d) in the fp64 spill plane. Synthetic pileups exercise only the small classes; here a generator plants
pairs of chosen classes and states what each plane must hold, and the oracle states which classes the reference can
evaluate at all: the device must refuse exactly those (SGPU_E_CLASS_RANGE), and an accumulation it refuses half way
must not leave counts behind that a later accumulation or a zeroing would not account for."""
import functools
from concurrent.futures import ThreadPoolExecutor
from types import SimpleNamespace

import numpy as np
import pytest

from conftest import assert_matrix_close, load_golden
from oracle import pyoracle as po
from secedo_b200 import api
from secedo_b200.pileup import Pileup

TOL = 1e-6
PARAMS = (0.01, 0.5, 0.01)  # mutation rate, homozygous rate, sequencing error rate
N_CELLS = 12
SGPU_E_ARG, SGPU_E_CLASS_RANGE = -2, -5
MAX_CLASS = po.MAX_CLASS
TBL = 132  # the oracle's power tables hold min(max(L, 2), 132) entries


@functools.lru_cache(maxsize=None)
def _full_log_probs(e, h, t):
    return po.log_probs(e, h, t, 1000, MAX_CLASS)


def warm_log_probs():
    """the full tables of every parameter set below, evaluated side by side (ctypes drops the GIL)"""
    params = golden_params()
    with ThreadPoolExecutor(len(params)) as ex:
        list(ex.map(lambda p: _full_log_probs(*p), params))
    return params


def oracle_log_probs(e, h, t, L):
    """po.log_probs(e, h, t, L, min(64, L)). The full 64 x 64 table takes the oracle ~20 s, so it is evaluated once per
    parameter set (at L = 1000, where its power tables have all 132 entries) and cut down: the oracle's entry (s, d)
    does not depend on L except that it is NaN from s + d >= min(max(L, 2), 132) on, where its tables end.
    test_cut_log_prob_tables_are_the_oracles checks this against the oracle wherever that is quick."""
    ls, ld = (x[:min(MAX_CLASS, L), :min(MAX_CLASS, L)].copy() for x in _full_log_probs(e, h, t))
    gone = np.add.outer(np.arange(len(ls)), np.arange(len(ls))) >= min(max(L, 2), TBL)
    ls[gone] = ld[gone] = np.nan
    return ls, ld


def golden_params():
    g = load_golden("log_probs")
    return [tuple(float(x) for x in g[f"params{i}"][:3]) for i in range(len(g.files) // 3)]


def planted_pileup(L, windows, n_cells=N_CELLS, seed=0, n_fill=24):
    """One chromosome holding one window of loci per entry of ``windows``: (cell_a, cell_b, x_s, x_d) plants a read
    pair of that overlap class, (cell_a, cell_b, x_s, x_d, cell_c) adds a third read with random bases over the same
    loci. Both (all) reads cover every locus of their window; the bases of the pair agree at x_s loci and differ at
    x_d, in shuffled order. A window spans less than L bp, and windows lie L bp apart, so no read reaches the next
    one. Loci of fresh single-locus reads follow, so that the reference's tail cutoff lies behind every planted read.

    Returns the pileup and what the multi-locus correction must record: the class histogram (orders >= 2), the
    order-2 planes (symmetric, like Counts.download), the order-3 planes and the spill plane sum G(x_s, x_d) (upper
    triangle, cell pair (lo, hi) at [lo, hi]) with, beside it, sum |F| + x_s |F(1,0)| + x_d |F(0,1)| of its terms.
    G and F are the oracle's (F = LD - LS, G = F - x_s F(1,0) - x_d F(0,1))."""
    rng = np.random.default_rng(seed)
    ls, ld = oracle_log_probs(*PARAMS, L)
    F = ld - ls
    n = n_cells
    exp = SimpleNamespace(hist=np.zeros((MAX_CLASS, MAX_CLASS), np.uint64), H2=np.zeros((3, n, n), np.int32),
                          H3=np.zeros((4, n, n), np.int32), spill=np.zeros((n, n)), terms=np.zeros((n, n)))
    loci = []
    rid = iter(range(1, 1 << 30))
    pos = 1000
    for w in windows:
        a, b, xs, xd = w[:4]
        m = xs + xd
        step = min(13, (L - 1) // (m - 1)) if m > 1 else 1
        base_a = rng.integers(0, 4, m)
        same = rng.permutation(np.r_[np.ones(xs, bool), np.zeros(xd, bool)])
        base_b = np.where(same, base_a, (base_a + rng.integers(1, 4, m)) % 4)
        reads = [(a, next(rid), base_a), (b, next(rid), base_b)]
        if len(w) > 4:
            reads.append((w[4], next(rid), rng.integers(0, 4, m)))
        for k in range(m):
            loci.append((pos + k * step, [r for _, r, _ in reads], [(c << 2) | int(bs[k]) for c, _, bs in reads]))
        for i in range(len(reads)):
            for j in range(i + 1, len(reads)):
                ci, cj = reads[i][0], reads[j][0]
                if ci == cj:
                    continue
                s = int((reads[i][2] == reads[j][2]).sum())
                d = m - s
                lo, hi = min(ci, cj), max(ci, cj)
                if max(s, d) >= len(F):
                    continue  # refused (x_s or x_d >= min(64, L)): nothing to expect
                if m >= 2:
                    exp.hist[s, d] += 1
                if m == 2:
                    exp.H2[d, lo, hi] += 1
                    exp.H2[d, hi, lo] += 1
                elif m == 3:
                    exp.H3[d, lo, hi] += 1
                elif m >= 4:
                    exp.spill[lo, hi] += F[s, d] - s * F[1, 0] - d * F[0, 1]
                    exp.terms[lo, hi] += abs(F[s, d]) + s * abs(F[1, 0]) + d * abs(F[0, 1])
        pos += (m - 1) * step + L
    for k in range(n_fill):
        cells = rng.choice(n, 2, replace=False)
        loci.append((pos + k * L, [next(rid), next(rid)], [(int(c) << 2) | int(rng.integers(0, 4)) for c in cells]))
    return Pileup.from_pos_data([loci]), exp


def small_classes():
    """every class of order 1 .. 6 once, on varying cell pairs (so that one cell pair collects several classes), every
    third one with a third read"""
    out = []
    k = 0
    for m in range(1, 7):
        for xs in range(m + 1):
            a, b = k % 5, 5 + k % 3
            out.append((a, b, xs, m - xs) + ((10 + k % 2,) if k % 3 == 0 else ()))
            k += 1
    return out


# name -> (L, windows). "orders_1_to_32" has no read of more than 65 loci, so the second-order GEMM really runs on it;
# the reads of "wide_1000" (126 loci) and "wide_100" (99 loci) make it fall back to enumeration.
DESIGNS = {
    "orders_1_to_32": (1000, small_classes() + [(0, 5, 4, 0), (1, 6, 0, 4), (2, 7, 10, 10), (0, 5, 31, 32, 11)]),
    "wide_1000": (1000, [(0, 5, 63, 0), (1, 6, 0, 63), (2, 7, 63, 63), (0, 5, 2, 1, 11), (3, 8, 1, 1)]),
    "wide_100": (100, [(0, 5, 60, 39), (1, 6, 50, 49), (2, 7, 2, 1, 11), (3, 8, 0, 2)]),
}

# (L, class, whether the oracle evaluates it): the oracle refuses x_s or x_d >= 64 or >= L, and x_s + x_d >= the length
# min(max(L, 2), 132) of its power tables
REFUSALS = [
    (1000, (64, 0), False), (1000, (0, 64), False), (1000, (63, 63), True), (1000, (63, 0), True),
    (100, (60, 40), False), (100, (60, 39), True), (100, (50, 49), True),
    (4, (2, 1), True), (3, (2, 1), False), (2, (1, 1), False),
]


def refusal_design(L, cls):
    return [(0, 5, 1, 0), (1, 6, cls[0], cls[1]), (2, 7, 0, 1)]


def oracle(p, L, threads):
    return po.similarity(p, N_CELLS, L, np.arange(N_CELLS, dtype=np.uint32), *PARAMS, threads, "ADD_MIN")


def multi_hist(o):
    h = o.class_hist.copy()
    h[0, 0] = h[0, 1] = h[1, 0] = 0
    return h


# ------------------------------------------------------------------------------------------------ host only
@pytest.mark.parametrize("threads", [1, 8])
@pytest.mark.parametrize("name", sorted(DESIGNS))
def test_generator_matches_oracle(name, threads):
    """the generator's expectations are the oracle's: a device failure below cannot be blamed on the generator"""
    L, windows = DESIGNS[name]
    p, exp = planted_pileup(L, windows)
    o = oracle(p, L, threads)
    assert np.array_equal(multi_hist(o), exp.hist)
    assert np.array_equal(o.H, exp.H2)
    assert exp.H3.sum() > 0 and exp.spill.any()
    assert o.S1.sum() > 0 and o.D1.sum() > 0


@pytest.mark.parametrize("L,cls,accepted", REFUSALS)
def test_oracle_refusal_table(L, cls, accepted):
    p, exp = planted_pileup(L, refusal_design(L, cls))
    if accepted:
        assert np.array_equal(multi_hist(oracle(p, L, 1)), exp.hist)
    else:
        with pytest.raises(ValueError, match="rc=-4"):
            oracle(p, L, 1)


# ------------------------------------------------------------------------------------------------ on the GPU
def read_planes(ctx, c):
    """planes 5..8 (order 3) and the spill plane straight from the device buffers; all zero where not allocated"""
    import torch
    from secedo_b200.dist import tensor_from_ptr
    n = c.num_cells
    i32, n_i32, f64, n_f64, _, _ = c.buffers()
    ctx.synchronize()
    dev = torch.device("cuda", ctx.device)
    planes = tensor_from_ptr(i32, n_i32, torch.int32, dev).cpu().numpy().reshape(-1, n, n)
    H3 = planes[5:9] if planes.shape[0] >= 9 else np.zeros((4, n, n), np.int32)
    spill = tensor_from_ptr(f64, n_f64, torch.float64, dev).cpu().numpy().reshape(n, n) if n_f64 else np.zeros((n, n))
    upper = np.triu(np.ones((n, n), bool), 1)
    return np.where(upper, H3, 0), np.where(upper, spill, 0.0)


def check_exact(ctx, c, o, exp):
    S1, D1, H, hist = c.download()
    assert np.array_equal(S1, o.S1), "S1 differs"
    assert np.array_equal(D1, o.D1), "D1 differs"
    assert np.array_equal(H, o.H), "order-2 planes differ"
    assert np.array_equal(hist, multi_hist(o)), "class histogram differs"
    H3, spill = read_planes(ctx, c)
    assert np.array_equal(H3, exp.H3), "order-3 planes differ"
    assert not np.isnan(spill).any()
    # fp64 atomics add in any order, and G cancels the large x F(1,0) terms: bound by the terms, not by the result
    assert (np.abs(spill - exp.spill) <= 1e-12 * exp.terms).all(), np.abs(spill - exp.spill).max()


@pytest.mark.gpu
@pytest.mark.parametrize("threads", [1, 8])
@pytest.mark.parametrize("second", ["enum", "gemm"])
@pytest.mark.parametrize("path", ["scatter", "gemm"])
@pytest.mark.parametrize("name", sorted(DESIGNS))
def test_planted_classes(gpu_ctx, monkeypatch, name, path, second, threads):
    monkeypatch.setenv("SECEDO_B200_SECOND_ORDER", second)
    L, windows = DESIGNS[name]
    p, exp = planted_pileup(L, windows)
    o = oracle(p, L, threads)
    ident = np.arange(N_CELLS, dtype=np.uint32)
    c = api.Counts(gpu_ctx, N_CELLS)
    st = c.accumulate(p, L, ident, *PARAMS, threads, path)
    check_exact(gpu_ctx, c, o, exp)
    assert st["n_pairs_multi"] == int(exp.hist.sum())
    for norm in ("ADD_MIN", "EXPONENTIATE", "SCALE_MAX_1"):
        assert_matrix_close(c.finalize(L, *PARAMS, norm), po.normalize(o.raw, norm), TOL)
    c.free()


@pytest.mark.gpu
@pytest.mark.parametrize("second", ["enum", "gemm"])
@pytest.mark.parametrize("path", ["scatter", "gemm"])
@pytest.mark.parametrize("L,cls,accepted", REFUSALS)
def test_refusal_parity(gpu_ctx, monkeypatch, L, cls, accepted, path, second):
    """SGPU_E_CLASS_RANGE exactly where the oracle cannot evaluate the class"""
    monkeypatch.setenv("SECEDO_B200_SECOND_ORDER", second)
    p, exp = planted_pileup(L, refusal_design(L, cls))
    ident = np.arange(N_CELLS, dtype=np.uint32)
    c = api.Counts(gpu_ctx, N_CELLS)
    if accepted:
        c.accumulate(p, L, ident, *PARAMS, 1, path)
        check_exact(gpu_ctx, c, oracle(p, L, 1), exp)
    else:
        with pytest.raises(api.SgpuError) as e:
            c.accumulate(p, L, ident, *PARAMS, 1, path)
        assert e.value.code == SGPU_E_CLASS_RANGE
    c.free()


@pytest.mark.gpu
@pytest.mark.parametrize("second", ["enum", "gemm"])
@pytest.mark.parametrize("path", ["scatter", "gemm"])
def test_refused_accumulation_needs_zero(gpu_ctx, monkeypatch, path, second):
    """a pair refused by the multi-locus correction comes after the first-order counts and the other pairs' order-2 and
    order-3 counts have been issued: the object refuses further accumulations until zeroed, and the zeroing clears every
    plane, so the next accumulation starts from nothing"""
    monkeypatch.setenv("SECEDO_B200_SECOND_ORDER", second)
    good = small_classes()[:10]
    assert {w[2] + w[3] for w in good} >= {2, 3}
    p_bad, _ = planted_pileup(1000, good + [(3, 8, 64, 0)])
    p_good, exp = planted_pileup(1000, good)
    ident = np.arange(N_CELLS, dtype=np.uint32)
    c = api.Counts(gpu_ctx, N_CELLS)
    with pytest.raises(api.SgpuError) as e:
        c.accumulate(p_bad, 1000, ident, *PARAMS, 1, path)
    assert e.value.code == SGPU_E_CLASS_RANGE
    for _ in range(2):
        with pytest.raises(api.SgpuError) as e:
            c.accumulate(p_good, 1000, ident, *PARAMS, 1, path)
        assert e.value.code == SGPU_E_ARG
    c.zero()
    c.accumulate(p_good, 1000, ident, *PARAMS, 1, path)
    check_exact(gpu_ctx, c, oracle(p_good, 1000, 1), exp)
    c.free()


LOG_PROB_L = [2, 3, 4, 5, 12, 40, 63, 64, 65, 100, 126, 127, 128, 132, 133, 1000]


@pytest.mark.parametrize("L", LOG_PROB_L)
def test_cut_log_prob_tables_are_the_oracles(L):
    """oracle_log_probs against the oracle itself on the leading 24 x 24 block (the oracle evaluates that in well under
    a second): same values bit for bit, NaN where the oracle's tables end (here from s + d >= L for L <= 40)"""
    n = min(24, L)
    for e, h, t in warm_log_probs():
        want = po.log_probs(e, h, t, L, n)
        got = oracle_log_probs(e, h, t, L)
        for a, b in zip(got, want):
            assert np.array_equal(a[:n, :n], b, equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("L", LOG_PROB_L)
def test_log_prob_tables_up_to_64(gpu_ctx, L):
    """LS and LD up to n = min(64, L) for the parameter sets of the golden tables: the same NaN mask (classes past the
    power tables), and the same values up to the last bits of log() (the summation order is the reference's). F = LD -
    LS is not compared: it cancels to ~1e-14 for some high classes."""
    for e, h, t in warm_log_probs():
        ls, ld = api.log_probs(e, h, t, L, min(MAX_CLASS, L), ctx=gpu_ctx)
        ols, old = oracle_log_probs(e, h, t, L)
        assert np.array_equal(np.isnan(ls), np.isnan(ols)) and np.array_equal(np.isnan(ld), np.isnan(old))
        ok = ~np.isnan(ols)
        assert np.allclose(ls[ok], ols[ok], rtol=1e-13, atol=0)
        assert np.allclose(ld[ok], old[ok], rtol=1e-13, atol=0)
