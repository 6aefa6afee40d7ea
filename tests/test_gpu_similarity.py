"""Parity of the CUDA similarity-matrix path (through the C ABI) with the oracle and with golden
matrices from the compiled reference. Integer read-pair counts are compared bit-exactly; the final
fp64 matrix within 1e-6 * max|M| (north_star tolerance; SURVEY.md §8c explains the scaling)."""
import numpy as np
import pytest

from conftest import assert_matrix_close, golden_pileup, load_golden
from oracle import pyoracle as po
from secedo_b200 import api
from secedo_b200.pileup import NO_POS, Pileup
from secedo_b200.synth import SynthConfig, make_pileup

pytestmark = pytest.mark.gpu
TOL = 1e-6
PATHS = ["scatter", "gemm"]

CASES = ["sim_ten_rows", "sim_six_cells", "sim_three_rows", "sim_reference_test_style", "sim_synth_multi",
         "sim_synth_subcluster"]


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("name", CASES)
def test_golden_matrices(gpu_ctx, name, path):
    g = load_golden(name)
    p = golden_pileup(g)
    for t in g["threads"]:
        for norm in g["norms"]:
            M = api.compute_similarity_matrix(p, int(g["num_cells"]), int(g["L"]), g["gmap"], float(g["eps"]),
                                              float(g["h"]), float(g["theta"]), int(t), "", str(norm), ctx=gpu_ctx,
                                              path=path)
            assert_matrix_close(M, g[f"M_t{t}_{norm}"], TOL)


@pytest.mark.parametrize("path", PATHS)
def test_read_id_chained_over_fragment_length(gpu_ctx, path, monkeypatch):
    """ADVICE r1: a read id chained over >= max_fragment_length (long-insert pair with kept loci in between) must not
    abort a drop-in run. The chain is split where the reference retires the read; checked against the COMPILED REFERENCE
    (golden) and, count for count, against the oracle on the relabelled pileup. SECEDO_B200_STRICT_SPAN=1 keeps the error."""
    g = load_golden("sim_span_chain")
    p = golden_pileup(g)
    args = (int(g["num_cells"]), int(g["L"]), g["gmap"], float(g["eps"]), float(g["h"]), float(g["theta"]))
    split = Pileup(p.chr_ptr, p.row_ptr, p.position, g["split_read_id"], p.gid_base)
    for t in g["threads"]:
        M = api.compute_similarity_matrix(p, *args, int(t), "", "ADD_MIN", ctx=gpu_ctx, path=path)
        assert_matrix_close(M, g[f"M_t{t}_ADD_MIN"], TOL)
        o = po.similarity(split, *args, int(t))
        c = api.Counts(gpu_ctx, args[0])
        st = c.accumulate(p, args[1], args[2], args[3], args[4], args[5], int(t), path)
        S1, D1, H, _ = c.download()
        assert np.array_equal(S1, o.S1) and np.array_equal(D1, o.D1) and np.array_equal(H, o.H)
        assert st["n_span_splits"] == np.unique(split.read_id[p.read_id != split.read_id]).size - 1
        c.free()
    monkeypatch.setenv("SECEDO_B200_STRICT_SPAN", "1")
    with pytest.raises(api.SgpuError):
        api.compute_similarity_matrix(p, *args, 1, "", "ADD_MIN", ctx=gpu_ctx, path=path)


def check_counts(ctx, f, n_cells, L, gmap, eps, h, theta, threads, path):
    o = po.similarity(f, n_cells, L, gmap, eps, h, theta, threads, "ADD_MIN")
    c = api.Counts(ctx, n_cells)
    st = c.accumulate(f, L, gmap, eps, h, theta, threads, path)
    S1, D1, H, hist = c.download()
    assert np.array_equal(S1, o.S1), "S1 (same-base incidences) differs"
    assert np.array_equal(D1, o.D1), "D1 (different-base incidences) differs"
    assert np.array_equal(H, o.H), "second-order class counts differ"
    oh = o.class_hist.copy()
    oh[0, 0] = oh[0, 1] = oh[1, 0] = 0
    assert np.array_equal(hist, oh), "overlap class histogram differs"
    assert st["n_pairs_multi"] == int(oh.sum())
    for norm in ("ADD_MIN", "EXPONENTIATE", "SCALE_MAX_1"):
        M = c.finalize(L, eps, h, theta, norm)
        assert_matrix_close(M, po.normalize(o.raw, norm), TOL)
    c.free()
    return st, o


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("threads", [1, 2, 8])
def test_counts_bit_exact_multilocus(gpu_ctx, threads, path):
    cfg = SynthConfig(n_cells=60, coverage=0.3, n_loci=900, n_chr=3, p_multi=0.45, p_mate=0.15, theta=0.02, seed=7)
    p = make_pileup(cfg)
    ident = np.arange(cfg.n_cells, dtype=np.uint32)
    f, _ = api.Filter(0.01, 4, gpu_ctx).filter(p, ident, "", 1)
    st, o = check_counts(gpu_ctx, f, cfg.n_cells, 1000, ident, 0.01, 0.5, 0.01, threads, path)
    assert st["n_multi_reads"] > 0 and st["n_dropped_entries"] > 0 and st["n_tail_reads"] > 0


@pytest.mark.parametrize("path", PATHS)
def test_cfg1_style_500_cells(gpu_ctx, path):
    """BASELINE.json configs[0] shape: 500 cells, 0.05x, one chromosome (scaled to a few seconds of oracle)."""
    cfg = SynthConfig(n_cells=500, coverage=0.05, n_loci=20000, n_chr=1, p_multi=0.05, p_mate=0.02, seed=21)
    p = make_pileup(cfg)
    ident = np.arange(cfg.n_cells, dtype=np.uint32)
    f, _ = api.Filter(0.01, 4, gpu_ctx).filter(p, ident, "", 1)
    assert f.n_loci > 1000
    check_counts(gpu_ctx, f, cfg.n_cells, 1000, ident, 0.01, 0.5, 0.01, 8, path)


@pytest.mark.parametrize("path", PATHS)
def test_cfg2_style_2000_cells(gpu_ctx, path):
    """configs[1] shape: 2000 cells at 0.1x (prefix of loci the oracle finishes in seconds)."""
    cfg = SynthConfig(n_cells=2000, coverage=0.1, n_loci=1500, n_chr=2, p_multi=0.03, p_mate=0.02, theta=0.001,
                      seed=22)
    p = make_pileup(cfg)
    ident = np.arange(cfg.n_cells, dtype=np.uint32)
    f, _ = api.Filter(0.001, 4, gpu_ctx).filter(p, ident, "", 1)
    check_counts(gpu_ctx, f, cfg.n_cells, 1000, ident, 0.01, 0.15, 0.001, 8, path)


@pytest.mark.parametrize("path", PATHS)
def test_subcluster_remap(gpu_ctx, path):
    """second recursion level: cells outside the sub-cluster map to NO_POS, the rest to 0..n-1"""
    cfg = SynthConfig(n_cells=300, coverage=0.2, n_loci=2500, n_chr=2, n_clones=4, p_multi=0.1, p_mate=0.05, seed=23)
    p = make_pileup(cfg)
    rng = np.random.default_rng(5)
    members = np.sort(rng.choice(cfg.n_cells, 170, replace=False))
    gmap = np.full(cfg.n_cells, NO_POS, np.uint32)
    gmap[members] = np.arange(members.size)
    f, _ = api.Filter(0.01, 4, gpu_ctx).filter(p, gmap, "", 1)
    check_counts(gpu_ctx, f, members.size, 1000, gmap, 0.01, 0.5, 0.01, 4, path)


def test_high_order_overlaps(gpu_ctx):
    """fragments covering up to 6 close loci: classes of order >= 4 go through the fp64 spill plane"""
    cfg = SynthConfig(n_cells=25, coverage=1.5, n_loci=300, n_chr=1, spacing=40, p_multi=0.9, p_mate=0.1, seed=31)
    p = make_pileup(cfg)
    ident = np.arange(cfg.n_cells, dtype=np.uint32)
    st, o = check_counts(gpu_ctx, p, cfg.n_cells, 1000, ident, 0.01, 0.5, 0.01, 1, "scatter")
    hi = o.class_hist.copy()
    hi[:4, :4][np.add.outer(np.arange(4), np.arange(4)) < 4] = 0
    assert hi.sum() > 0, "the case must contain overlaps of order >= 4"


def test_edge_cases(gpu_ctx):
    ident = np.arange(4, dtype=np.uint32)
    # empty pileup, with and without chromosomes
    for p in (Pileup.empty(0), Pileup.empty(3)):
        M = api.compute_similarity_matrix(p, 4, 1000, ident, 0.01, 0.5, 0.01, 1, "", "ADD_MIN", ctx=gpu_ctx)
        assert M.shape == (4, 4) and not M.any()
    # a single locus: everything is tail -> zero
    p = Pileup.from_pos_data([[(5, [1, 2, 3], [0 << 2, (1 << 2) | 1, 2 << 2])]])
    assert not api.compute_similarity_matrix(p, 4, 1000, ident, 0.01, 0.5, 0.01, 1, ctx=gpu_ctx).any()
    # invalid normalization -> the reference throws std::logic_error
    with pytest.raises(ValueError):
        api.compute_similarity_matrix(p, 4, 1000, ident, 0.01, 0.5, 0.01, 1, "", "NOPE", ctx=gpu_ctx)
    # a read id that recurs >= L bp later with nothing in between is a new read (what the reference does
    # once the first one has been retired; the oracle calls the input undefined): same result as renaming
    loci = [(100 + 40 * i, [10 + i, 50 + i], [0 << 2, (1 << 2) | 1]) for i in range(30)]
    far = loci + [(5000, [10, 99], [2 << 2, 3 << 2]), (5100, [98, 97], [2 << 2, 3 << 2])]
    ren = loci + [(5000, [777, 99], [2 << 2, 3 << 2]), (5100, [98, 97], [2 << 2, 3 << 2])]
    Ma = api.compute_similarity_matrix(Pileup.from_pos_data([far]), 4, 1000, ident, 0.01, 0.5, 0.01, 1, ctx=gpu_ctx)
    Mb = api.compute_similarity_matrix(Pileup.from_pos_data([ren]), 4, 1000, ident, 0.01, 0.5, 0.01, 1, ctx=gpu_ctx)
    assert np.array_equal(Ma, Mb) and Ma.any()
    assert_matrix_close(Mb, po.similarity(Pileup.from_pos_data([ren]), 4, 1000, ident, 0.01, 0.5, 0.01, 1).M, TOL)
    # a read id chained over >= L bp through intermediate loci: split where the reference retires the read (start + L <=
    # position: the entry at 1300 opens a new read); same result as renaming that entry
    chain = [[(100, [1, 2], [0 << 2, 1 << 2]), (700, [1, 3], [0 << 2, 2 << 2]), (1300, [1, 4], [0 << 2, 2 << 2]),
              (1400, [5, 6], [1 << 2, 3 << 2]), (2600, [7, 8], [1 << 2, 3 << 2])]]
    renamed = [[(100, [1, 2], [0 << 2, 1 << 2]), (700, [1, 3], [0 << 2, 2 << 2]), (1300, [901, 4], [0 << 2, 2 << 2]),
                (1400, [5, 6], [1 << 2, 3 << 2]), (2600, [7, 8], [1 << 2, 3 << 2])]]
    Mc = api.compute_similarity_matrix(Pileup.from_pos_data(chain), 4, 1000, ident, 0.01, 0.5, 0.01, 1, ctx=gpu_ctx)
    Mr = api.compute_similarity_matrix(Pileup.from_pos_data(renamed), 4, 1000, ident, 0.01, 0.5, 0.01, 1, ctx=gpu_ctx)
    assert np.array_equal(Mc, Mr)
    assert_matrix_close(Mr, po.similarity(Pileup.from_pos_data(renamed), 4, 1000, ident, 0.01, 0.5, 0.01, 1).M, TOL)
    # cell outside the matrix
    p = Pileup.from_pos_data([[(100, [1, 2], [0 << 2, 3 << 2])]])
    with pytest.raises(api.SgpuError):
        api.compute_similarity_matrix(p, 2, 1000, ident, 0.01, 0.5, 0.01, 1, ctx=gpu_ctx)


def test_log_prob_tables(gpu_ctx):
    g = load_golden("log_probs")
    i = 0
    while f"params{i}" in g.files:
        e, h, t, L = g[f"params{i}"]
        n = g[f"ls{i}"].shape[0]
        ls, ld = api.log_probs(e, h, t, int(L), n, ctx=gpu_ctx)
        ok = ~np.isnan(g[f"ls{i}"])
        # identical formula and summation order, -fmad=false; CUDA's log() may differ by an ulp
        assert np.allclose(ls[ok], g[f"ls{i}"][ok], rtol=1e-14, atol=0) and np.allclose(ld[ok], g[f"ld{i}"][ok], rtol=1e-14, atol=0)
        i += 1


def test_linearity_and_idempotence(gpu_ctx):
    """size-independent properties: counts(A ++ B) == counts(A) + counts(B) for disjoint chromosome
    sets; accumulating in two calls equals one call; the result is symmetric with a zero diagonal."""
    cfg = SynthConfig(n_cells=400, coverage=0.3, n_loci=3000, n_chr=4, p_multi=0.05, p_mate=0.02, seed=41)
    p = make_pileup(cfg)
    ident = np.arange(cfg.n_cells, dtype=np.uint32)
    f, _ = api.Filter(0.01, 4, gpu_ctx).filter(p, ident, "", 1)
    halves = []
    for chrs in ((0, 1), (2, 3)):
        parts = [f.loci_range(c, 0, 1 << 40) for c in chrs]
        halves.append(Pileup.concat(parts))
    args = (1000, ident, 0.01, 0.5, 0.01, 8)
    whole = api.Counts(gpu_ctx, cfg.n_cells)
    whole.accumulate(f, *args, path="scatter")
    two = api.Counts(gpu_ctx, cfg.n_cells)
    two.accumulate(halves[0], *args, path="scatter")
    two.accumulate(halves[1], *args, path="gemm")
    a, b = whole.download(), two.download()
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    M = whole.finalize(1000, 0.01, 0.5, 0.01, "ADD_MIN")
    assert np.array_equal(M, M.T) and not np.diag(M).any() and M.min() == 0.0


@pytest.mark.parametrize("path", PATHS)
def test_device_generated_pileup(gpu_ctx, path):
    """the bench input generator (csrc/synth.cu): download a generated pileup and replay it through the
    oracle — validates the generator (increasing positions, fragment spans < L, mate duplicates,
    two-locus fragments) and the whole path on exactly the kind of data bench.py times"""
    dev = gpu_ctx.synth_pileup(700, 0.4, 3, 500, n_clones=2, theta=0.001, p_multi=0.08, p_mate=0.05, seed=9)
    p = dev.download()
    assert p.n_chr == 3 and p.n_loci == 1500
    ident = np.arange(700, dtype=np.uint32)
    kl, ke, _, cov64 = po.filter_flags(p, ident, 0.001)
    fdev, cov = api.Filter(0.001, 4, gpu_ctx).filter_device(dev, ident)
    f = fdev.download()
    assert f == p.select(kl, ke) and cov == cov64
    assert 200 < f.n_loci < 1300
    st, o = check_counts(gpu_ctx, f, 700, 1000, ident, 0.01, 0.15, 0.001, 8, path)
    assert st["n_multi_reads"] > 0 and st["n_dropped_entries"] > 0 and st["n_pairs_multi"] > 0


@pytest.mark.parametrize("path", PATHS)
def test_filtered_view_of_read_ids(gpu_ctx, path, monkeypatch):
    """at the root of the recursion (every group in the sub-cluster) the filter does not copy the read ids: the filtered
    pileup reads them through a view of the unfiltered one (sgpu_pileup::view_read_id). The read linking must see the same
    ids through the view, the source must outlive its views (it is freed FIRST here), and a download gathers them."""
    ident = np.arange(700, dtype=np.uint32)
    dev = gpu_ctx.synth_pileup(700, 0.4, 3, 500, n_clones=2, theta=0.001, p_multi=0.08, p_mate=0.05, seed=19)
    p = dev.download()
    kl, ke, _, _ = po.filter_flags(p, ident, 0.001)
    want = p.select(kl, ke)
    o = po.similarity(want, 700, 1000, ident, 0.01, 0.15, 0.001, 8, "ADD_MIN")
    flt = api.Filter(0.001, 4, gpu_ctx)
    fdev, _ = flt.filter_device(dev, ident)
    dev.free()  # the view keeps the source's read ids alive
    c = api.Counts(gpu_ctx, 700)
    st = c.accumulate(fdev, 1000, ident, 0.01, 0.15, 0.001, 8, path)
    S1, D1, H, _ = c.download()
    assert np.array_equal(S1, o.S1) and np.array_equal(D1, o.D1) and np.array_equal(H, o.H)
    assert st["n_multi_reads"] > 0 and st["n_dropped_entries"] > 0
    assert fdev.download() == want  # gathers the ids; the deferred free of the source happens here
    c.zero()
    c.accumulate(fdev, 1000, ident, 0.01, 0.15, 0.001, 8, path)  # now from the pileup's own ids
    S2, D2, H2, _ = c.download()
    assert np.array_equal(S2, o.S1) and np.array_equal(D2, o.D1) and np.array_equal(H2, o.H)
    fdev.free()
    # a sub-cluster (some groups outside) always copies; so does SECEDO_B200_FILTER_VIEW=0
    dev = gpu_ctx.synth_pileup(700, 0.4, 3, 500, n_clones=2, theta=0.001, p_multi=0.08, p_mate=0.05, seed=19)
    monkeypatch.setenv("SECEDO_B200_FILTER_VIEW", "0")
    f0, _ = flt.filter_device(dev, ident)
    assert f0.download() == want
    f0.free()
    monkeypatch.delenv("SECEDO_B200_FILTER_VIEW")
    sub = ident.copy()
    sub[::3] = NO_POS
    kl, ke, _, _ = po.filter_flags(p, sub, 0.001)
    fs, _ = flt.filter_device(dev, sub)
    assert fs.download() == p.select(kl, ke)
    fs.free()
    # filtering a filtered pileup that still reads through a view
    f1, _ = flt.filter_device(dev, ident)
    f2, _ = flt.filter_device(f1, ident)
    assert f2.download() == want
    for x in (f1, f2, dev):
        x.free()
    c.free()


def test_scheduling_options_do_not_change_results():
    """the tensor kernel beside the next batch (own stream, held-back launch, cache preference): whatever the knobs say, a
    filter -> accumulate loop over several batches gives the same count planes and the same matrix, and they are the
    oracle's; the knobs of earlier versions and out-of-range values are refused"""
    ctx = api.Context(0)
    n = 1536
    ident = np.arange(n, dtype=np.uint32)
    devs = [ctx.synth_pileup(n, 0.4, 2, 700, theta=0.001, p_multi=0.03, p_mate=0.02, seed=90 + k) for k in range(3)]
    flt = api.Filter(0.001, 4, ctx)
    want = None
    for fd in devs:
        f = flt.filter_device(fd, ident)[0].download()
        o = po.similarity(f, n, 1000, ident, 0.01, 0.15, 0.001, 8, "ADD_MIN")
        want = [o.S1, o.D1, o.H] if want is None else [want[0] + o.S1, want[1] + o.D1, want[2] + o.H]
    c = api.Counts(ctx, n)
    first_M = None
    for knobs in ({"async_gemm": 0}, {"async_gemm": 1, "prefer_shared": 0}, {"prefer_shared": 1}):
        for k, v in knobs.items():
            ctx.set_option(k, v)
        c.zero()
        for fd in devs:
            f, _ = flt.filter_device(fd, ident)
            c.accumulate(f, 1000, ident, 0.01, 0.15, 0.001, 8, "gemm")
            f.free()
        M = c.finalize(1000, 0.01, 0.15, 0.001, "ADD_MIN")
        S1, D1, H, _ = c.download()
        assert np.array_equal(S1, want[0]) and np.array_equal(D1, want[1]) and np.array_equal(H, want[2]), knobs
        if first_M is None:
            first_M = M
        assert np.array_equal(M, first_M), knobs
    for name, value in (("no_such_knob", 1), ("late_gemm", 1), ("gemm_stages", 5), ("win_smem_kb", 60), ("prefer_shared", 2)):
        with pytest.raises(api.SgpuError):
            ctx.set_option(name, value)
    c.free()
    for fd in devs:
        fd.free()
    ctx.close()


def test_two_counts_objects_interleaved(gpu_ctx):
    """the tensor kernel of an accumulation is held back until the next batch's read linking has been issued, and a join only
    concerns the planes it is asked for: a caller that alternates between two counts objects (bench.py's pipelined steps)
    must get each object's own sums, whatever is still in flight or held back for the other one"""
    ident = np.arange(1024, dtype=np.uint32)
    devs = [gpu_ctx.synth_pileup(1024, 0.5, 1, 1500, theta=0.001, p_multi=0.02, p_mate=0.02, seed=70 + k) for k in range(3)]
    flt = api.Filter(0.001, 4, gpu_ctx)
    fs = [flt.filter_device(d, ident)[0] for d in devs]
    args = (1000, ident, 0.01, 0.15, 0.001, 8, "gemm")
    single = []
    for f in fs:  # each batch alone
        c = api.Counts(gpu_ctx, 1024)
        c.accumulate(f, *args)
        single.append(c.download())
        c.free()
    a, b = api.Counts(gpu_ctx, 1024), api.Counts(gpu_ctx, 1024)
    a.accumulate(fs[0], *args)          # a: batch 0 (kernel held back)
    b.accumulate(fs[1], *args)          # b: batch 1 (a's kernel issued behind b's read linking, b's held back)
    Ma = a.finalize(1000, 0.01, 0.15, 0.001, "ADD_MIN")   # concerns a only
    b.accumulate(fs[2], *args)          # b: + batch 2
    a.zero()
    a.accumulate(fs[2], *args)
    got_b, got_a = b.download(), a.download()
    for k in range(3):
        assert np.array_equal(got_b[k], single[1][k] + single[2][k])
        assert np.array_equal(got_a[k], single[2][k])
    one = api.Counts(gpu_ctx, 1024)
    one.accumulate(fs[0], *args)
    assert np.array_equal(Ma, one.finalize(1000, 0.01, 0.15, 0.001, "ADD_MIN"))
    for x in (a, b, one, *fs, *devs):
        x.free()


def test_auto_path_and_stats(gpu_ctx):
    dev = gpu_ctx.synth_pileup(1024, 0.5, 1, 4000, theta=0.001, p_multi=0.01, seed=4)
    ident = np.arange(1024, dtype=np.uint32)
    fdev, _ = api.Filter(0.001, 4, gpu_ctx).filter_device(dev, ident)
    c = api.Counts(gpu_ctx, 1024)
    n0 = gpu_ctx.launch_count()
    gpu_ctx.tensor_times()  # forget the tensor kernels of earlier tests
    st = c.accumulate(fdev, 1000, ident, 0.01, 0.15, 0.001, 8, "auto")
    # the tensor kernel runs on its own stream: it is reported by the call during which it finishes, or by tensor_times()
    ms_left, n_left = gpu_ctx.tensor_times()
    assert st["path_used"] == "gemm" and st["gemm_launches"] + n_left == 1 and st["ms_gemm"] + ms_left > 0
    assert gpu_ctx.launch_count() > n0
    # the ultra-sparse end of the cost model (profiles/r1_path_crossover.txt): ~40 reads over 8000 cells per locus
    sparse = gpu_ctx.synth_pileup(8000, 0.005, 1, 2048, theta=0.001, seed=4)
    c2 = api.Counts(gpu_ctx, 8000)
    st2 = c2.accumulate(sparse, 1000, np.arange(8000, dtype=np.uint32), 0.01, 0.15, 0.001, 8, "auto")
    assert st2["path_used"] == "scatter"
    c2.free()


@pytest.mark.parametrize("n_cells,coverage,loci_per_chr", [(8000, 0.5, 384), (10000, 0.05, 4096), (16000, 0.25, 96)])
def test_full_size_paths_agree(gpu_ctx, n_cells, coverage, loci_per_chr):
    """BASELINE.json's cell counts (cfg3: 8 000 cells at 0.5x, cfg4: 10 000 cells at 0.05x, and the largest
    matrix the 14-bit group id allows) on device-generated pileups, too large for the oracle: the tcgen05
    GEMM path and the pair-scatter path — two independent implementations of the first-order counts — must
    agree bit for bit, counts must add up over disjoint chromosome sets, and the matrix is symmetric with
    a zero diagonal and minimum 0 (ADD_MIN)."""
    dev = gpu_ctx.synth_pileup(n_cells, coverage, 2, loci_per_chr, n_clones=4, theta=0.001, p_multi=0.01, p_mate=0.01, seed=13)
    ident = np.arange(n_cells, dtype=np.uint32)
    fdev, _ = api.Filter(0.001, 4, gpu_ctx).filter_device(dev, ident)
    assert fdev.n_loci > loci_per_chr // 4
    args = (1000, ident, 0.01, 0.5, 0.001, 8)
    res = {}
    for path in ("gemm", "scatter"):
        c = api.Counts(gpu_ctx, n_cells)
        st = c.accumulate(fdev, *args, path=path)
        res[path] = c.download()
        if path == "gemm":
            M = c.finalize(1000, 0.01, 0.5, 0.001, "ADD_MIN")
            assert np.array_equal(M, M.T) and not np.diag(M).any() and M.min() == 0.0 and np.isfinite(M).all()
            assert st["n_multi_reads"] > 0 and st["n_dropped_entries"] > 0 and st["n_tail_reads"] > 0
        c.free()
    for a, b, name in zip(res["gemm"], res["scatter"], ("S", "D", "H", "hist")):
        assert np.array_equal(a, b), f"{name} differs between the GEMM and the scatter path"
    assert res["gemm"][0].sum() > 0 and res["gemm"][1].sum() > 0
    # linearity over chromosomes: the two chromosomes one after the other == both at once
    f = fdev.download()
    two = api.Counts(gpu_ctx, n_cells)
    for c_ in range(2):
        two.accumulate(f.loci_range(c_, 0, 1 << 40), *args, path="gemm")
    for a, b in zip(res["gemm"], two.download()):
        assert np.array_equal(a, b)
    two.free()


@pytest.mark.parametrize("path", PATHS)
def test_cfg3_full_cell_count_vs_oracle(gpu_ctx, path):
    """BASELINE.json configs[2] at its REAL cell count: 8 000 cells at 0.5x (about 4 000 reads per locus, 8 M cross-cell
    pairs per locus) with the multi-locus share SURVEY F1 measured on the reference's own fixture (16 % of reads cover
    >= 2 loci) and the reference's flags_sim likelihood parameters, on a locus prefix the enumerating oracle finishes in
    ~20 s: integer counts bit-exact, matrix within 1e-6 * max|M| for all three normalisations."""
    cfg = SynthConfig(n_cells=8000, coverage=0.5, n_loci=30, n_chr=1, p_multi=0.16, p_mate=0.02, theta=0.001, seed=5)
    p = make_pileup(cfg)
    ident = np.arange(cfg.n_cells, dtype=np.uint32)
    f, _ = api.Filter(0.001, 4, gpu_ctx).filter(p, ident, "", 1)
    assert f.n_loci >= 10
    st, o = check_counts(gpu_ctx, f, cfg.n_cells, 1000, ident, 0.01, 0.15, 0.001, 8, path)
    assert st["n_multi_reads"] > 1000 and st["n_tail_reads"] > 0 and o.H.sum() > 0


@pytest.mark.parametrize("path", PATHS)
def test_cfg4_full_cell_count_vs_oracle(gpu_ctx, path):
    """configs[3] at its real cell count: 10 000 cells at 0.05x, 4 clones, flags_breast parameters (h = 0.5,
    theta = 0.001, eps = 0.01), ~600 pre-filter loci: counts bit-exact against the oracle, matrix within tolerance."""
    cfg = SynthConfig(n_cells=10000, coverage=0.05, n_loci=600, n_chr=2, n_clones=4, p_multi=0.16, p_mate=0.02,
                      theta=0.001, seed=6)
    p = make_pileup(cfg)
    ident = np.arange(cfg.n_cells, dtype=np.uint32)
    f, _ = api.Filter(0.001, 4, gpu_ctx).filter(p, ident, "", 1)
    assert f.n_loci >= 300
    st, o = check_counts(gpu_ctx, f, cfg.n_cells, 1000, ident, 0.01, 0.5, 0.001, 8, path)
    assert st["n_multi_reads"] > 1000 and o.H.sum() > 0


@pytest.mark.parametrize("threads", [1, 2, 8])
def test_second_order_gemm_vs_oracle(gpu_ctx, threads, monkeypatch):
    """the pairs that overlap at two loci counted by the tcgen05 path on the derived pileup of locus pairs
    (forced; by default it only takes over from a few hundred multi-locus reads per locus): exact against
    the oracle incl. mate duplicates, the tail rule and fragments of up to 6 loci, whose pairs of order >= 3
    are enumerated and taken back out of the second-order planes"""
    monkeypatch.setenv("SECEDO_B200_SECOND_ORDER", "gemm")
    ident = np.arange(60, dtype=np.uint32)
    cfg = SynthConfig(n_cells=60, coverage=0.3, n_loci=900, n_chr=3, p_multi=0.45, p_mate=0.15, theta=0.02, seed=7)
    f, _ = api.Filter(0.01, 4, gpu_ctx).filter(make_pileup(cfg), ident, "", 1)
    st, o = check_counts(gpu_ctx, f, 60, 1000, ident, 0.01, 0.5, 0.01, threads, "gemm")
    assert st["n_multi_reads"] > 0 and st["n_tail_reads"] > 0 and st["n_pairs_multi"] > 0
    cfg = SynthConfig(n_cells=25, coverage=1.5, n_loci=300, n_chr=1, spacing=40, p_multi=0.9, p_mate=0.1, seed=31)
    ident = np.arange(25, dtype=np.uint32)
    st, o = check_counts(gpu_ctx, make_pileup(cfg), 25, 1000, ident, 0.01, 0.5, 0.01, threads, "gemm")
    hi = o.class_hist.copy()
    hi[:3, :3][np.add.outer(np.arange(3), np.arange(3)) < 3] = 0
    assert hi.sum() > 0, "the case must contain overlaps of order >= 3"


def test_second_order_gemm_vs_enumeration_full_size(gpu_ctx, monkeypatch):
    """8 000 cells, 20 % two-locus fragments (the share seen in real pileups): both ways of counting the
    second-order pairs agree bit for bit, on both first-order paths' worth of planes"""
    dev = gpu_ctx.synth_pileup(8000, 0.5, 2, 192, n_clones=4, theta=0.001, p_multi=0.2, p_mate=0.05, seed=17)
    ident = np.arange(8000, dtype=np.uint32)
    fdev, _ = api.Filter(0.001, 4, gpu_ctx).filter_device(dev, ident)
    res = {}
    for mode in ("enum", "gemm"):
        monkeypatch.setenv("SECEDO_B200_SECOND_ORDER", mode)
        c = api.Counts(gpu_ctx, 8000)
        st = c.accumulate(fdev, 1000, ident, 0.01, 0.5, 0.001, 8, "gemm")
        res[mode] = c.download() + (st["n_pairs_multi"],)
        c.free()
    for a, b, name in zip(res["enum"], res["gemm"], ("S", "D", "H", "hist", "n_pairs_multi")):
        assert np.array_equal(a, b), name
    assert res["gemm"][2].sum() > 0 and res["gemm"][4] > 10 ** 6


def test_async_upload_pipeline(gpu_ctx):
    """chromosome by chromosome with asynchronous uploads running ahead of the kernels (the end-to-end
    path of bench.py): same counts as one synchronous call on the whole pileup"""
    cfg = SynthConfig(n_cells=350, coverage=0.3, n_loci=2400, n_chr=4, p_multi=0.08, p_mate=0.04, seed=71)
    p = make_pileup(cfg)
    ident = np.arange(cfg.n_cells, dtype=np.uint32)
    flt = api.Filter(0.01, 4, gpu_ctx)
    args = (1000, ident, 0.01, 0.5, 0.01, 8)
    whole = api.Counts(gpu_ctx, cfg.n_cells)
    f_all, _ = flt.filter_device(p, ident)
    whole.accumulate(f_all, *args, path="gemm")
    parts = [p.loci_range(c, 0, 1 << 40) for c in range(p.n_chr)]
    piped = api.Counts(gpu_ctx, cfg.n_cells)
    queue = [gpu_ctx.upload_async(parts[0]), gpu_ctx.upload_async(parts[1])]
    for c in range(p.n_chr):
        cur = queue.pop(0)
        if c + 2 < p.n_chr:
            queue.append(gpu_ctx.upload_async(parts[c + 2]))
        f, _ = flt.filter_device(cur, ident)
        piped.accumulate(f, *args, path="gemm")
        f.free()
        cur.free()
    for x, y in zip(whole.download(), piped.download()):
        assert np.array_equal(x, y)
    assert np.array_equal(whole.finalize(1000, 0.01, 0.5, 0.01, "ADD_MIN"), piped.finalize(1000, 0.01, 0.5, 0.01, "ADD_MIN"))


@pytest.mark.parametrize("panel_loci", [32, 96, 256])
def test_several_gemm_panels(gpu_ctx, panel_loci, monkeypatch):
    """inputs larger than one operand panel (3 GB) are processed panel by panel: the first panel stores
    into the fresh count planes and carries the tail k-blocks, the later ones add in place. Forced here
    with tiny panels; also accumulates twice into the same counts object (load-add-store epilogue)."""
    monkeypatch.setenv("SECEDO_B200_PANEL_LOCI", str(panel_loci))
    cfg = SynthConfig(n_cells=300, coverage=0.3, n_loci=1200, n_chr=3, p_multi=0.1, p_mate=0.05, seed=61)
    p = make_pileup(cfg)
    ident = np.arange(cfg.n_cells, dtype=np.uint32)
    f, _ = api.Filter(0.01, 4, gpu_ctx).filter(p, ident, "", 1)
    assert f.n_loci > 3 * panel_loci
    check_counts(gpu_ctx, f, cfg.n_cells, 1000, ident, 0.01, 0.5, 0.01, 4, "gemm")
    c = api.Counts(gpu_ctx, cfg.n_cells)
    c.accumulate(f, 1000, ident, 0.01, 0.5, 0.01, 4, "gemm")
    c.accumulate(f, 1000, ident, 0.01, 0.5, 0.01, 4, "gemm")
    o = po.similarity(f, cfg.n_cells, 1000, ident, 0.01, 0.5, 0.01, 4, "ADD_MIN")
    S1, D1, H, _ = c.download()
    assert np.array_equal(S1, 2 * o.S1) and np.array_equal(D1, 2 * o.D1) and np.array_equal(H, 2 * o.H)
    c.free()


@pytest.mark.parametrize("reps", [127, 128, 200, 256, 300, 520])
def test_int8_count_range(gpu_ctx, reps):
    """the GEMM path holds per-(cell, locus) base counts in int8: up to 127 reads of one cell at a locus
    are exact, more must be refused (also when a byte of the packed counts wraps) — the scatter path
    takes them"""
    rid = iter(range(1, 10 ** 6))
    loci = []
    for i in range(40):
        gb = [(0 << 2) | 1] * reps + [(1 << 2) | 2, (2 << 2) | 1, (3 << 2) | (i & 3)]
        loci.append((100 + 30 * i, [next(rid) for _ in gb], gb))
    p = Pileup.from_pos_data([loci])
    ident = np.arange(4, dtype=np.uint32)
    ref = api.compute_similarity_matrix(p, 4, 1000, ident, 0.01, 0.5, 0.01, 1, ctx=gpu_ctx, path="scatter")
    if reps <= 127:
        M = api.compute_similarity_matrix(p, 4, 1000, ident, 0.01, 0.5, 0.01, 1, ctx=gpu_ctx, path="gemm")
        assert_matrix_close(M, ref, TOL)
        assert_matrix_close(M, po.similarity(p, 4, 1000, ident, 0.01, 0.5, 0.01, 1).M, TOL)
    else:
        with pytest.raises(api.SgpuError):
            api.compute_similarity_matrix(p, 4, 1000, ident, 0.01, 0.5, 0.01, 1, ctx=gpu_ctx, path="gemm")


def test_auto_path_falls_back_when_int8_overflows(gpu_ctx):
    """ADVICE r1: with SGPU_PATH_AUTO a pileup dense enough for the GEMM path but with > 127 reads of one cell at one
    locus must not fail half way: the first panel's range check is read before the tensor kernel touches the planes and
    the call takes the scatter path. The explicit GEMM path still refuses, and the counts object stays usable."""
    cfg = SynthConfig(n_cells=300, coverage=2.0, n_loci=400, n_chr=1, frac_somatic=1.0, frac_germline=0.0, seed=33)
    p = make_pileup(cfg)
    l = 7
    a = int(p.row_ptr[l])
    extra = 200
    rid = np.concatenate([p.read_id[:a], (4_100_000_000 + np.arange(extra)).astype(np.uint32), p.read_id[a:]])
    gb = np.concatenate([p.gid_base[:a], np.full(extra, (0 << 2) | 1, np.uint16), p.gid_base[a:]])
    row = p.row_ptr.copy()
    row[l + 1:] += np.uint64(extra)
    q = Pileup(p.chr_ptr, row, p.position, rid, gb)
    ident = np.arange(cfg.n_cells, dtype=np.uint32)
    o = po.similarity(q, cfg.n_cells, 1000, ident, 0.01, 0.5, 0.01, 2, "ADD_MIN")
    c = api.Counts(gpu_ctx, cfg.n_cells)
    st = c.accumulate(q, 1000, ident, 0.01, 0.5, 0.01, 2, "auto")
    assert st["path_used"] == "scatter"
    S1, D1, H, _ = c.download()
    assert np.array_equal(S1, o.S1) and np.array_equal(D1, o.D1) and np.array_equal(H, o.H)
    # without the overflow the same shape takes the GEMM path
    c.zero()
    assert c.accumulate(p, 1000, ident, 0.01, 0.5, 0.01, 2, "auto")["path_used"] == "gemm"
    # explicit GEMM: refused BEFORE the tensor kernel touches the planes (the range check of the staging is read first),
    # so the object stays usable and holds exactly what it held before the failed call
    c.zero()
    with pytest.raises(api.SgpuError):
        c.accumulate(q, 1000, ident, 0.01, 0.5, 0.01, 2, "gemm")
    c.accumulate(p, 1000, ident, 0.01, 0.5, 0.01, 2, "gemm")
    op = po.similarity(p, cfg.n_cells, 1000, ident, 0.01, 0.5, 0.01, 2, "ADD_MIN")
    S1, D1, H, _ = c.download()
    assert np.array_equal(S1, op.S1) and np.array_equal(D1, op.D1) and np.array_equal(H, op.H)
    c.free()


def test_int8_overflow_in_a_later_panel_poisons(gpu_ctx, monkeypatch):
    """several panels (forced small): an int8 overflow found while staging the SECOND panel comes after the first panel
    has been added - the object then says that it holds a partial sum until it is zeroed"""
    monkeypatch.setenv("SECEDO_B200_PANEL_LOCI", "64")
    cfg = SynthConfig(n_cells=300, coverage=2.0, n_loci=400, n_chr=1, frac_somatic=1.0, frac_germline=0.0, seed=34)
    p = make_pileup(cfg)
    l = 200  # in the fourth panel
    a = int(p.row_ptr[l])
    extra = 200
    rid = np.concatenate([p.read_id[:a], (4_100_000_000 + np.arange(extra)).astype(np.uint32), p.read_id[a:]])
    gb = np.concatenate([p.gid_base[:a], np.full(extra, (0 << 2) | 1, np.uint16), p.gid_base[a:]])
    row = p.row_ptr.copy()
    row[l + 1:] += np.uint64(extra)
    q = Pileup(p.chr_ptr, row, p.position, rid, gb)
    ident = np.arange(cfg.n_cells, dtype=np.uint32)
    c = api.Counts(gpu_ctx, cfg.n_cells)
    with pytest.raises(api.SgpuError):
        c.accumulate(q, 1000, ident, 0.01, 0.5, 0.01, 2, "gemm")
    with pytest.raises(api.SgpuError):
        c.accumulate(p, 1000, ident, 0.01, 0.5, 0.01, 2, "gemm")
    c.zero()
    c.accumulate(p, 1000, ident, 0.01, 0.5, 0.01, 2, "gemm")
    op = po.similarity(p, cfg.n_cells, 1000, ident, 0.01, 0.5, 0.01, 2, "ADD_MIN")
    S1, D1, H, _ = c.download()
    assert np.array_equal(S1, op.S1) and np.array_equal(D1, op.D1) and np.array_equal(H, op.H)
    c.free()


def test_huge_loci(gpu_ctx):
    """loci of > 11 000 entries: the shared-memory link table runs at its largest geometry"""
    cfg = SynthConfig(n_cells=3000, coverage=4.0, n_loci=8, n_chr=1, frac_somatic=1.0, frac_germline=0.0,
                      p_multi=0.05, p_mate=0.02, seed=51)
    p = make_pileup(cfg)
    assert np.diff(p.row_ptr.astype(np.int64)).max() > 11000
    ident = np.arange(cfg.n_cells, dtype=np.uint32)
    check_counts(gpu_ctx, p, cfg.n_cells, 1000, ident, 0.01, 0.5, 0.01, 1, "gemm")


@pytest.mark.parametrize("path", PATHS)
def test_global_hash_linking(gpu_ctx, path, monkeypatch):
    """loci too large for the shared-memory link table (> ~26 000 entries) are linked through a global
    (chromosome, read id) hash; forced here on a small case so that the oracle can follow"""
    monkeypatch.setenv("SECEDO_B200_FORCE_GLOBAL_HASH", "1")
    cfg = SynthConfig(n_cells=60, coverage=0.3, n_loci=900, n_chr=3, p_multi=0.45, p_mate=0.15, theta=0.02, seed=8)
    p = make_pileup(cfg)
    ident = np.arange(cfg.n_cells, dtype=np.uint32)
    f, _ = api.Filter(0.01, 4, gpu_ctx).filter(p, ident, "", 1)
    st, o = check_counts(gpu_ctx, f, cfg.n_cells, 1000, ident, 0.01, 0.5, 0.01, 2, path)
    assert st["n_multi_reads"] > 0 and st["n_dropped_entries"] > 0


def test_finalize_async_matches_finalize(gpu_ctx):
    """the matrix downloaded on its own stream (sgpu_similarity_finalize_async + sgpu_output_wait) while the next batch is
    already being accumulated equals the synchronous result; a second download first waits for the first"""
    import torch
    cfg = SynthConfig(n_cells=500, coverage=0.3, n_loci=1500, n_chr=2, p_multi=0.1, p_mate=0.05, theta=0.01, seed=19)
    ident = np.arange(cfg.n_cells, dtype=np.uint32)
    f, _ = api.Filter(0.01, 4, gpu_ctx).filter(make_pileup(cfg), ident, "", 1)
    c = api.Counts(gpu_ctx, cfg.n_cells)
    c.accumulate(f, 1000, ident, 0.01, 0.5, 0.01, 8, "gemm")
    want = c.finalize(1000, 0.01, 0.5, 0.01, "ADD_MIN")
    bufs = [torch.zeros((cfg.n_cells, cfg.n_cells), dtype=torch.float64).pin_memory().numpy() for _ in range(2)]
    c.finalize_async(1000, 0.01, 0.5, 0.01, "ADD_MIN", bufs[0])
    c.accumulate(f, 1000, ident, 0.01, 0.5, 0.01, 8, "gemm")  # twice the counts, while the first matrix travels
    c.finalize_async(1000, 0.01, 0.5, 0.01, "EXPONENTIATE", bufs[1])
    gpu_ctx.output_wait()
    assert np.array_equal(bufs[0], want)
    assert np.array_equal(bufs[1], c.finalize(1000, 0.01, 0.5, 0.01, "EXPONENTIATE"))
    gpu_ctx.output_wait()  # nothing in flight: returns at once
    c.free()


def test_sparse_plane_lists(gpu_ctx):
    """sgpu_counts_sparse_pack / sgpu_counts_sparse_add and the plane-range pack: the non-zeros of the second-order
    planes of one counts object added into another equal the sum of the planes (what the cross-rank reduction does
    with them), and S, D survive a pack / unpack round trip of their range alone"""
    cfg = SynthConfig(n_cells=300, coverage=0.4, n_loci=1200, n_chr=2, p_multi=0.3, p_mate=0.05, theta=0.01, seed=23)
    p = make_pileup(cfg)
    ident = np.arange(cfg.n_cells, dtype=np.uint32)
    f, _ = api.Filter(0.01, 4, gpu_ctx).filter(p, ident, "", 1)
    halves = [f.loci_range(0, 0, 1 << 40), f.loci_range(1, 0, 1 << 40)]
    a, b, whole = (api.Counts(gpu_ctx, cfg.n_cells) for _ in range(3))
    a.accumulate(halves[0], 1000, ident, 0.01, 0.5, 0.01, 8, "gemm")
    b.accumulate(halves[1], 1000, ident, 0.01, 0.5, 0.01, 8, "gemm")
    whole.accumulate(f, 1000, ident, 0.01, 0.5, 0.01, 8, "gemm")
    planes = max(a.buffers()[1], b.buffers()[1]) // (cfg.n_cells ** 2)
    assert planes >= 5
    a.set_layout(planes, False)
    b.set_layout(planes, False)
    ha, hb, hw = a.download()[2], b.download()[2], whole.download()[2]
    assert np.array_equal(ha + hb, hw) and hw.sum() > 0
    idx, val, nnz = a.sparse_pack(2)
    assert nnz >= np.count_nonzero(np.triu(ha, 1).reshape(3, -1).any(0)) and nnz > 0
    b.sparse_add(2, idx, val, nnz)
    assert np.array_equal(b.download()[2], hw)
    s_before = a.download()[:2]
    a.pack_range(0, 2)
    a.unpack_range(0, 2)
    for x, y in zip(a.download()[:2], s_before):
        assert np.array_equal(x, y)
    with pytest.raises(api.SgpuError):
        a.pack_range(1, planes)  # beyond the planes in use
    for c in (a, b, whole):
        c.free()
