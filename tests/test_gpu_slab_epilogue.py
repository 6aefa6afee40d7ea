"""The peer-memory epilogue (sgpu_slab_raw / sgpu_slab_finalize) and the plane checksum, on ONE GPU.

A peer is only a device pointer that is valid on this GPU, so the count planes of G counts objects on one device stand
for G GPUs: object g accumulates piece g of the pileup, and every share of the 32 x 32 tiles is computed by a host object
of its own (the slab state belongs to the counts object). The matrix must equal the single-GPU epilogue
(sgpu_similarity_finalize) of an object that accumulated the whole pileup: bit for bit while no read pair overlaps at
>= 4 loci (integer sums, the same fp64 expression) and while only one spill plane is non-zero; to rounding when the
spill is spread over several planes. The checksum is compared with a numpy restatement of checksum_kernel, and the
exchange primitives of dist.reduce_counts (dense packs, sparse lists) are run with torch doing the reduction."""
from dataclasses import replace

import numpy as np
import pytest
import torch

from conftest import assert_matrix_close
from oracle import pyoracle as po
from secedo_b200 import api, dist
from secedo_b200.pileup import Pileup
from secedo_b200.synth import SynthConfig, make_pileup
from test_gpu_pieces import chrom_positions, cutoffs_from_ends, piece_pileup

pytestmark = pytest.mark.gpu
L, EPS, HOM, THETA = 1000, 0.01, 0.5, 0.01
PARAMS = (L, EPS, HOM, THETA)
NORMS = ("ADD_MIN", "EXPONENTIATE", "SCALE_MAX_1")
MAX_PEERS = 16  # SGPU_MAX_PEERS
# read pairs overlapping at 2 and 3 loci, none at >= 4: planes 0..8 in use, no spill plane
ORDER3 = SynthConfig(n_cells=200, coverage=0.3, n_loci=600, n_chr=3, p_multi=0.08, p_mate=0.05, theta=0.02, seed=21)
# test_gpu_similarity.test_high_order_overlaps: fragments over up to 6 close loci, classes of order >= 4 in the spill plane
SPILL = SynthConfig(n_cells=25, coverage=1.5, n_loci=300, n_chr=1, spacing=40, p_multi=0.9, p_mate=0.1, seed=31)
# every read covers one locus: S and D only
PLAIN = SynthConfig(n_cells=SPILL.n_cells, coverage=0.5, n_loci=400, n_chr=1, seed=5)


@pytest.fixture
def pool(gpu_ctx):
    """pool(n) makes a counts object of n cells; all of them are freed when the test ends, whatever its outcome"""
    made = []

    def make(n):
        c = api.Counts(gpu_ctx, n)
        made.append(c)
        return c

    yield make
    for c in made:
        c.free()
    torch.cuda.empty_cache()


def device(ctx):
    return torch.device("cuda", ctx.device)


def ident(n):
    return np.arange(n, dtype=np.uint32)


def planes_in_use(c):
    return c.buffers()[1] // c.num_cells ** 2


def has_spill(c):
    return c.buffers()[3] > 0


def accumulate_pieces(objs, p, n, path, threads, params=PARAMS):
    """object g accumulates piece g of the pileup (owned loci + halos, tails decided from the chromosome ends)"""
    Lf, eps, h, theta = params
    tail, _ = cutoffs_from_ends(objs[0].ctx, p, threads)
    for c, piece in zip(objs, dist.plan_pieces(chrom_positions(p), len(objs), Lf)):
        if piece:
            c.accumulate_range(piece_pileup(p, piece), Lf, ident(n), eps, h, theta, [d["own_pos_begin"] for d in piece],
                               [d["own_pos_end"] for d in piece], [tail[d["chrom"]] for d in piece], path)


def emulate(pool, p, n, G, split, path, threads=2):
    """(G objects standing for G GPUs, the reference object that accumulated the whole pileup). split "pieces": object g
    holds piece g; "lopsided": object 0 holds everything, the others nothing (their layouts differ from object 0's)."""
    ref = pool(n)
    ref.accumulate(p, L, ident(n), EPS, HOM, THETA, threads, path)
    objs = [pool(n) for _ in range(G)]
    if split == "lopsided":
        objs[0].accumulate(p, L, ident(n), EPS, HOM, THETA, threads, path)
    else:
        accumulate_pieces(objs, p, n, path, threads)
    return objs, ref


def hosts_for(pool, peers, n_slabs):
    """one host object per share: the peers themselves, then empty objects"""
    return peers[:n_slabs] + [pool(peers[0].num_cells) for _ in range(n_slabs - len(peers))]


def agree_layout(objs, spill_everywhere=True):
    """what SlabEpilogue.agree does over the ranks: the most planes any object uses, and a spill plane on every object
    once one of them has one (or, with spill_everywhere=False, only where there already is one)"""
    planes = max(planes_in_use(c) for c in objs)
    spill = any(has_spill(c) for c in objs)
    for c in objs:
        c.set_layout(planes, spill and (spill_everywhere or has_spill(c)))
    return planes, spill


def run_slabs(hosts, peers, n_slabs, norm, out_ptr=None, spill_everywhere=True, params=PARAMS):
    """SlabEpilogue.run over all ranks: share s is computed by hosts[s]; returns the pointers the shares went to"""
    ctx = hosts[0].ctx
    _, spill = agree_layout(peers + hosts, spill_everywhere)  # also joins every object's held-back tensor kernel
    peer_planes = [c.buffers()[0] for c in peers]
    peer_spill = [c.buffers()[2] for c in peers] if spill else None  # None where an object holds no spill plane
    ext = [hosts[s].slab_raw(peer_planes, s, n_slabs, *params, peer_spill=peer_spill) for s in range(n_slabs)]
    ctx.synchronize()
    pairs = [dist.tensor_from_ptr(e, 2, torch.float64, device(ctx)) for e in ext]
    both = torch.stack(pairs).amax(dim=0)  # the all-reduce MAX of {-min, max}
    for t in pairs:
        t.copy_(both)
    torch.cuda.synchronize()
    return [hosts[s].slab_finalize(norm, out_ptr) for s in range(n_slabs)]


def slab_matrix(hosts, peers, n_slabs, norm, **kw):
    """all shares written into one device matrix that starts as NaN: nothing may be left out"""
    ctx = hosts[0].ctx
    n = peers[0].num_cells
    out = torch.full((n, n), float("nan"), dtype=torch.float64, device=device(ctx))
    torch.cuda.synchronize()
    assert run_slabs(hosts, peers, n_slabs, norm, out.data_ptr(), **kw) == [out.data_ptr()] * n_slabs
    ctx.synchronize()
    return out.cpu().numpy()


def single_gpu(c, norms=NORMS, params=PARAMS):
    return {norm: c.finalize(*params, norm) for norm in norms}


def assert_rounding_close(got, want, span):
    """equal up to fp64 sums of the spill planes taken in another order: within 1e-12 * max|M|. EXPONENTIATE maps a raw
    value v to 1 / (exp(v) + 1), which turns an error dv into a relative error dv of the entry, so there the bound is
    element-wise, 1e-12 * span * |M|, where span >= max|v| is the largest entry of the ADD_MIN matrix (max - min of the
    raw values, the zero diagonal included)."""
    for norm in NORMS:
        if norm == "EXPONENTIATE":
            assert (np.abs(got[norm] - want[norm]) <= 1e-12 * span * np.abs(want[norm])).all(), norm
        else:
            assert_matrix_close(got[norm], want[norm], 1e-12)


def oracle_matrices(p, n, threads=2):
    return {norm: po.similarity(p, n, L, ident(n), EPS, HOM, THETA, threads, norm).M for norm in NORMS}


# ------------------------------------------------------------------------------------------------ the matrix
@pytest.mark.parametrize("split", ["pieces", "lopsided"])
@pytest.mark.parametrize("G", [2, 3, 5, MAX_PEERS])
@pytest.mark.parametrize("path", ["scatter", "gemm"])
def test_slabs_equal_one_gpu_bit_for_bit(gpu_ctx, pool, path, G, split):
    """G peers, 1, G and G + 1 shares (G + 1 is coprime to G and needs a host that is not a peer)"""
    p, n = make_pileup(ORDER3), ORDER3.n_cells
    objs, ref = emulate(pool, p, n, G, split, path)
    assert planes_in_use(ref) == 9 and not has_spill(ref), "overlaps of order 3 and none of order >= 4"
    want, oracle = single_gpu(ref), oracle_matrices(p, n)
    for n_slabs in (1, G, G + 1):
        hosts = hosts_for(pool, objs, n_slabs)
        for norm in NORMS:
            got = slab_matrix(hosts, objs, n_slabs, norm)
            assert np.array_equal(got, want[norm], equal_nan=True), f"{n_slabs} shares, {norm}"
            assert_matrix_close(got, oracle[norm], 1e-6)


@pytest.mark.parametrize("n", [SPILL.n_cells, 70])
@pytest.mark.parametrize("path", ["scatter", "gemm"])
def test_slabs_with_spill_planes(gpu_ctx, pool, path, n):
    """One non-zero spill plane, the others null or zero: bit for bit the single-GPU epilogue of the object holding that
    plane (it adds the same plane once). Spill spread over several planes (pieces): to rounding."""
    cfg = SPILL if n == SPILL.n_cells else replace(SPILL, n_cells=n, coverage=0.6)
    p = make_pileup(cfg)
    G = 3
    objs, ref = emulate(pool, p, n, G, "lopsided", path, threads=1)
    assert has_spill(objs[0]) and not any(has_spill(c) for c in objs[1:])
    want, want_ref, oracle = single_gpu(objs[0]), single_gpu(ref), oracle_matrices(p, n, threads=1)
    for spill_everywhere, peers in ((False, objs), (False, objs[::-1]), (True, objs)):
        for n_slabs in (1, G, G + 1):
            hosts = hosts_for(pool, peers, n_slabs)
            for norm in NORMS:
                got = slab_matrix(hosts, peers, n_slabs, norm, spill_everywhere=spill_everywhere)
                assert np.array_equal(got, want[norm], equal_nan=True), f"spill on every peer: {spill_everywhere}, {n_slabs} shares, {norm}"
            assert [has_spill(c) for c in peers] == [c is objs[0] or spill_everywhere for c in peers]
    span = want_ref["ADD_MIN"].max()
    assert_rounding_close(want, want_ref, span)
    for norm in NORMS:
        assert_matrix_close(want[norm], oracle[norm], 1e-6)
    # the spill spread over the pieces
    pieces = [pool(n) for _ in range(G)]
    accumulate_pieces(pieces, p, n, path, threads=1)
    agree_layout(pieces)
    gpu_ctx.synchronize()
    spills = [dist.counts_tensors(c, device(gpu_ctx))[1] for c in pieces]
    assert sum(bool(s.any()) for s in spills) >= 2, "the spill must be spread over several planes"
    for n_slabs in (1, G, G + 1):
        hosts = hosts_for(pool, pieces, n_slabs)
        assert_rounding_close({norm: slab_matrix(hosts, pieces, n_slabs, norm) for norm in NORMS}, want_ref, span)


@pytest.mark.parametrize("n", [2, 3, 31, 32, 33, 65, 257, 1000])
def test_shapes_and_coverage_of_the_output(gpu_ctx, pool, n):
    """partial tiles, one tile, more shares than tiles (those shares have none): every element written once, and
    equal to one GPU"""
    cfg = SynthConfig(n_cells=n, coverage=min(1.0, 40.0 / n), n_loci=300, n_chr=2, p_multi=0.08, p_mate=0.05, theta=0.02,
                      seed=40 + n)
    p = make_pileup(cfg)
    objs, ref = emulate(pool, p, n, 3, "pieces", "auto")
    assert not has_spill(ref)
    want = single_gpu(ref)
    for n_slabs in (1, 3, 5):
        hosts = hosts_for(pool, objs, n_slabs)
        for norm in NORMS:
            got = slab_matrix(hosts, objs, n_slabs, norm)
            assert np.array_equal(got, want[norm], equal_nan=True), f"{n_slabs} shares, {norm}"
        if n_slabs > dist.tri_tile_count(n):
            assert any(h.slab_range()[0] == h.slab_range()[1] for h in hosts), "a share without tiles"


def test_empty_pileup(gpu_ctx, pool):
    """nothing accumulated anywhere: ADD_MIN gives zeros, SCALE_MAX_1 divides by max = 0 (NaN off the diagonal), on one
    GPU and in shares"""
    n = 40
    objs, ref = emulate(pool, Pileup.empty(2), n, 3, "pieces", "auto")
    want = single_gpu(ref)
    off = ~np.eye(n, dtype=bool)
    assert not want["ADD_MIN"].any()
    assert np.isnan(want["SCALE_MAX_1"][off]).all() and not want["SCALE_MAX_1"][~off].any()
    for n_slabs in (1, 3, 5):
        hosts = hosts_for(pool, objs, n_slabs)
        for norm in NORMS:
            assert np.array_equal(slab_matrix(hosts, objs, n_slabs, norm), want[norm], equal_nan=True), (n_slabs, norm)


@pytest.mark.parametrize("n,G,n_slabs", [(257, 3, 4), (2, 2, 3)])
def test_output_targets(gpu_ctx, pool, monkeypatch, n, G, n_slabs):
    """out = NULL: every host's own matrix holds exactly its tiles and their mirror images; mapped host memory
    (sgpu_host_register): every share written over the mapping"""
    cfg = SynthConfig(n_cells=n, coverage=min(1.0, 40.0 / n), n_loci=300, n_chr=2, p_multi=0.08, p_mate=0.05, theta=0.02,
                      seed=60 + n)
    objs, ref = emulate(pool, make_pileup(cfg), n, G, "pieces", "scatter")
    want = single_gpu(ref)
    hosts = hosts_for(pool, objs, n_slabs)
    nb = (n + 31) // 32
    ptrs = run_slabs(hosts, objs, n_slabs, "ADD_MIN")
    gpu_ctx.synchronize()
    assert len(set(ptrs)) == n_slabs, "every host writes into a matrix of its own"
    covered = np.zeros((n, n), bool)
    for s, (h, ptr) in enumerate(zip(hosts, ptrs)):
        assert h.slab_range() == dist.slab_tiles(n, s, n_slabs)
        mine = dist.tensor_from_ptr(ptr, n * n, torch.float64, device(gpu_ctx)).cpu().numpy().reshape(n, n)
        for t in range(*h.slab_range()):
            bi, bj = dist.tri_tile(t, nb)
            rows, cols = slice(bi * 32, bi * 32 + 32), slice(bj * 32, bj * 32 + 32)
            assert np.array_equal(mine[rows, cols], want["ADD_MIN"][rows, cols]), (s, t)
            assert np.array_equal(mine[cols, rows], want["ADD_MIN"][cols, rows]), (s, t)
            covered[rows, cols] = covered[cols, rows] = True
    assert covered.all()
    # SharedHostMatrix as world 1. Its segment is unlinked by close(); the resource tracker of multiprocessing would
    # start a helper process to do the same at exit.
    from multiprocessing import resource_tracker
    monkeypatch.setattr(resource_tracker, "register", lambda *a, **k: None)
    monkeypatch.setattr(resource_tracker, "unregister", lambda *a, **k: None)
    shared = dist.SharedHostMatrix(gpu_ctx, n)
    try:
        for norm in NORMS:
            shared.array[:] = np.nan
            assert run_slabs(hosts, objs, n_slabs, norm, shared.dev_ptr) == [shared.dev_ptr] * n_slabs
            gpu_ctx.synchronize()
            assert np.array_equal(shared.array, want[norm], equal_nan=True), norm
    finally:
        shared.close()


def peer_checksum(hosts, peers, n_slabs):
    """the checksums of the peer-summed shares, added up mod 2^64"""
    planes = [c.buffers()[0] for c in peers]
    return sum(hosts[s % len(hosts)].checksum(planes, s, n_slabs) for s in range(n_slabs)) % 2 ** 64


def test_full_size_8000_cells_8_shares(gpu_ctx, pool):
    """8 000 cells at 0.5x on the device generator, 8 pieces, 8 shares (nb = 250): bit-identical to one GPU"""
    n, params = 8000, (L, 0.01, 0.15, 0.001)
    dev = gpu_ctx.synth_pileup(n, 0.5, 2, 256, n_clones=2, theta=0.001, p_multi=0.02, p_mate=0.01, seed=31)
    fdev, _ = api.Filter(0.001, 4, gpu_ctx).filter_device(dev, ident(n))
    dev.free()
    ref = pool(n)
    ref.accumulate(fdev, L, ident(n), *params[1:], 8, "gemm")
    f = fdev.download()
    fdev.free()
    objs = [pool(n) for _ in range(8)]
    accumulate_pieces(objs, f, n, "gemm", 8, params)
    assert planes_in_use(ref) > 2 and not has_spill(ref), "overlaps at several loci, none at >= 4"
    want = single_gpu(ref, params=params)
    for norm in NORMS:
        assert np.array_equal(slab_matrix(objs, objs, 8, norm, params=params), want[norm], equal_nan=True), norm
    assert peer_checksum(objs, objs, 8) == ref.checksum() != 0


def test_full_size_20000_wide_cells_3_shares(gpu_ctx, pool):
    """20 000 cells (wide entries), 2 pieces, 3 shares (nb = 625: the device tile decode far from tile 0); the third share
    is computed by the reference object, which is not a peer. 3 x 14.4 GB of planes, two 3.2 GB matrices."""
    n, params = 20000, (L, 0.01, 0.5, 0.001)
    dev = gpu_ctx.synth_pileup(n, 0.25, 2, 64, n_clones=4, theta=0.001, p_multi=0.02, p_mate=0.01, seed=19)
    fdev, _ = api.Filter(0.001, 4, gpu_ctx).filter_device(dev, ident(n))
    dev.free()
    ref = pool(n)
    ref.accumulate(fdev, L, ident(n), *params[1:], 8, "gemm")
    f = fdev.download()
    fdev.free()
    objs = [pool(n) for _ in range(2)]
    accumulate_pieces(objs, f, n, "gemm", 8, params)
    assert not has_spill(ref), "no overlaps of order >= 4"
    want = ref.finalize(*params, "ADD_MIN")
    got = slab_matrix(objs + [ref], objs, 3, "ADD_MIN", params=params)
    assert [h.slab_range() for h in objs + [ref]] == [dist.slab_tiles(n, s, 3) for s in range(3)]
    assert np.array_equal(got, want)
    del got, want
    assert peer_checksum(objs + [ref], objs, 3) == ref.checksum() != 0


# ------------------------------------------------------------------------------------------------ the checksum
def mix_weight(x):
    """splitmix64 (increment and finaliser) of uint64 positions, as mix_weight in abi.cu"""
    x = x + np.uint64(0x9E3779B97F4A7C15)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def host_checksum(planes, n, planes_used):
    """checksum_kernel restated: over the planes in use and i < j, uint64(int64(value)) * weight(pl n^2 + i n + j), summed
    with wrap-around"""
    planes = np.asarray(planes).reshape(-1, n, n)
    i, j = np.triu_indices(n, 1)
    pos = i.astype(np.uint64) * np.uint64(n) + j.astype(np.uint64)
    acc = 0
    for pl in range(planes_used):
        v = planes[pl][i, j].astype(np.int64).astype(np.uint64)
        acc += int(np.sum(v * mix_weight(pos + np.uint64(pl * n * n)), dtype=np.uint64))
    return acc % 2 ** 64


def read_planes(c):
    """the planes in use, lower triangles zeroed (only i < j is meaningful)"""
    c.ctx.synchronize()
    n = c.num_cells
    planes = dist.counts_tensors(c, device(c.ctx))[0].cpu().numpy().astype(np.int64).reshape(-1, n, n)
    return planes * np.triu(np.ones((n, n), np.int64), 1)


@pytest.mark.parametrize("split", ["pieces", "lopsided"])
def test_checksum_against_host_reference(gpu_ctx, pool, split):
    p, n = make_pileup(ORDER3), ORDER3.n_cells
    G = 3
    objs, ref = emulate(pool, p, n, G, split, "gemm")
    own = []
    for c in objs + [ref]:
        own.append(c.checksum())
        assert own[-1] == host_checksum(read_planes(c), n, planes_in_use(c))
        # the shares of one object's own planes add up to its checksum
        assert sum(c.checksum(None, s, 4) for s in range(4)) % 2 ** 64 == own[-1]
    planes, _ = agree_layout(objs)
    assert [c.checksum() for c in objs] == own[:G], "planes that were never used are zero"
    summed = sum(read_planes(c) for c in objs)
    assert np.array_equal(summed, read_planes(ref))
    n_tiles = dist.tri_tile_count(n)
    for n_slabs in (1, G, G + 1, n_tiles + 5):  # the last: more shares than tiles
        total = peer_checksum(objs, objs, n_slabs)
        assert total == sum(own[:G]) % 2 ** 64 == host_checksum(summed, n, planes) == own[G]
    # one count more in one peer: above the diagonal it changes the sum by the weight of its position, below it is not read
    t = dist.counts_tensors(objs[1], device(gpu_ctx))[0]
    i, j, pl = 5, n - 7, 6
    for (a, b), delta in (((i, j), int(mix_weight(np.array([pl * n * n + i * n + j], np.uint64))[0])), ((j, i), 0)):
        t[pl * n * n + a * n + b] += 1
        torch.cuda.synchronize()
        for n_slabs in (1, n_tiles + 5):
            assert (peer_checksum(objs, objs, n_slabs) - own[G]) % 2 ** 64 == delta, ((a, b), n_slabs)
        t[pl * n * n + a * n + b] -= 1
        torch.cuda.synchronize()


def test_layout_growth(gpu_ctx, pool):
    """an object that used 2 planes, grown to 9 planes and a spill plane: same checksum, the new planes and the spill
    plane are zero, and as a peer it adds nothing beyond its S and D. Also for an object whose planes 2..8 and spill
    plane held counts before sgpu_counts_zero."""
    n = SPILL.n_cells
    plain = make_pileup(PLAIN)
    fresh, reused, full = pool(n), pool(n), pool(n)
    full.accumulate(make_pileup(SPILL), L, ident(n), EPS, HOM, THETA, 1, "scatter")
    reused.accumulate(make_pileup(SPILL), L, ident(n), EPS, HOM, THETA, 1, "scatter")
    assert planes_in_use(reused) == 9 and has_spill(reused)
    reused.zero()
    for c in (fresh, reused):
        c.accumulate(plain, L, ident(n), EPS, HOM, THETA, 1, "scatter")
        assert planes_in_use(c) == 2
    assert not has_spill(fresh)
    before = [c.checksum() for c in (fresh, reused)]
    assert before[0] == before[1] == host_checksum(read_planes(fresh), n, 2) != 0
    for c, b in zip((fresh, reused), before):
        c.set_layout(9, True)
        assert planes_in_use(c) == 9 and has_spill(c)
        assert c.checksum() == b
        gpu_ctx.synchronize()
        i32, f64, _ = dist.counts_tensors(c, device(gpu_ctx))
        assert not i32[2 * n * n:].any() and not f64.any()
    for n_slabs in (1, 2):
        assert peer_checksum([full], [fresh, reused, full], n_slabs) == (sum(before) + full.checksum()) % 2 ** 64


# ------------------------------------------------------------------------------------------------ reduce_counts on one GPU
@pytest.mark.parametrize("route", ["dense", "sparse"])
def test_exchange_primitives(gpu_ctx, pool, route):
    """reduce_counts with torch doing the collectives: the upper triangles packed on every object (planes 0..8, or S and
    D with the planes 2..8 as lists of non-zeros) and summed onto object 0, which then equals the reference"""
    p, n = make_pileup(ORDER3), ORDER3.n_cells
    objs, ref = emulate(pool, p, n, 4, "pieces", "gemm")
    dev = device(gpu_ctx)
    planes, spill = agree_layout(objs)
    assert planes == 9 and not spill
    dense = planes if route == "dense" else 2
    packed = [c.pack_range(0, dense) for c in objs]
    lists = [c.sparse_pack(2) for c in objs] if route == "sparse" else []
    gpu_ctx.synchronize()
    assert all(m == dense * n * (n - 1) // 2 for _, m in packed)
    dst = dist.tensor_from_ptr(packed[0][0], packed[0][1], torch.int32, dev)
    for ptr, m in packed[1:]:
        dst += dist.tensor_from_ptr(ptr, m, torch.int32, dev)
    hist = dist.counts_tensors(objs[0], dev)[2]
    for c in objs[1:]:
        hist += dist.counts_tensors(c, dev)[2]
    torch.cuda.synchronize()
    objs[0].unpack_range(0, dense)
    if route == "sparse":
        assert all(nnz for _, _, nnz in lists)
        for idx, val, nnz in lists[1:]:
            objs[0].sparse_add(2, idx, val, nnz)
    for a, b, name in zip(objs[0].download(), ref.download(), ("S", "D", "H", "hist")):
        assert np.array_equal(a, b), name
    assert np.array_equal(read_planes(objs[0]), read_planes(ref)), "planes 0..8"
    assert np.array_equal(objs[0].finalize(*PARAMS, "ADD_MIN"), ref.finalize(*PARAMS, "ADD_MIN"))


# ------------------------------------------------------------------------------------------------ refusals
def refused(fn, *args, **kw):
    with pytest.raises(api.SgpuError) as e:
        fn(*args, **kw)
    assert e.value.code == -2, str(e.value)


def test_refusals(gpu_ctx, pool):
    n = SPILL.n_cells
    plain, spilled = pool(n), pool(n)
    plain.accumulate(make_pileup(PLAIN), L, ident(n), EPS, HOM, THETA, 1, "scatter")
    spilled.accumulate(make_pileup(SPILL), L, ident(n), EPS, HOM, THETA, 1, "scatter")
    assert not has_spill(plain) and has_spill(spilled)
    agree_layout([plain, spilled], spill_everywhere=False)
    own = plain.buffers()[0]
    refused(plain.slab_finalize, "ADD_MIN")  # before any slab_raw
    refused(plain.slab_raw, [], 0, 1, *PARAMS)
    refused(plain.slab_raw, [own] * (MAX_PEERS + 1), 0, 1, *PARAMS)
    refused(plain.slab_raw, [own], 1, 1, *PARAMS)
    refused(plain.slab_raw, [own], 0, 0, *PARAMS)
    refused(plain.checksum, [own], 2, 2)
    refused(plain.checksum, None, 1, 1)
    peers, spills = [spilled.buffers()[0]], [spilled.buffers()[2]]
    refused(spilled.slab_raw, peers, 0, 1, *PARAMS)  # a spill plane and no peer_spill
    # the spill plane holds G(x_s, x_d) of the accumulation's parameters: no others
    for other in ((L // 2, EPS, HOM, THETA), (L, 2 * EPS, HOM, THETA), (L, EPS, 0.25, THETA), (L, EPS, HOM, 2 * THETA)):
        refused(spilled.slab_raw, peers, 0, 1, *other, peer_spill=spills)
    spilled.slab_raw(peers, 0, 1, *PARAMS, peer_spill=spills)
    spilled.slab_finalize("ADD_MIN")
    # without a spill plane the integer planes are evaluated with whatever parameters are given, as by finalize
    plain.slab_raw([own], 0, 1, L, 2 * EPS, HOM, THETA)
    plain.slab_finalize("ADD_MIN")
    plain.slab_raw([own] * MAX_PEERS, 0, 1, *PARAMS)
    gpu_ctx.synchronize()
