"""bench.py's --steps and --dump-outputs: the timed loops run the number of steps asked for, and the dump holds the
similarity matrix of the timed workload, checked against the oracle on the same seeded pileup. The reference arm runs on
the host; the device-resident path needs a GPU."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, assert_matrix_close
from oracle import pyoracle as po

ROWS, INDEX = "similarity_matrix_rows.npy", "similarity_matrix_row_index.npy"


def oracle_matrix(p, n, threads):
    import bench
    w = bench.WORKLOAD
    ident = np.arange(n, dtype=np.uint32)
    kl, ke, _, _ = po.filter_flags(p, ident, w["theta"])
    return po.similarity(p.select(kl, ke), n, w["L"], ident, w["eps"], w["h"], w["theta"], threads, w["normalization"]).M


def test_reference_arm_steps_and_dump(tmp_path, monkeypatch, capsys):
    import bench
    n, threads = 300, 2
    monkeypatch.setitem(bench.WORKLOAD, "n_cells", n)
    monkeypatch.setenv("SECEDO_BENCH_THREADS", str(threads))
    monkeypatch.delenv("RANK", raising=False)
    calls = []
    step = bench.run_reference_step
    monkeypatch.setattr(bench, "run_reference_step", lambda *a, **k: calls.append(k.get("want_matrix")) or step(*a, **k))
    args = argparse.Namespace(gpus=1, steps=3, warmup=2, dump_outputs=str(tmp_path))
    assert bench.main_reference(args) == 0
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["steps"] == 3 and calls == [False] * 4 + [True]  # 2 warm-up + 3 timed steps, the matrix of the last one
    assert sorted(os.listdir(tmp_path)) == [INDEX, ROWS]
    M, idx = np.load(tmp_path / ROWS), np.load(tmp_path / INDEX)
    assert M.dtype == idx.dtype == np.float64 and np.array_equal(idx, np.arange(n))
    assert_matrix_close(M, oracle_matrix(bench.cpu_sample(), n, threads), 1e-9)


def test_large_matrix_is_sampled_by_rows(tmp_path):
    import bench
    n = 2100  # 35 MB of float64: more than the dump budget
    M = np.arange(n * n, dtype=np.float64).reshape(n, n)
    bench.dump_matrix(str(tmp_path), M)
    rows, idx = np.load(tmp_path / ROWS), np.load(tmp_path / INDEX)
    assert rows.nbytes <= bench.DUMP_MATRIX_BYTES and 0 < idx.size < n and np.all(np.diff(idx) > 0)
    assert np.array_equal(rows, M[idx.astype(np.int64)])
    bench.dump_matrix(str(tmp_path / "again"), M)
    assert np.array_equal(np.load(tmp_path / "again" / INDEX), idx)


@pytest.mark.gpu
def test_device_bench_steps_and_dump(gpu_ctx, tmp_path, monkeypatch):
    """the headline (device-resident) path on a small workload of one sub-batch: K timed steps issue K times the kernels of
    one, and the dump is the matrix of the generated pileup"""
    import bench
    n, loci, threads = 300, 512, 4
    env = dict(os.environ, SECEDO_BENCH_CELLS=str(n), SECEDO_BENCH_LOCI_PER_CHR=str(loci), SECEDO_BENCH_SUB_BATCHES="1",
               SECEDO_BENCH_THREADS=str(threads))
    lines = {}
    for steps in (1, 3):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                            "--skip-extras", "--dump-outputs", str(tmp_path / str(steps))],
                           capture_output=True, text=True, env=env, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        lines[steps] = json.loads(r.stdout.strip().splitlines()[-1])
    assert lines[3]["steps"] == 3 and lines[3]["e2e"]["steps"] == 3
    assert lines[1]["gpu_launches"] > 0 and lines[3]["gpu_launches"] == 3 * lines[1]["gpu_launches"]
    M, idx = np.load(tmp_path / "1" / ROWS), np.load(tmp_path / "1" / INDEX)
    assert np.array_equal(M, np.load(tmp_path / "3" / ROWS)) and np.array_equal(idx, np.arange(n))
    monkeypatch.setitem(bench.WORKLOAD, "n_cells", n)
    monkeypatch.setitem(bench.WORKLOAD, "loci_per_chr", loci)
    dev = bench.synth_sub_batch(gpu_ctx, 0, 0)
    p = dev.download()
    dev.free()
    assert M.max() > 0.0
    assert_matrix_close(M, oracle_matrix(p, n, threads), 1e-6)
