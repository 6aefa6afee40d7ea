#!/usr/bin/env python
"""Benchmark of the similarity-matrix hot path (BASELINE.json metric: similarity-matrix build time &
loci/s at 8K cells, 0.5x, on 1/2/4/8 B200, next to the reference's OpenMP CPU path).

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched with torchrun)
    python bench.py --impl reference --steps K --warmup W    (the reference's own CPU path)
    python bench.py --workload cfg3-genome --gpus N          (whole genome, 23 chromosomes, strong scaling, absolute seconds)

A step = one pass of the hot path over this GPU's share of the pileup and ONE similarity matrix:
    for each of SUB sub-batches of chromosomes: Filter::filter -> read linking / mate rule / cutoff
        -> first-order counts (int8 tcgen05 GEMM) -> multi-locus correction, accumulated into one set of count planes
    -> the multi-GPU epilogue over peer memory (every GPU sums the planes of all GPUs over its share of the matrix through
       NVLink and applies the log-likelihood transform in the same kernel; one scalar all-reduce) -> N x N matrix.
Weak scaling: every rank owns its own chromosomes (its own seeds). `value` times the steps with the pileup already
resident in HBM; `e2e` times the same call sequence with HOST (pinned) buffers: the H2D copy of the whole pileup and
the transfer of the matrix into host memory are inside the timed region. The CPU baseline / reference arm run the
UNMODIFIED reference compiled into oracle/_ref (or, if that .so is absent, the oracle port) on a bounded sample of the
same workload, and the GPU path is checked against that very run (`parity_vs_reference`).

--steps K sets the number of timed steps of the headline (device-resident), end-to-end, whole-genome and reference
regions. The side measurements reported next to them have fixed counts: the tensor kernel alone (2 steps), the eigen-solver
(3 runs), EM (one call) and the C++ shim driver (2 steps). --dump-outputs DIR writes, after the timed steps, the
similarity matrix the timed path computed in its last step as DIR/*.npy (float64; a fixed sample of its rows when the
whole matrix exceeds 32 MB). The inputs are generated from fixed seeds, so two builds run with the same arguments can be
compared output for output. The bench writes nothing into the source tree (which may be read-only).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # no __pycache__ in the source tree

# ---- workload: BASELINE.json configs[2] (headline) ---------------------------------------------------------------
WORKLOAD = dict(
    name="cfg3: 8000 cells x 0.5x, whole-genome-style pileup: %d sub-batches of 4 chromosomes x %d pre-filter loci per GPU "
         "and step, one similarity matrix per step",
    n_cells=int(os.environ.get("SECEDO_BENCH_CELLS", 8000)),
    coverage=float(os.environ.get("SECEDO_BENCH_COVERAGE", 0.5)),
    n_chr=4,
    loci_per_chr=int(os.environ.get("SECEDO_BENCH_LOCI_PER_CHR", 32768)),
    sub_batches=int(os.environ.get("SECEDO_BENCH_SUB_BATCHES", 4)),
    n_clones=2, frac_somatic=0.5, frac_germline=0.1, spacing=400,
    p_multi=float(os.environ.get("SECEDO_BENCH_P_MULTI", 0.005)),
    p_mate=float(os.environ.get("SECEDO_BENCH_P_MATE", 0.01)), p_mate_mismatch=0.2,
    # flags_sim of the reference: h = 0.15, theta = 0.001, eps = 0.01; with theta = 0.01 the reference's
    # filter accepts pure noise at this pooled coverage (SURVEY.md F7)
    theta=0.001, eps=0.01, h=0.15, L=1000, normalization="ADD_MIN",
)
CPU_SAMPLE_LOCI = int(os.environ.get("SECEDO_BENCH_CPU_LOCI", 28))  # pre-filter loci of the CPU sample
# BASELINE.json configs[4]: dense-filter stress, 20 000 cells at 1x (20 000 reads per locus), 1.6 GB int32 count planes;
# beyond the reference's 14-bit group ids -> wide pileups, and the CPU arm is the (widened) oracle port
CFG5 = dict(
    name="cfg5: 20000 cells x 1x (wide group ids), %d sub-batches of 4 chromosomes x %d pre-filter loci per GPU and step, one "
         "similarity matrix (1.6 GB int32 count planes) per step",
    n_cells=20000, coverage=1.0, loci_per_chr=int(os.environ.get("SECEDO_BENCH_LOCI_PER_CHR", 2048)),
    sub_batches=int(os.environ.get("SECEDO_BENCH_SUB_BATCHES", 2)), cpu_sample_loci=int(os.environ.get("SECEDO_BENCH_CPU_LOCI", 3)),
)


def select_workload(name):
    global CPU_SAMPLE_LOCI
    if name == "cfg5":
        WORKLOAD.update({k: v for k, v in CFG5.items() if k != "cpu_sample_loci"})
        CPU_SAMPLE_LOCI = CFG5["cpu_sample_loci"]
# human chromosome lengths (the reference's own table, pileup.cpp:30-34): proportions of the whole-genome workload
CHROMOSOME_LENGTHS = [248956422, 242193529, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636, 138394717,
                      133797422, 135086622, 133275309, 114364328, 107043718, 101991189, 90338345, 83257441, 80373285,
                      58617616, 64444167, 46709983, 50818468, 156040895]


def clocks_sampler(stop, out, device_index):
    """nvidia-smi sampled during the timed region (B200_PROFILING.md)."""
    q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    try:
        p = subprocess.Popen(["nvidia-smi", f"--id={device_index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                              "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except OSError:
        return
    def reader():
        for line in p.stdout:
            out.append(line.strip())
    t = threading.Thread(target=reader, daemon=True)
    t.start()
    stop.wait()
    p.terminate()


def summarize_clocks(lines):
    sm, mx, reasons = [], 0, set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for ln in lines:
        f = [x.strip() for x in ln.split(",")]
        if len(f) < 7:
            continue
        try:
            sm.append(float(f[0]))
            mx = max(mx, float(f[1]))
        except ValueError:
            continue
        for name, v in zip(names, f[3:7]):
            if v.lower().startswith("active"):
                reasons.add(name)
    return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
            "samples": len(sm)}


ALL_CPUS = None  # the cores this process was given, before bind_to_gpu_numa narrowed them


def bind_to_gpu_numa(torch, local_rank):
    """Run this rank, and allocate its pinned buffers, on the NUMA node its GPU hangs off (best effort: the container's
    cpuset may forbid it). Returns what was done, for the JSON line."""
    global ALL_CPUS
    info = {"numa_node": None, "cpus": None, "affinity_set": False, "mempolicy_set": False}
    try:
        ALL_CPUS = os.sched_getaffinity(0)
        pr = torch.cuda.get_device_properties(local_rank)
        bus = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        base = f"/sys/bus/pci/devices/{bus}"
        node = int(open(base + "/numa_node").read().strip())
        cpulist = open(base + "/local_cpulist").read().strip()
        cpus = set()
        for part in cpulist.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        info["numa_node"], info["pci"] = node, bus
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        info["cpus"] = len(use)
        if use and use != allowed:
            os.sched_setaffinity(0, use)
            info["affinity_set"] = True
        if node >= 0:
            libc = ctypes.CDLL(None, use_errno=True)
            mask = ctypes.c_ulong(1 << node)
            MPOL_PREFERRED, SYS_set_mempolicy = 1, 238  # x86_64
            if libc.syscall(SYS_set_mempolicy, MPOL_PREFERRED, ctypes.byref(mask), ctypes.c_ulong(64)) == 0:
                info["mempolicy_set"] = True
    except Exception as ex:  # noqa: BLE001
        info["error"] = f"{type(ex).__name__}: {ex}"
    return info


# ---------------------------------------------------------------------------------------- reference arm
def cpu_sample(seed=77):
    """A bounded sample of the workload, generated on the host (same model as the device generator)."""
    from secedo_b200.synth import SynthConfig, make_pileup
    w = WORKLOAD
    cfg = SynthConfig(n_cells=w["n_cells"], coverage=w["coverage"], n_loci=CPU_SAMPLE_LOCI, n_chr=1,
                      n_clones=w["n_clones"], frac_somatic=w["frac_somatic"], frac_germline=w["frac_germline"],
                      theta=w["theta"], spacing=w["spacing"], max_fragment_length=w["L"], p_multi=w["p_multi"],
                      p_mate=w["p_mate"], p_mate_mismatch=w["p_mate_mismatch"], seed=seed)
    return make_pileup(cfg)


def run_reference_step(p, threads, want_matrix=False):
    """Filter::filter + computeSimilarityMatrix of the reference on pileup p. Returns (seconds,
    significant loci, kind[, matrix])."""
    from oracle import pyoracle as po
    from secedo_b200.pileup import Pileup
    w = WORKLOAD
    ident = np.arange(w["n_cells"], dtype=np.uint32)
    if po.have_ref() and not p.wide:  # the reference holds 14-bit group ids: beyond them only the widened port exists
        t0 = time.perf_counter()
        rf, _, _ = po.ref_filter(p, ident, w["theta"], 4, threads)
        f = Pileup(rf.chr_ptr, rf.row_ptr, rf.position, rf.read_id, rf.gid_base)
        M, _ = po.ref_similarity(f, w["n_cells"], w["L"], ident, w["eps"], w["h"], w["theta"], threads, w["normalization"])
        secs = time.perf_counter() - t0
        return (secs, f.n_loci, "reference", M) if want_matrix else (secs, f.n_loci, "reference")
    t0 = time.perf_counter()
    kl, ke, _, _ = po.filter_flags(p, ident, w["theta"])
    f = p.select(kl, ke)
    o = po.similarity(f, w["n_cells"], w["L"], ident, w["eps"], w["h"], w["theta"], threads, w["normalization"],
                      instrument=False)
    secs = time.perf_counter() - t0
    return (secs, f.n_loci, "port", o.M) if want_matrix else (secs, f.n_loci, "port")


def reference_threads():
    """all host cores the process may use (torchrun exports OMP_NUM_THREADS=1; the reference takes its
    thread count as an argument, so that variable does not limit it). Also the `num_threads` BOTH arms pass to the
    path: it selects the reference's tail cutoff (SURVEY F2), so parity is defined at this value."""
    env = os.environ.get("SECEDO_BENCH_THREADS")
    if env:
        return max(1, int(env))
    if ALL_CPUS:
        return len(ALL_CPUS)
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


DUMP_MATRIX_BYTES = 32 << 20


def dump_matrix(out_dir, M):
    """The N x N similarity matrix as DIR/similarity_matrix_rows.npy (float64): all of its rows when they fit in
    DUMP_MATRIX_BYTES, else a sample of rows drawn with a fixed seed (the same rows for the same N), whose indices are
    DIR/similarity_matrix_row_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    n = M.shape[0]
    k = min(n, max(1, DUMP_MATRIX_BYTES // (8 * n)))
    rows = np.arange(n) if k == n else np.sort(np.random.default_rng(0).choice(n, k, replace=False))
    np.save(os.path.join(out_dir, "similarity_matrix_rows.npy"), np.ascontiguousarray(M[rows], dtype=np.float64))
    np.save(os.path.join(out_dir, "similarity_matrix_row_index.npy"), rows.astype(np.float64))


def host_matrix(rig, counts, epi, lik, normalization):
    """The matrix of the planes in `counts`: the epilogue the timed steps ran on them, once more, into host memory.
    Rank 0 gets it, the other ranks None."""
    if rig.world == 1:
        return counts.finalize(*lik, normalization)
    from secedo_b200 import dist as sdist
    shared = sdist.SharedHostMatrix(rig.ctx, counts.num_cells)
    epi.run(*lik, normalization, out_ptr=shared.dev_ptr, same_stream=True)
    rig.ctx.synchronize()
    rig.barrier()
    M = shared.array.copy() if rig.rank == 0 else None
    rig.barrier()
    shared.close()
    return M


def metric_name():
    w = WORKLOAD
    return "similarity-matrix significant loci/s (%dK cells, %gx)" % (w["n_cells"] // 1000, w["coverage"])


def workload_name():
    w = WORKLOAD
    return w["name"] % (w["sub_batches"], w["loci_per_chr"])


def main_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return 0
    threads = reference_threads()
    p = cpu_sample()
    times, loci, kind = [], 0, "reference"
    for i in range(args.warmup + args.steps):
        last = i == args.warmup + args.steps - 1
        r = run_reference_step(p, threads, want_matrix=bool(args.dump_outputs) and last)
        s, loci, kind = r[:3]
        if i >= args.warmup:
            times.append(s)
    if args.dump_outputs:
        dump_matrix(args.dump_outputs, r[3])
    total = sum(times)
    value = loci * len(times) / total
    sample = (f"{CPU_SAMPLE_LOCI} pre-filter loci ({loci} significant, {p.n_entries} pileup entries) of the workload per "
              f"step; Filter::filter + computeSimilarityMatrix, num_threads={threads}")
    line = {
        "impl": "reference", "metric": metric_name(), "value": value,
        "unit": "loci/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64 log-likelihoods over integer read-pair counts", "data": "synthetic",
        "config": {"workload": workload_name(), "sample": sample,
                   "n_cells": WORKLOAD["n_cells"], "coverage": WORKLOAD["coverage"], "num_threads": threads},
        "cpu_baseline": {"value": value, "unit": "loci/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "loci/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------ ours
def int8_peak_tops(torch, device):
    """Dense int8 tensor-core rate of cuBLASLt on this GPU (8192^3), the denominator the survey asks
    to measure because MEASURED_PEAKS.json only holds bf16. Returns (TOP/s, how)."""
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    bf16 = float(peaks.get("bf16_tflops", 1590.0))
    src_bf16 = "MEASURED_PEAKS.json bf16_tflops" if peaks else "fallback 1590 (B200_PROFILING.md)"
    try:
        tops, at = 0.0, 0
        for n in (8192, 16384):  # the larger problem amortises launch and tail effects: take the better one
            a = torch.randint(-8, 8, (n, n), dtype=torch.int8, device=device)
            b = torch.randint(-8, 8, (n, n), dtype=torch.int8, device=device)
            for _ in range(3):
                torch._int_mm(a, b)
            best = 1e9
            for _ in range(10):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                torch._int_mm(a, b)
                e1.record()
                e1.synchronize()
                best = min(best, e0.elapsed_time(e1))
            t = 2 * n ** 3 / (best * 1e-3) / 1e12
            if t > tops:
                tops, at = t, n
            del a, b
        return tops, bf16, f"torch._int_mm {at}^3 int8 (cuBLASLt), best of 10 over 8192^3 and 16384^3, measured in this run; bf16 from {src_bf16}"
    except Exception as ex:  # noqa: BLE001
        return 2 * bf16, bf16, f"2 x {src_bf16} (torch._int_mm unavailable: {type(ex).__name__})"


class Rig:
    """torch / distributed / library set-up shared by the bench modes"""

    def __init__(self):
        import torch
        import torch.distributed as dist
        from secedo_b200 import api
        self.torch, self.dist, self.api = torch, dist, api
        self.world = int(os.environ.get("WORLD_SIZE", 1))
        self.rank = int(os.environ.get("RANK", 0))
        self.local_rank = int(os.environ.get("LOCAL_RANK", 0))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: secedo_b200 has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.device = torch.device("cuda", self.local_rank)
        self.numa = bind_to_gpu_numa(torch, self.local_rank)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.device)
        self.ctx = api.Context(self.local_rank)
        # one explicit stream for everything: the library's kernels, the collectives and the timing events
        self.stream = torch.cuda.Stream(self.device)
        torch.cuda.set_stream(self.stream)
        self.ctx.set_stream(self.stream.cuda_stream)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], device=self.device, dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x):
        t = self.torch.tensor([x], device=self.device, dtype=self.torch.int64)
        if self.world > 1:
            self.dist.all_reduce(t)
        return int(t.item())

    def timed(self, fn, steps, warmup, finish=None):
        """W untimed + K timed steps bracketed by barrier + synchronize on both sides; CUDA events on the stream all
        work is ordered on; the MAX over ranks. finish() (e.g. waiting for the last matrix) runs inside the region."""
        torch = self.torch
        for _ in range(warmup):
            fn()
        if finish:
            finish()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stop, lines = threading.Event(), []
        th = threading.Thread(target=clocks_sampler, args=(stop, lines, self.local_rank), daemon=True)
        if self.rank == 0:
            th.start()
            time.sleep(0.25)  # let nvidia-smi come up BEFORE the barrier, so that all ranks start together
        self.barrier()
        torch.cuda.synchronize()
        self.ctx.tensor_times()  # tensor kernels of the warm-up steps: not part of the timed statistics
        launches0 = self.ctx.launch_count()
        acc = {}
        e0.record(self.stream)
        for _ in range(steps):
            st = fn()
            for k, v in st.items():
                if isinstance(v, (int, float)):
                    acc[k] = acc.get(k, 0) + v
        if finish:
            finish()
        # the first-order tensor kernels run on a stream of their own (beside the next sub-batch's filter / staging): the
        # region ends when the last of them has, and the ones no accumulate() statistics reported yet are added here
        ms_left, n_left = self.ctx.tensor_times()
        if "ms_gemm" in acc:
            acc["ms_gemm"] += ms_left
            acc["gemm_launches"] = acc.get("gemm_launches", 0) + n_left
        e1.record(self.stream)
        self.barrier()
        torch.cuda.synchronize()
        ms = self.max_over_ranks(e0.elapsed_time(e1))
        stop.set()
        return ms, acc, self.ctx.launch_count() - launches0, summarize_clocks(lines)


PHASES = ("ms_link", "ms_first_order", "ms_stage", "ms_gemm", "ms_multi", "gemm_launches")


def synth_sub_batch(ctx, rank, b):
    """sub-batch b of rank `rank` of the workload, generated in HBM from its own seed"""
    w = WORKLOAD
    return ctx.synth_pileup(w["n_cells"], w["coverage"], w["n_chr"], w["loci_per_chr"], n_clones=w["n_clones"],
                            frac_somatic=w["frac_somatic"], frac_germline=w["frac_germline"], theta=w["theta"],
                            spacing=w["spacing"], p_multi=w["p_multi"], p_mate=w["p_mate"],
                            p_mate_mismatch=w["p_mate_mismatch"], seed=1000 + 64 * rank + b)


def main_ours(args):
    from secedo_b200 import dist as sdist
    from secedo_b200.pileup import Pileup

    rig = Rig()
    torch, dist, api, ctx = rig.torch, rig.dist, rig.api, rig.ctx
    world, rank, device, stream = rig.world, rig.rank, rig.device, rig.stream
    w = WORKLOAD
    N, SUB = w["n_cells"], w["sub_batches"]
    threads = reference_threads()  # the num_threads of BOTH arms (selects the reference's tail cutoff)
    ident = np.arange(N, dtype=np.uint32)
    lik = (w["L"], w["eps"], w["h"], w["theta"])
    raw_dev = [synth_sub_batch(ctx, rank, b) for b in range(SUB)]
    dims = [r.dims() for r in raw_dev]
    n_chr = dims[0][0]
    P, E = sum(d[1] for d in dims), sum(d[2] for d in dims)
    flt = api.Filter(w["theta"], 4, ctx)
    counts = api.Counts(ctx, N)
    epi = sdist.SlabEpilogue(counts, device) if world > 1 else None
    last = {}
    # Consecutive steps of the device-resident run alternate between TWO sets of count planes, and the epilogue of a step is
    # issued after the first sub-batch of the next one: the last tensor kernel of a matrix (held back until the next
    # link_window kernel has been issued, DESIGN 4 "Scheduling") then runs beside the next matrix's first sub-batch instead
    # of alone in front of its epilogue (4.4 of 35 ms per step). Every step still filters and accumulates its four
    # sub-batches and produces its own matrix; the K-th matrix is finished by finish_prev() inside the timed region.
    # SECEDO_BENCH_PIPELINE_STEPS=0: one set of planes, the epilogue at the end of its own step.
    pipeline = os.environ.get("SECEDO_BENCH_PIPELINE_STEPS", "1") == "1"
    counts_ab = [counts, api.Counts(ctx, N)] if pipeline else [counts]
    epi_ab = [epi, (sdist.SlabEpilogue(counts_ab[1], device) if world > 1 else None)] if pipeline else [epi]
    pipe = {"i": 0, "prev": None, "ev": None}
    # Filter::filter of sub-batch k + 1 next to computeSimilarityMatrix of sub-batch k: a second context (own stream, own
    # host thread) filters ahead, so that its memory-bound kernels run under the tensor-bound GEMM of the sub-batch before
    # (they need 2 KB of shared memory per CTA and fit beside the GEMM's CTAs). Measured at N = 1: 42.30 against 42.62 ms per
    # step (profiles/r2_bench_overlap_ab.txt) - the filter slows the read linking it runs beside by as much as it hides
    # itself - so it is off by default; SECEDO_BENCH_OVERLAP=1 switches it on.
    overlap = os.environ.get("SECEDO_BENCH_OVERLAP", "0") == "1"
    ctx2 = api.Context(rig.local_rank) if overlap else None
    flt2 = api.Filter(w["theta"], 4, ctx2) if overlap else None

    def filtered_stream(sources):
        """the sources filtered in order; with `overlap` one sub-batch ahead on the second context's thread"""
        if not overlap or len(sources) < 2:
            for src in sources:
                yield flt.filter_device(src, ident)[0]
            return
        import queue
        q = queue.Queue(maxsize=1)
        def producer():
            try:
                for src in sources:
                    q.put(flt2.filter_device(src, ident)[0])
            except Exception as ex:  # noqa: BLE001
                q.put(ex)
        th = threading.Thread(target=producer, daemon=True)
        th.start()
        for _ in sources:
            item = q.get()
            if isinstance(item, Exception):
                raise item
            yield item
        th.join()

    def accumulate_all(sources, st, free_sources=False, top_up=None, into=None, after_first=None):
        feed = filtered_stream(sources) if not (free_sources or top_up) else None
        for n_done, src in enumerate(sources):
            filtered = next(feed) if feed else flt.filter_device(src, ident)[0]
            if top_up:
                top_up()
            s1 = (into or counts).accumulate(filtered, w["L"], ident, w["eps"], w["h"], w["theta"], threads, args.path)
            if after_first and n_done == 0:
                after_first()
            st["sig_loci"] = st.get("sig_loci", 0) + filtered.n_loci
            st["kept_entries"] = st.get("kept_entries", 0) + filtered.n_entries
            for k in PHASES:
                st[k] = st.get(k, 0) + (s1.get(k, 0) or 0)
            st["path_used"] = s1.get("path_used")
            filtered.free()
            if free_sources:
                src.free()

    def epilogue(st, out_ptr=None, out_host=None, async_out=False, which=0):
        """N x N matrix from the planes of all ranks. One GPU: the single-GPU epilogue. Several: the peer-memory epilogue
        (every rank its share; into the shared host matrix at out_ptr, or left in the ranks' HBM)."""
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record(stream)
        if world > 1:
            epi_ab[which].run(*lik, w["normalization"], out_ptr=out_ptr, same_stream=True)
        elif async_out:
            counts_ab[which].finalize_async(*lik, w["normalization"], out_host)
        else:
            counts_ab[which].finalize(*lik, w["normalization"], out=out_host, to_host=out_host is not None)
        r1.record(stream)
        st["_ev"] = (r0, r1)

    def finish_prev():
        """the epilogue of the step before (pipelined steps): its matrix"""
        if pipe["prev"] is not None:
            e = {}
            epilogue(e, which=pipe["prev"])
            pipe["prev"], pipe["ev"] = None, e["_ev"]

    def step_resident():
        st = {}
        k = pipe["i"] % len(counts_ab)
        pipe["i"] += 1
        counts_ab[k].zero()
        if pipeline:
            accumulate_all(raw_dev, st, into=counts_ab[k], after_first=finish_prev)
            pipe["prev"] = k
        else:
            accumulate_all(raw_dev, st)
            epilogue(st)
            pipe["ev"] = st.pop("_ev")
        if pipe["ev"] is not None:  # pipelined: the epilogue issued during this step (the matrix of the step before)
            r0, r1 = pipe["ev"]
            pipe["ev"] = None
            r1.synchronize()
            st["ms_epilogue_total"] = r0.elapsed_time(r1)
        last.update(st)
        return st

    # ---- device-resident input ------------------------------------------------------------------------
    l2_0 = ctx2.launch_count() if ctx2 else 0
    ms_dev, acc, launches, clocks = rig.timed(step_resident, args.steps, args.warmup, finish=finish_prev)
    if args.dump_outputs:  # now: the steps below overwrite the planes of the last timed step
        k = (pipe["i"] - 1) % len(counts_ab)
        M = host_matrix(rig, counts_ab[k], epi_ab[k], lik, w["normalization"])
        if rank == 0:
            dump_matrix(args.dump_outputs, M)
        del M
    if ctx2:  # warm-up launches of the second context are not part of the timed region
        launches += (ctx2.launch_count() - l2_0) * args.steps // (args.steps + args.warmup)
    sig_local = acc["sig_loci"] // args.steps
    sig_total = rig.sum_over_ranks(sig_local)
    # the tensor kernel ALONE (untimed, after the headline): in the timed region it shares the SMs with the next sub-batch's
    # special-entry chain / partition / staging kernels and takes longer per launch; two steps with the overlap switched off
    # give its time with the SMs to itself (the roofline reports both)
    overlapped = os.environ.get("SECEDO_B200_ASYNC_GEMM", "1") != "0"
    alone = None
    if overlapped:
        ctx.set_option("async_gemm", 0)
        step_resident()
        ctx.tensor_times()
        a2 = {"ms_gemm": 0.0, "gemm_launches": 0}
        for _ in range(2):
            st = step_resident()
            a2["ms_gemm"] += st["ms_gemm"]
            a2["gemm_launches"] += st["gemm_launches"]
        ms_left, n_left = ctx.tensor_times()
        a2["ms_gemm"] += ms_left
        a2["gemm_launches"] += n_left
        finish_prev()
        ctx.set_option("async_gemm", 1)
        alone = a2["ms_gemm"] / max(1, a2["gemm_launches"])

    # ---- verification of the multi-GPU result (untimed): the ranks' planes, summed through the peer mappings over the
    # shares the epilogue uses, carry the checksum of the planes the ranks accumulated
    reduce_checksum_ok = None
    if world > 1:
        own_sum, peer_sum = epi.checksums()
        reduce_checksum_ok = bool(own_sum == peer_sum)

    # ---- end to end: host (pinned) pileup in, host matrix out ------------------------------------------
    # The reference-facing call sequence with HOST buffers: every step uploads its whole pileup (one asynchronous upload
    # per chromosome on the library's copy stream, running ahead of the kernels; the read ids stay in pinned host memory
    # and the filter pulls those of the loci it keeps), filters and accumulates chromosome by chromosome into one counts
    # object, and delivers the N x N matrix into host memory: one GPU -> D2H on a stream of its own while the next step
    # starts; several GPUs -> every GPU writes its share of the matrix straight into a host matrix shared by the ranks.
    # All H2D / D2H bytes of all timed steps are inside the timed region.
    pinned = []
    def pin(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        pinned.append(t)
        return t.numpy()
    chunks, h2d_fixed, h2d_full = [], 0, 0
    # page-locked host copies of this rank's sub-batches: all of them, unless the ranks together would pin more than
    # 40 % of the host memory that is free (then the end-to-end step runs over the first sub-batches only, and says so)
    e2e_sub = SUB
    try:
        import psutil
        avail = psutil.virtual_memory().available
        per_sub = 6.2 * E / SUB
        while e2e_sub > 1 and world * e2e_sub * per_sub > 0.4 * avail:
            e2e_sub -= 1
    except Exception:  # noqa: BLE001
        pass
    for rd in raw_dev[:e2e_sub]:
        host = rd.download()
        pos_p, rid_p, gb_p = pin(host.position), pin(host.read_id), pin(host.gid_base)
        h2d_full += host.row_ptr.nbytes + host.position.nbytes + host.read_id.nbytes + host.gid_base.nbytes + host.chr_ptr.nbytes
        h2d_fixed += host.row_ptr.nbytes + host.position.nbytes + host.gid_base.nbytes + host.chr_ptr.nbytes
        for c in range(n_chr):
            l0, l1 = int(host.chr_ptr[c]), int(host.chr_ptr[c + 1])
            e0, e1 = int(host.row_ptr[l0]), int(host.row_ptr[l1])
            hp = Pileup.__new__(Pileup)  # views of the pinned arrays, no copies
            hp.chr_ptr = np.array([0, l1 - l0], np.uint64)
            hp.row_ptr = pin(host.row_ptr[l0:l1 + 1] - np.uint64(e0))
            hp.position, hp.read_id, hp.gid_base = pos_p[l0:l1], rid_p[e0:e1], gb_p[e0:e1]
            chunks.append(hp)
        del host
    n_chunks = len(chunks)
    shared = sdist.SharedHostMatrix(ctx, N) if world > 1 else None
    out_bufs = [None, None]
    if world == 1:
        # second result buffer: the matrix of step s travels to the host (own stream) while step s + 1 is computed
        out_bufs = [torch.empty((N, N), dtype=torch.float64).pin_memory().numpy() for _ in range(2)]
    e2e_steps = args.steps
    E2E_WARMUP = 2
    # uploads run up to LOOKAHEAD chromosomes ahead of the kernels, but never across the warm-up / timed boundary nor past
    # the last step: every timed step's H2D bytes are copied inside the timed region
    LOOKAHEAD = 4
    runs = [[(s, c) for s in range(E2E_WARMUP) for c in range(n_chunks)],
            [(s, c) for s in range(e2e_steps) for c in range(n_chunks)]]
    state = {"queue": [], "issued": 0, "run": [], "n_out": 0}

    def top_up(target):
        while len(state["queue"]) < target and state["issued"] < len(state["run"]):
            # read ids stay in pinned host memory: the filter pulls those of the loci it keeps (zero copy)
            chunk = chunks[state["run"][state["issued"]][1]]
            state["queue"].append(ctx.upload_async(chunk) if chunk.wide else ctx.upload_lazy_async(chunk))
            state["issued"] += 1

    def e2e_step():
        if state["issued"] == len(state["run"]) and not state["queue"]:  # next run (warm-up, then the timed steps)
            state["run"], state["issued"] = runs.pop(0), 0
        counts.zero()
        st = {}
        for _ in range(n_chunks):
            top_up(1)
            cur = state["queue"].pop(0)
            # DMA of the coming chromosomes is queued where the kernels leave the H2D direction of the bus idle
            # (accumulate, and the transfer of the matrix below), not next to the filter's zero-copy pull
            accumulate_all([cur], st, free_sources=True, top_up=lambda: top_up(2))
        state["n_out"] += 1
        top_up(LOOKAHEAD)
        epilogue(st, out_ptr=shared.dev_ptr if shared else None, out_host=out_bufs[state["n_out"] % 2], async_out=True)
        st.pop("_ev")
        state["pulled_entries"] = state.get("pulled_entries", 0) + st["kept_entries"]
        return st

    def e2e_finish():
        if world == 1:
            ctx.output_wait()  # the last matrix is complete in host memory
        else:
            ctx.synchronize()  # this rank's share has been written (the barrier of `timed` covers the other ranks)

    ms_e2e, acc_e2e, _, _ = rig.timed(e2e_step, e2e_steps, E2E_WARMUP, finish=e2e_finish)
    ctx.synchronize()
    # bytes that crossed PCIe host -> device per step: the CSR without the read ids, plus the read ids of the
    # entries of the loci the filter kept (all cells take part: every entry of a kept locus is pulled once)
    pulled = state.get("pulled_entries", 0) // (E2E_WARMUP + e2e_steps)
    h2d = h2d_full if chunks[0].wide else h2d_fixed + 4 * pulled  # wide pileups are uploaded whole
    d2h = N * N * 8 // world
    sig_e2e = rig.sum_over_ranks(acc_e2e["sig_loci"] // e2e_steps)
    assert e2e_sub < SUB or sig_e2e == sig_total, "the chromosome-wise end-to-end path must see the same significant loci"
    if rank == 0:
        M = shared.array if shared else out_bufs[state["n_out"] % 2]
        assert np.array_equal(M, M.T) and not np.diag(M).any() and np.isfinite(M).all(), \
            "result must be symmetric with a zero diagonal"
        assert M.min() == 0.0 and M.max() > 0.0, "ADD_MIN: the smallest entry is exactly 0"

    # ---- roofline of the dominant kernel (syrk2_kernel, tensor bound) ---------------------------------------
    ms_gemm_step = acc["ms_gemm"] / args.steps
    launches_gemm = max(1, int(acc["gemm_launches"]) // args.steps)
    alg_ops_step = 5.0 * N * N * sig_local                      # SURVEY.md §8(d): 5 N^2 per significant locus
    n_pad = ((N + 255) // 256) * 256
    n_tiles = sum(1 for cb in range(n_pad // 256) for rb in range(n_pad // 128)
                  if cb * 256 + 255 > rb * 128 and rb * 128 < N and cb * 256 < N)
    kbs = (sig_local + 31) // 32
    executed_ops_step = 2.0 * n_tiles * 128 * 256 * kbs * 128  # MACs x 2 the tcgen05 kernel issues: tiles x k-blocks of 128 B
    # ---- CPU baseline: the unmodified reference on a bounded sample (all cores; at N = 1 also one core), and the GPU path
    # on the SAME sample at the SAME num_threads, compared with the matrix of that very reference run. At N > 1 the sample
    # goes through the multi-GPU path: cut into one piece per rank inside its chromosome, accumulated by the ranks,
    # peer-memory epilogue into the shared host matrix.
    cpu, parity = None, None
    sample_p = cpu_sample()
    M_ref = None
    if rank == 0:
        if ALL_CPUS:
            os.sched_setaffinity(0, ALL_CPUS)  # the reference gets every core this process was given
        secs, cpu_loci, kind, M_ref = run_reference_step(sample_p, threads, want_matrix=True)
        what = f"{CPU_SAMPLE_LOCI} pre-filter loci ({cpu_loci} significant, {sample_p.n_entries} entries) of the same workload, " \
               f"Filter::filter + computeSimilarityMatrix"
        cpu = {"value": cpu_loci / secs, "unit": "loci/s", "cores": threads if kind == "reference" else 1, "kind": kind,
               "sample": f"{what}, {secs:.1f} s"}
        if world == 1:
            secs1 = secs if kind == "port" else run_reference_step(sample_p, 1)[0]  # the port is single-threaded anyway
            cpu["single_thread"] = {"value": cpu_loci / secs1, "unit": "loci/s", "cores": 1, "seconds": secs1,
                                    "note": "num_threads = 1 (SURVEY 8d: the reference often slows down with threads); its tail "
                                            "cutoff differs from the all-cores run, the significant loci are the same"}
    f_s, _ = flt.filter(sample_p, ident, "", threads)
    if world == 1:
        M_gpu = api.compute_similarity_matrix(f_s, N, w["L"], ident, w["eps"], w["h"], w["theta"], threads, "",
                                              w["normalization"], ctx=ctx, path=args.path)
    else:
        pos = [f_s.position[int(f_s.chr_ptr[c]):int(f_s.chr_ptr[c + 1])] for c in range(f_s.n_chr)]
        tail, ok = api.chromosome_cutoff(f_s, w["L"], threads, [True] * f_s.n_chr, ctx=ctx)
        piece = sdist.plan_pieces(pos, world, w["L"])[rank]
        counts.zero()
        if piece:
            counts.accumulate_range(Pileup.concat([f_s.loci_range(d["chrom"], d["lo"], d["hi"]) for d in piece]), w["L"], ident,
                                    w["eps"], w["h"], w["theta"], [d["own_pos_begin"] for d in piece],
                                    [d["own_pos_end"] for d in piece], [tail[d["chrom"]] for d in piece], args.path)
        epi.run(*lik, w["normalization"], out_ptr=shared.dev_ptr, same_stream=True)
        ctx.synchronize()
        rig.barrier()
        M_gpu = shared.array
    if rank == 0:
        scale = float(np.abs(M_ref).max())
        diff = float(np.abs(M_gpu - M_ref).max())
        parity = {"ok": bool(f_s.n_loci == cpu_loci and diff <= 1e-6 * max(scale, 1e-300)), "max_abs_diff": diff,
                  "max_abs_reference": scale, "tolerance": "1e-6 * max|M_reference|", "num_threads": threads,
                  "significant_loci": int(f_s.n_loci), "reference_kind": kind, "n_gpus": world,
                  "what": "Filter::filter + computeSimilarityMatrix through the C ABI on the CPU baseline's sample (same cell "
                          "count as the workload" + (f", cut into {world} pieces, one per rank, peer-memory epilogue" if world > 1 else "")
                          + "), against the matrix of that CPU run"}
        assert parity["ok"], f"GPU path differs from the reference on the baseline sample: {parity}"
    rig.barrier()
    line = None
    if rank == 0:
        int8_peak, bf16_peak, how = int8_peak_tops(torch, device)
        achieved = alg_ops_step / (ms_gemm_step * 1e-3) / 1e12 if ms_gemm_step > 0 else 0.0
        # DRAM bytes of one launch from the committed ncu capture of this exact per-launch workload
        traffic, tensor_active, traffic_src = None, None, None
        for name in ("r2_syrk_traffic.json", "r1_syrk_traffic.json"):
            try:
                tr = json.load(open(os.path.join(ROOT, "profiles", name)))
                tw = tr["workload"]
                if (tw["n_cells"], tw["n_chr"], tw["loci_per_chr"], tw["coverage"]) == (N, w["n_chr"], w["loci_per_chr"], w["coverage"]):
                    traffic = tr["dram_bytes_read"] + tr["dram_bytes_write"]
                    tensor_active = tr.get("tensor_pipe_active_pct")
                    traffic_src = f"profiles/{name} (ncu, dram__bytes_read.sum + dram__bytes_write.sum of one launch)"
                    break
            except Exception:  # noqa: BLE001
                pass
        NOMINAL_INT8 = 4500.0  # dense int8 TOP/s of a B200 (B200_PROFILING.md: 2 x the 2.25 PFLOP/s bf16 figure)
        roofline = {
            "bound": "tensor", "kernel": "syrk2_kernel (tcgen05.mma.cta_group::2.kind::i8)", "achieved": achieved, "peak": int8_peak,
            "unit": "TFLOP/s", "frac": achieved / int8_peak if int8_peak else None, "traffic": traffic,
            "op": "int8 multiply-add = 2 ops; algorithmic ops = 5*N^2 per significant locus (SURVEY 8d); the kernel "
                  "issues 4*N_pad^2*(upper-triangle tiles) of them (Hadamard planes: 4 K-slices per 32 loci instead of 5)",
            "peak_source": how, "bf16_peak_measured": bf16_peak,
            "launches_per_step": launches_gemm, "avg_launch_ms": ms_gemm_step / launches_gemm,
            "overlapped": overlapped, "avg_launch_ms_alone": alone,
            "achieved_alone": (alg_ops_step / launches_gemm / (alone * 1e-3) / 1e12) if alone else None,
            "frac_alone": (alg_ops_step / launches_gemm / (alone * 1e-3) / 1e12 / int8_peak) if alone and int8_peak else None,
            "algorithmic_ops_per_launch": alg_ops_step / launches_gemm,
            "executed_ops_frac_of_algorithmic": executed_ops_step / alg_ops_step if alg_ops_step else None,
            "achieved_executed": achieved * executed_ops_step / alg_ops_step if alg_ops_step else None,
            "frac_executed": (achieved * executed_ops_step / alg_ops_step / int8_peak) if alg_ops_step and int8_peak else None,
            "kernel_share_of_step": ms_gemm_step / (ms_dev / args.steps),
            "nominal_peak": NOMINAL_INT8,
            "frac_executed_of_nominal": (achieved * executed_ops_step / alg_ops_step / NOMINAL_INT8) if alg_ops_step else None,
            "tensor_pipe_active_pct_ncu": tensor_active,
            "note": "`achieved` / `frac` / `avg_launch_ms` are measured live in the timed region, where the kernel runs on its own "
                    "stream BESIDE the next sub-batch's special-entry chain, partition and staging kernels (they take shared "
                    "memory, registers and DRAM bandwidth on the same SMs: slower per launch, but off the critical path; "
                    "kernel_share_of_step is then the share of the step during which the tensor pipe is busy); *_alone: the same "
                    "kernel with the SMs to itself. frac > 1: `achieved` counts SURVEY's algorithmic ops, the Hadamard form issues 0.86 of them; and the "
                    "measured cuBLASLt int8 peak (like the bf16 one in MEASURED_PEAKS.json, 74 % of nominal) is a long "
                    "power-capped GEMM loop, while this kernel runs for a few ms between memory-bound kernels. In issued "
                    "ops it reaches frac_executed_of_nominal of the 4.5 POP/s dense int8 rate",
            "traffic_source": traffic_src,
        }
        # ---- the same path through the C++ drop-in shim (what an unmodified SECEDO calls): pageable vector<vector<PosData>>
        # in, Matd out, host-side flattening and rebuilding inside the timed calls; a quarter sub-batch of the workload's shape
        e2e_shim = None
        if not args.skip_extras and world == 1:
            try:
                import subprocess
                import tempfile
                import __graft_entry__ as ge
                with tempfile.TemporaryDirectory() as tmp:
                    # the driver build() left next to the library if it is fresh, else one compiled outside the tree
                    # (which may be read-only)
                    exe = ge.build_shim_bench(tmp)
                    env = dict(os.environ, SECEDO_B200_DEVICES=str(rig.local_rank))
                    r = subprocess.run([exe, str(N), str(w["coverage"]), "4",
                                        str(int(os.environ.get("SECEDO_BENCH_SHIM_LOCI", 8192))), str(threads), "2"],
                                       capture_output=True, text=True, timeout=600, env=env)
                e2e_shim = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else {"error": (r.stderr or r.stdout)[-300:]}
            except Exception as ex:  # noqa: BLE001
                e2e_shim = {"error": str(ex)[-300:]}
        # ---- SURVEY 8(f) row 3: Laplacian + the 7 leading eigenpairs of a matrix of this workload, resident in HBM ----
        spectral, em = None, None
        if not args.skip_extras and world == 1:
            try:
                one = api.Counts(ctx, N)
                f1, _ = flt.filter_device(raw_dev[0], ident)
                one.accumulate(f1, w["L"], ident, w["eps"], w["h"], w["theta"], threads, args.path)
                runs_ = []
                for _ in range(3):
                    t0 = time.perf_counter()
                    ev, _, sst, _ = one.finalize_spectral(*lik, w["normalization"], k=7, tol=1e-10)
                    sst["wall_ms"] = (time.perf_counter() - t0) * 1e3
                    runs_.append(sst)
                one.free()
                best = min(runs_[1:], key=lambda r: r["wall_ms"])
                hbm = 6650.0
                try:
                    hbm = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
                except Exception:  # noqa: BLE001
                    pass
                gbs = 8.0 * N * N * best["matvec_launches"] / (best["ms_matvec"] * 1e-3) / 1e9
                spectral = {"what": "epilogue + laplacian() + the 7 smallest eigenpairs (spectral_clustering.cpp:33-52,127-138), "
                                    "similarity matrix never leaves HBM; residuals <= 1e-10", "k": 7,
                            "ms": best["wall_ms"], "ms_solver": best["ms_solver"], "ms_laplacian": best["ms_laplacian"],
                            "outer_iterations": best["outer_iterations"], "block": best["block"],
                            "block_products": best["matvec_launches"], "max_residual": best["max_residual"],
                            "eigenvalues": [float(x) for x in ev],
                            "roofline": {"bound": "hbm", "kernel": "symm_block_kernel (fp64, M read once per product)",
                                         "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm,
                                         "avg_launch_ms": best["ms_matvec"] / best["matvec_launches"],
                                         "algorithmic_bytes_per_launch": 8.0 * N * N}}
                # ---- SURVEY 8(f) row 4: EM refinement on a filtered sub-batch (device resident) -------------------
                start = np.random.default_rng(1).uniform(0.3, 0.7, N)
                EM_IT = 4
                api.expectation_maximization(f1, ident, 1, w["theta"], start, ctx=ctx, max_iterations=1)  # warm
                _, est = api.expectation_maximization(f1, ident, 1, w["theta"], start, ctx=ctx, max_iterations=EM_IT,
                                                      return_stats=True)
                n_ent = f1.n_entries
                f1.free()
                gpu_eps = n_ent * est["iterations"] / (est["ms"] * 1e-3)
                em = {"what": "expectation_maximization (expectation_maximization.cpp:131-160) on a filtered sub-batch in HBM, "
                              f"{EM_IT} iterations incl. H2D/D2H of the probabilities", "entries": int(n_ent),
                      "ms_per_iteration": est["ms"] / est["iterations"], "entries_per_s": gpu_eps,
                      "algorithmic_bytes_per_entry": 4, "achieved_GBps": 4.0 * gpu_eps / 1e9,
                      "bound": "L2 reductions (one RED.ADD.64 per entry) + two dependent gathers per entry"}
            except Exception as ex:  # noqa: BLE001
                spectral = spectral or {"error": f"{type(ex).__name__}: {ex}"}
                em = em or {"error": f"{type(ex).__name__}: {ex}"}
        # ---- CPU baseline: the unmodified reference on a bounded sample, all cores and one core; and the GPU path on
        # the SAME sample at the SAME num_threads, compared with the matrix of that very reference run ---------------
        value = sig_total * args.steps / (ms_dev * 1e-3)
        e2e_value = sig_e2e * e2e_steps / (ms_e2e * 1e-3)
        line = {
            "metric": metric_name(), "value": value, "unit": "loci/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int8 tensor-core counts (int32 accumulate) + f64 log-likelihood epilogue", "data": "synthetic",
            "config": {
                "workload": workload_name(), "n_cells": N, "coverage": w["coverage"],
                "prefilter_loci_per_gpu_step": P, "significant_loci_per_step_all_gpus": sig_total,
                "pileup_entries_per_gpu_step": E, "sub_batches_per_step": SUB, "p_multi": w["p_multi"], "p_mate": w["p_mate"],
                "theta": w["theta"], "eps": w["eps"], "h": w["h"], "max_fragment_length": w["L"],
                "num_threads_for_cutoff": threads, "normalization": w["normalization"],
                "path": last.get("path_used"), "filter_overlaps_previous_gemm": overlap,
                "tensor_kernel_overlaps_next_sub_batch": os.environ.get("SECEDO_B200_ASYNC_GEMM", "1") != "0",
                "steps_pipelined_over_two_sets_of_count_planes": pipeline,
                "parallelism": f"loci sharded by chromosome over {world} GPU(s); per step every GPU accumulates its "
                               f"{SUB} sub-batches into its own int32 count planes" + (
                    ", then the peer-memory epilogue: each GPU sums the planes of all GPUs over 1/%d of the matrix through "
                    "NVLink (CUDA IPC mappings) and transforms them in the same kernel; one all-reduce of two doubles" % world
                    if world > 1 else ", single-GPU epilogue"),
                "result": ("each rank's share of the N x N matrix in its own HBM (value) / one N x N matrix in host memory "
                           "shared by the ranks (e2e)" if world > 1 else "N x N matrix in HBM (value) / in host memory (e2e)"),
                "l2": "inputs larger than L2 (pileup %.1f GB, Hadamard panel %.1f GB per sub-batch)" % (
                    h2d_full / 1e9, 4.0 * N * sig_local / SUB / 1e9),
                "host_topology": rig.numa,
            },
            "build_time_s_per_step": ms_dev / args.steps * 1e-3,
            "prefilter_loci_per_s": P * world * args.steps / (ms_dev * 1e-3),
            "phase_ms_per_step_rank0": dict({k: acc[k] / args.steps for k in ("ms_link", "ms_first_order", "ms_stage", "ms_gemm",
                                                                               "ms_multi")},
                                            ms_epilogue=acc["ms_epilogue_total"] / args.steps),
            "roofline": roofline, "cpu_baseline": cpu, "parity_vs_reference": parity,
            "reduce_checksum_ok": reduce_checksum_ok,
            "e2e": {"value": e2e_value, "unit": "loci/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": ms_e2e / e2e_steps, "steps": e2e_steps, "sub_batches_per_step": e2e_sub,
                    "significant_loci_per_step_all_gpus": sig_e2e,
                    "host_pileup_bytes_per_step": int(h2d_full),
                    "how": "host pinned pileup -> sgpu_pileup_upload_lazy_async per chromosome (copy stream, running ahead of "
                           "the kernels; the read ids stay in pinned host memory) -> filter (pulls the read ids of the loci it "
                           "keeps straight over PCIe: h2d_bytes_per_step counts what crossed the bus, "
                           "host_pileup_bytes_per_step the whole input) -> accumulate -> epilogue -> N x N fp64 matrix in host "
                           "memory, every step (per rank: d2h_bytes_per_step = its share)"},
            "gpu_launches": int(launches), "clocks": clocks, "e2e_shim": e2e_shim, "spectral": spectral, "em": em,
        }
        print(json.dumps(line))
    rig.barrier()
    if shared:
        shared.close()
    if epi:
        epi.close()
    if pipeline and epi_ab[1]:
        epi_ab[1].close()
    if world > 1:
        dist.destroy_process_group()
    return 0


# --------------------------------------------------------------------------------------- whole genome, strong scaling
def main_genome(args):
    """BASELINE.json configs[2] as ONE job: 23 chromosomes with the human length ratios (pileup.cpp:30-34), 8 000 cells at
    0.5x, cut into segments of 32 768 pre-filter loci INSIDE the chromosomes, contiguous runs of segments per GPU
    (balanced to one segment), accumulated into one set of count planes per GPU through sgpu_counts_accumulate_range
    (a segment that ends a chromosome decides that chromosome's tail cutoff, the others have none), ONE peer-memory
    epilogue at the end. Strong scaling: the same genome at every N; `value` = significant loci of the whole genome /
    seconds for the whole matrix. SECEDO_BENCH_GENOME_LOCI sets the pre-filter loci of the genome: default 1.63 M (40 GB
    of pileup, resident in HBM at every N); 16 300 000 is the real size (~8 M significant loci, 390 GB): a GPU whose
    share does not fit in HBM regenerates every batch of segments in front of its timed region and the per-batch device
    times (CUDA events) are added up — the generator is not part of the path."""
    from secedo_b200 import dist as sdist
    rig = Rig()
    torch, dist, api, ctx = rig.torch, rig.dist, rig.api, rig.ctx
    world, rank, device, stream = rig.world, rig.rank, rig.device, rig.stream
    w = WORKLOAD
    N = w["n_cells"]
    threads = reference_threads()
    ident = np.arange(N, dtype=np.uint32)
    lik = (w["L"], w["eps"], w["h"], w["theta"])
    SEG, PER_CALL = 32768, 4
    total_len = float(sum(CHROMOSOME_LENGTHS))
    G = int(os.environ.get("SECEDO_BENCH_GENOME_LOCI", round(131072 * total_len / CHROMOSOME_LENGTHS[0])))
    n_seg = [max(1, int(round(G * x / total_len / SEG))) for x in CHROMOSOME_LENGTHS]
    segments = [(c, k) for c, n in enumerate(n_seg) for k in range(n)]       # in genome order
    all_calls = [segments[i:i + PER_CALL] for i in range(0, len(segments), PER_CALL)]  # the same batches whatever N
    n_calls_all = len(all_calls)
    lo, hi = len(all_calls) * rank // world, len(all_calls) * (rank + 1) // world
    calls = [(lo + i, call) for i, call in enumerate(all_calls[lo:hi])]
    bytes_per_call = PER_CALL * SEG * N * w["coverage"] * 6.1
    resident = len(calls) * bytes_per_call < float(os.environ.get("SECEDO_BENCH_RESIDENT_BYTES", 110e9))

    def generate(call):
        # the (up to 4) segments of a batch are the "chromosomes" of one device pileup; the seed names the batch
        # -> the same genome whatever the number of GPUs
        idx, segs = call
        return ctx.synth_pileup(N, w["coverage"], len(segs), SEG, n_clones=w["n_clones"], frac_somatic=w["frac_somatic"],
                                frac_germline=w["frac_germline"], theta=w["theta"], spacing=w["spacing"], p_multi=w["p_multi"],
                                p_mate=w["p_mate"], p_mate_mismatch=w["p_mate_mismatch"], seed=7000 + idx)

    flt = api.Filter(w["theta"], 4, ctx)
    counts = api.Counts(ctx, N)
    epi = sdist.SlabEpilogue(counts, device) if world > 1 else None
    raw = [generate(call) for call in calls] if resident else None
    def accumulate_call(call, src, st):
        segs = call[1]
        filtered, _ = flt.filter_device(src, ident)
        # every segment is owned whole; only a segment that ends a chromosome has tail reads, and decides them itself
        tails = [api.TAIL_AUTO if k == n_seg[c] - 1 else api.TAIL_NONE for c, k in segs]
        s1 = counts.accumulate_range(filtered, w["L"], ident, w["eps"], w["h"], w["theta"], [0] * len(segs),
                                     [api.TAIL_NONE] * len(segs), tails, args.path, num_threads=threads)
        st["sig_loci"] += filtered.n_loci
        st["ms_gemm"] += s1["ms_gemm"]
        st["gemm_launches"] += s1["gemm_launches"]
        filtered.free()

    def finish(st):
        if world > 1:
            epi.run(*lik, w["normalization"], same_stream=True)
        else:
            counts.finalize(*lik, w["normalization"], to_host=False)

    def genome_resident():
        st = {"sig_loci": 0, "ms_gemm": 0.0, "gemm_launches": 0}
        counts.zero()
        for call, parts in zip(calls, raw):
            accumulate_call(call, parts, st)
        finish(st)
        return st

    steps, warmup = args.steps, args.warmup
    if resident:
        ms, acc, launches, clocks = rig.timed(genome_resident, steps, warmup)
        how = "whole share resident in HBM; barrier + events around the whole genome, max over ranks"
    else:
        # `steps` passes (after a one-call warm-up): every batch of segments is generated, then timed on its own
        warmup = 0
        st = {"sig_loci": 0, "ms_gemm": 0.0, "gemm_launches": 0}
        parts = generate(calls[0])
        counts.zero()
        accumulate_call(calls[0], parts, dict(st))
        ctx.tensor_times()
        parts.free()
        stop, lines = threading.Event(), []
        th = threading.Thread(target=clocks_sampler, args=(stop, lines, rig.local_rank), daemon=True)
        if rank == 0:
            th.start()
        rig.barrier()
        launches0 = ctx.launch_count()
        ms = 0.0
        for _ in range(steps):
            counts.zero()
            ms_local = 0.0
            for call in calls:
                parts = generate(call)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                accumulate_call(call, parts, st)
                # this batch's tensor kernel (on its own stream) belongs to this batch's timed region: wait for it, so that
                # it does not run hidden under the untimed generation of the next batch
                ms_left, n_left = ctx.tensor_times()
                st["ms_gemm"] += ms_left
                st["gemm_launches"] += n_left
                e1.record(stream)
                e1.synchronize()
                ms_local += e0.elapsed_time(e1)
                parts.free()
            rig.barrier()  # the slowest rank's accumulation ends here
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            finish(st)
            e1.record(stream)
            torch.cuda.synchronize()
            ms += rig.max_over_ranks(ms_local) + rig.max_over_ranks(e0.elapsed_time(e1))
        stop.set()
        acc, launches, clocks = st, ctx.launch_count() - launches0, summarize_clocks(lines)
        how = ("share larger than HBM: every batch of 4 segments generated in front of its own timed region; time = max over "
               "ranks of the summed per-batch device times + the epilogue, summed over the steps")
    if args.dump_outputs:
        M = host_matrix(rig, counts, epi, lik, w["normalization"])
        if rank == 0:
            dump_matrix(args.dump_outputs, M)
        del M
    sig_local = acc["sig_loci"] // steps
    sig_total = rig.sum_over_ranks(sig_local)
    ok = None
    if world > 1:
        a, b = epi.checksums()
        ok = bool(a == b)
    if rank == 0:
        secs = ms / steps * 1e-3
        line = {
            "metric": "similarity-matrix significant loci/s (8K cells, 0.5x, whole genome)", "value": sig_total / secs,
            "unit": "loci/s", "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms / steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int8 tensor-core counts (int32 accumulate) + f64 log-likelihood epilogue", "data": "synthetic",
            "whole_genome_matrix_seconds": secs,
            "config": {"workload": f"cfg3-genome: 8000 cells x 0.5x, 23 chromosomes with the human length ratios in segments of "
                                   f"{SEG} pre-filter loci, {len(segments) * SEG} pre-filter loci ({sig_total} significant); one "
                                   "step = the whole matrix",
                       "n_cells": N, "coverage": w["coverage"], "segments_per_chromosome": n_seg,
                       "batches_of_4_segments_per_gpu": [n_calls_all * (r + 1) // world - n_calls_all * r // world for r in range(world)],
                       "num_threads_for_cutoff": threads, "p_multi": w["p_multi"], "timing": how,
                       "parallelism": f"contiguous runs of segments (pieces of chromosomes) over {world} GPU(s), "
                                      "sgpu_counts_accumulate_range; one epilogue over peer memory at the end",
                       "host_topology": rig.numa},
            "gemm_ms_per_genome_rank0": acc["ms_gemm"] / steps, "reduce_checksum_ok": ok,
            "gpu_launches": int(launches), "clocks": clocks,
        }
        print(json.dumps(line))
    rig.barrier()
    if epi:
        epi.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--path", default="auto", choices=["auto", "scatter", "gemm"])
    ap.add_argument("--workload", default="cfg3", choices=["cfg3", "cfg3-genome", "cfg5"])
    ap.add_argument("--skip-extras", action="store_true", help="skip the spectral / EM side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the similarity matrix of the last timed step to DIR/*.npy")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    select_workload(a.workload)
    if a.workload == "cfg5":
        a.skip_extras = True  # the eigen-solver / EM side measurements belong to the headline workload
    if a.impl == "reference":
        sys.exit(main_reference(a))
    if a.workload == "cfg3-genome":
        sys.exit(main_genome(a))
    sys.exit(main_ours(a))
