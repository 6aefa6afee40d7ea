"""Device-resident hot-path steps of the bench workload (4 sub-batches -> one matrix per step), nothing else: A/B probe for
the library's env knobs that are read at context creation (SECEDO_B200_ASYNC_GEMM, SECEDO_B200_PREFER_SHARED,
...).   python profiles/overlap_probe.py [steps] [warmup] [label]
Prints one JSON line: ms per step (host clock around synchronised regions), per-phase device times, tensor kernel average,
and a checksum of the count planes of the last step (must not depend on the knobs)."""
import json, os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from secedo_b200 import api

w = bench.WORKLOAD
steps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
warmup = int(sys.argv[2]) if len(sys.argv) > 2 else 2
label = sys.argv[3] if len(sys.argv) > 3 else ""
ctx = api.Context(0)
N, SUB = w["n_cells"], w["sub_batches"]
ident = np.arange(N, dtype=np.uint32)
raw = [ctx.synth_pileup(N, w["coverage"], w["n_chr"], w["loci_per_chr"], n_clones=w["n_clones"], frac_somatic=w["frac_somatic"],
                        frac_germline=w["frac_germline"], theta=w["theta"], spacing=w["spacing"], p_multi=w["p_multi"],
                        p_mate=w["p_mate"], p_mate_mismatch=w["p_mate_mismatch"], seed=1000 + b) for b in range(SUB)]
flt = api.Filter(w["theta"], 4, ctx)
counts = api.Counts(ctx, N)
KEYS = ("ms_link", "ms_first_order", "ms_stage", "ms_gemm", "ms_multi", "gemm_launches")


def step(acc):
    counts.zero()
    for src in raw:
        f, _ = flt.filter_device(src, ident)
        st = counts.accumulate(f, w["L"], ident, w["eps"], w["h"], w["theta"], 24, "gemm")
        f.free()
        acc["sig"] = acc.get("sig", 0) + st["n_loci"]
        for k in KEYS:
            acc[k] = acc.get(k, 0) + st[k]
    counts.finalize(w["L"], w["eps"], w["h"], w["theta"], "ADD_MIN", to_host=False)


for _ in range(warmup):
    step({})
ctx.synchronize()
ctx.tensor_times()
acc = {}
t0 = time.perf_counter()
for _ in range(steps):
    step(acc)
ms_left, n_left = ctx.tensor_times()
ctx.synchronize()
t1 = time.perf_counter()
acc["ms_gemm"] += ms_left
acc["gemm_launches"] += n_left
chk = counts.checksum()
out = {"label": label, "env": {k: v for k, v in os.environ.items() if k.startswith("SECEDO_B200_")},
       "ms_per_step": (t1 - t0) * 1e3 / steps, "ms_per_sub_batch": (t1 - t0) * 1e3 / steps / SUB,
       "sig_loci_per_s": acc["sig"] / (t1 - t0),
       "phase_ms_per_step": {k: acc[k] / steps for k in KEYS},
       "gemm_avg_ms": acc["ms_gemm"] / max(1, acc["gemm_launches"]), "checksum": int(chk)}
print(json.dumps(out), flush=True)
