"""One device-resident hot-path step of the bench workload per iteration (filter -> accumulate -> finalize), nothing else:
the command that the ncu captures of the hot-path kernels wrap.   python profiles/hot_step.py [iterations]
Env knobs of the library (SECEDO_B200_ASYNC_GEMM, SECEDO_B200_PREFER_SHARED, ...) apply."""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from secedo_b200 import api
w = bench.WORKLOAD
iters = int(sys.argv[1]) if len(sys.argv) > 1 else 2
ctx = api.Context(0)
N = w["n_cells"]; ident = np.arange(N, dtype=np.uint32)
raw = ctx.synth_pileup(N, w["coverage"], w["n_chr"], w["loci_per_chr"], n_clones=w["n_clones"], frac_somatic=w["frac_somatic"],
                       frac_germline=w["frac_germline"], theta=w["theta"], spacing=w["spacing"], p_multi=w["p_multi"],
                       p_mate=w["p_mate"], p_mate_mismatch=w["p_mate_mismatch"], seed=1000)
flt = api.Filter(w["theta"], 4, ctx); counts = api.Counts(ctx, N)
for it in range(iters):
    f, _ = flt.filter_device(raw, ident)
    counts.zero()
    st = counts.accumulate(f, w["L"], ident, w["eps"], w["h"], w["theta"], 8, "auto")
    f.free()
    counts.finalize(w["L"], w["eps"], w["h"], w["theta"], "ADD_MIN", to_host=False)
    print(it, {k: (round(v, 3) if isinstance(v, float) else v) for k, v in st.items()}, flush=True)
ctx.synchronize()
