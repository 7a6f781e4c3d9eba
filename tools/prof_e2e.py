"""tools/prof_e2e.py <workload> [mode] -- wall-clock breakdown of the end-to-end loop (fill / submit / wait per batch)"""
import os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from vcfgl_b200 import capi
wl = bench.Workload(sys.argv[1] if len(sys.argv) > 1 else "cfg5")
mode = {"bgzf": capi.HOST_BGZF, "bcf": capi.HOST_BCF, "narrow": capi.HOST_NARROW}[sys.argv[2] if len(sys.argv) > 2 else "bgzf"]
a = wl.sim_args(); gt, _ = wl.genotypes(1)
NS = int(sys.argv[3]) if len(sys.argv) > 3 else 3
ctx = capi.Context(capi.params_from_args(a, wl.S, max_batch_sites=wl.B, n_slots=NS, host_output=mode, bcf_dict=dict(DP=1, GL=2, PL=3, GP=4, AD=5, ADF=6, ADR=7, QS=8, I16=9)))
bufs = [ctx.input_buffer(s) for s in range(NS)]
sins = [ctx.bcf_input(s)[0] for s in range(NS)] if mode != capi.HOST_NARROW else None
pend = []
t_fill = t_sub = t_wait = 0.0
N = 14
t00 = None
for i in range(N):
    if i == 2:
        t00 = time.perf_counter(); t_fill = t_sub = t_wait = 0.0
    s = i % NS
    t0 = time.perf_counter()
    if len(pend) == NS:
        ctx.wait(pend.pop(0))
    t1 = time.perf_counter()
    bufs[s][:] = gt
    if sins:
        sins[s]["pos"][:wl.B] = np.arange(wl.B); sins[s]["qual_bits"][:wl.B] = capi.F32_MISSING_BITS
    t2 = time.perf_counter()
    ctx.submit(s, i * wl.B, wl.B)
    t3 = time.perf_counter()
    pend.append(s)
    t_wait += t1 - t0; t_fill += t2 - t1; t_sub += t3 - t2
for s in pend:
    t0 = time.perf_counter(); ctx.wait(s); t_wait += time.perf_counter() - t0
tot = time.perf_counter() - t00
nb = N - 2
print("per batch: total %.1f ms = wait %.1f + fill %.1f + submit %.1f ; %.3g cells/s" % (1e3 * tot / nb, 1e3 * t_wait / nb, 1e3 * t_fill / nb, 1e3 * t_sub / nb, nb * wl.B * wl.S / tot))
for s in range(NS):
    print("slot", s, "timing ms [h2d sim site scan emit d2h total]:", np.round(ctx.timing(s), 2))
