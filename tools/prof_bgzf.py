import os, sys, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from vcfgl_b200 import capi
wl = bench.Workload(sys.argv[1] if len(sys.argv) > 1 else "cfg2")
a = wl.sim_args(); gt, _ = wl.genotypes(1)
ctx = capi.Context(capi.params_from_args(a, wl.S, max_batch_sites=wl.B, n_slots=1, host_output=capi.HOST_BGZF, bcf_dict=dict(DP=1, GL=2, PL=3, GP=4, AD=5, ADF=6, ADR=7, QS=8, I16=9)))
sin, _ = ctx.bcf_input(0)
for i in range(3):
    ctx.input_buffer(0)[:] = gt
    sin["pos"][:wl.B] = np.arange(wl.B); sin["qual_bits"][:wl.B] = capi.F32_MISSING_BITS
    ctx.submit(0, i * wl.B, wl.B)
    b = ctx.wait(0)
print("raw", b.bcf_bytes, "bgzf", b.bgzf_bytes, "ratio", b.bcf_bytes / b.bgzf_bytes, "B/cell", b.bgzf_bytes / (wl.B * wl.S))
try:      # the per-phase counters of the development build (make -C vcfgl_b200/csrc bgzfprof; VGL_LIB=build/variants/libvgl_bgzfprof.so)
    capi.load().vgl_bgzf_prof_dump()
except AttributeError:
    pass
