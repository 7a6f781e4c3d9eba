#!/usr/bin/env python3
"""bench.py -- benchmark of the vcfgl simulate-and-score hot path on B200.

Metric (BASELINE.json): simulate+GL throughput in site x sample cells/s, and the fraction of the HBM roofline.
Headline workload: the scaling config (configs[4]): 10 000 diploid samples, Poisson depth 30, error 0.01, GL model 1,
tags GL+PL+AD(+DP) on synthetic msprime-shaped genotypes.  The other BASELINE configs (cfg2, cfg3(i), cfg3(ii), cfg4) run
as sub-legs of the same JSON line (`configs`), each with its kernel time, throughput and roofline fraction.

One STEP = `launches_per_step` batches of `batch_sites` sites pushed through the hot path back to back (>= 50 ms of device
work; four slots in flight so the stream never waits for the host).  Each batch writes more than the 126 MB L2 holds, so no
L2 flush is needed between launches.

  value  kernel-side throughput: genotypes resident in HBM, results left in HBM, CUDA events on the launching stream
         (torch's current stream, handed to libvgl); max over ranks.
  e2e    the same metric through the C ABI with HOST buffers: pinned H2D of the packed genotypes and D2H of the results
         inside the timed region.  Headline: VGL_HOST_BGZF -- finished BCF records, BGZF-compressed on the device (what the
         reference writes by default); `e2e.bcf_records` the same records uncompressed (VGL_HOST_BCF), `e2e.narrow_planes`
         the tag planes (GL float32; PL / AD / DP as the 8-bit values BCF stores, narrowed on the device), `e2e.i32_planes`
         the int32 planes of VGL_HOST_I32 (add_tags() layout).  gVCF workloads: the narrowed planes (the block merger
         consumes arrays).
  roofline      algorithmic bytes (SURVEY.md 8(d)) of one launch / the kernel's average launch duration (CUDA events inside
                the timed region), against the measured HBM copy bandwidth in MEASURED_PEAKS.json.
  cpu_baseline  the reference binary itself (oracle/_ref/vcfgl_ref, built from /root/reference) on a bounded sample of the
                same workload on this box's host, 1 thread.
  configs       (N=1) the other BASELINE.json configs, kernel side: value, kernel_ms, roofline {frac, traffic}.
  input_path    (N=1) SURVEY.md 8(f) row 1: one batch of msprime-shaped VCF text through k_vcf_*.
  gvcf_merge    (cfg4) SURVEY.md 8(f) row 3: the block merger on the batch resident in HBM.

`--impl reference` times the reference CPU binary with one process per host core on contiguous site shards (the reference
cannot thread its simulation; SURVEY.md 8(d)); each process runs long enough (>= 65 536 sites at 100 samples, the same
number of cells at other sample counts) that its start-up cost is below 3 % of its run.

Launch: python bench.py [--gpus N --steps K --warmup W]; for N > 1 via torch.distributed.run.  K sets the timed steps of
the kernel-side loop and of each e2e mode.  `--dump-outputs DIR` writes a fixed, seeded sample of the batches the last timed
step left in HBM as DIR/<name>.npy (dump_outputs()); the inputs depend only on the arguments, so two builds run with the same
arguments can be compared array for array.
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "sim+GL site x sample cells/s"
UNIT = "cells/s"
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "vcfgl_ref")
RTA3_BINS = [(0, 2, 2), (3, 14, 12), (15, 30, 23), (31, 63, 37)]   # test/data/rta3_qs_bins.csv, last range opened to 63

# name -> samples, sites per batch (launch), launches per >= 50 ms step, launches of a sub-leg, reference-arm sites per process,
#         vcfgl options, --qs-bins, share of invariant sites, description
WORKLOADS = {
    "cfg5": dict(S=10000, B=4440, L=32, sub=64, ref_sites=256,
                 args="-d 30 -e 0.01 -GL 1 -addGL 1 -addPL 1 -addFormatAD 1",
                 text="cfg5 shape: 10000 samples, Poisson depth 30, e=0.01, GL model 1, tags GL+PL+AD+DP, seed 42"),
    "cfg2": dict(S=100, B=131072, L=110, sub=220, ref_sites=65536,
                 args="-d 10 -e 0.01 -GL 1 -addGL 1 -addPL 1 -addFormatAD 1",
                 text="cfg2: 100 samples x 1M sites, Poisson depth 10, e=0.01, GL model 1, tags GL+PL+AD+DP, seed 42"),
    "cfg3a": dict(S=1000, B=8192, L=64, sub=128, ref_sites=6554,
                  args="-d 10 -e 0.01 -GL 2 -eq 1 -bv 1e-5 -addGL 1 -addPL 1",
                  text="cfg3(i): 1000 samples, Poisson depth 10, GL model 2, per-site beta error (mean 0.01, var 1e-5), "
                       "tags GL+PL+DP, seed 42"),
    "cfg3b": dict(S=1000, B=8192, L=48, sub=96, ref_sites=2048, bins=RTA3_BINS,
                  args="-d 10 -e 0.01 -GL 2 -eq 2 -bv 1e-5 -addGL 1 -addPL 1",
                  text="cfg3(ii): 1000 samples, Poisson depth 10, GL model 2, per-read beta error (mean 0.01, var 1e-5) + RTA3 "
                       "qs bins, tags GL+PL+DP, seed 42"),
    "cfg4": dict(S=100, B=131072, L=48, sub=96, ref_sites=65536, invariant=0.99,
                 args="-d 10 -e 0.001 -GL 1 -doUnobserved 1 -doGVCF 1 --gvcf-dps 1,5,10 -addGL 1 -addPL 1 -addI16 1 -addQS 1",
                 text="cfg4: 100 samples, 99% invariant sites (-explode), Poisson depth 10, e=0.001, GL model 1, <*> allele, gVCF, "
                      "tags GL+PL+DP+I16+QS, seed 42"),
}
N_SLOTS = 4


class Workload:
    def __init__(self, name):
        w = WORKLOADS[name]
        self.name, self.S, self.B, self.L, self.sub = name, w["S"], w["B"], w["L"], w["sub"]
        self.ref_sites = w["ref_sites"]
        self.argv = w["args"].split()
        self.bins = w.get("bins")
        self.invariant = w.get("invariant", 0.0)
        self.text = "%s (launches of %d sites)" % (w["text"], self.B)

    def sim_args(self):
        from vcfgl_b200 import args as vargs
        return vargs.parse_args(["--seed", "42"] + self.argv, qs_bins=self.bins)

    def genotypes(self, seed):
        """packed genotypes of one batch [B, S] and the haplotype matrix they came from"""
        import numpy as np
        from vcfgl_b200 import synth
        hap = synth.sfs_genotypes(self.B, self.S, seed)
        if self.invariant > 0:      # positions absent from the input VCF: hom-ref records synthesised by -explode
            hap[np.random.default_rng(7 + seed).random(self.B) < self.invariant] = 0
        return synth.pack_gt(hap), hap      # binary source: REF=0 -> A, ALT=1 -> C (vcfgl.cpp:103-128)


def measured_peak():
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(pk["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu = gpu
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- reference CPU arm
def run_reference_shards(wl, n_proc, sites_per_proc, seed, tmp):
    """P processes of the unmodified reference on P contiguous site shards; returns (cells, wall_s)"""
    import numpy as np
    from vcfgl_b200 import synth
    paths = []
    for r in range(n_proc):
        hap = synth.sfs_genotypes(sites_per_proc, wl.S, seed + r)
        if wl.invariant > 0:
            hap[np.random.default_rng(7 + seed + r).random(sites_per_proc) < wl.invariant] = 0
        pos = synth.positions(sites_per_proc, sites_per_proc * 10, seed + r)
        path = os.path.join(tmp, "shard%d.vcf" % r)
        synth.write_vcf(path, hap, pos, sites_per_proc * 10)
        paths.append(path)
    argv = list(wl.argv)
    if wl.bins:
        bins_path = os.path.join(tmp, "qs_bins.csv")
        with open(bins_path, "w") as fh:
            fh.write("".join("%d,%d,%d\n" % b for b in wl.bins))
        argv += ["--qs-bins", bins_path]
    t0 = time.perf_counter()
    procs = [subprocess.Popen([REF_BIN, "-i", path, "-o", path + ".out", "-O", "u", "--seed", "42"] + argv,
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL) for path in paths]
    rcs = [p.wait() for p in procs]
    wall = time.perf_counter() - t0
    if any(rcs):
        raise RuntimeError("reference binary failed: %s" % rcs)
    for path in paths:
        for ext in (".out.bcf", ".out.arg"):
            try:
                os.remove(path + ext)
            except OSError:
                pass
    return n_proc * sites_per_proc * wl.S, wall


def reference_arm(opt):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if not os.path.exists(REF_BIN):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/vcfgl_ref was not built (needs /root/reference at build time)"}))
        return
    wl = Workload(opt.workload)
    cores = os.cpu_count() or 1
    sites_per_proc = wl.ref_sites
    tmp = tempfile.mkdtemp(prefix="vgl_refbench_")
    try:
        for w in range(opt.warmup):
            run_reference_shards(wl, cores, max(2, sites_per_proc // 64), 1000 + w, tmp)
        cells = 0
        wall = 0.0
        for k in range(opt.steps):
            c, t = run_reference_shards(wl, cores, sites_per_proc, 2000 + 97 * k, tmp)
            cells += c
            wall += t
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    value = cells / wall
    sample = "%d steps x %d processes x %d sites x %d samples, -O u, one process per host core" % (
        opt.steps, cores, sites_per_proc, wl.S)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": opt.gpus, "steps": opt.steps,
        "warmup": opt.warmup, "ms_per_step": 1e3 * wall / opt.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl.text, "note": "reference CPU binary (vcfgl v1.3.0 da6a334), whole program: VCF parse + simulate + BCF -O u"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# --------------------------------------------------------------------------- GPU arm
def load_traffic(name):
    """DRAM bytes of one launch from the last `ncu --set full` capture of this workload (profiles/traffic.json)"""
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[name]
        return tr["dram_bytes_per_launch"], tr["source"], tr.get("cells_per_launch")
    except Exception:
        return None, None, None


class KernelLeg:
    """The hot path of one workload with genotypes resident in HBM and results left in HBM: N_SLOTS slots of one context
    on one stream, every launch on its own range of global site ids."""

    def __init__(self, wl, local, rank, stream, site0):
        from vcfgl_b200 import capi
        self.capi, self.wl, self.stream = capi, wl, stream
        self.a = wl.sim_args()
        self.gt, self.hap = wl.genotypes(20260002 + rank)
        self.ctx = capi.Context(capi.params_from_args(self.a, wl.S, max_batch_sites=wl.B, n_slots=N_SLOTS, device_id=local, host_output=False))
        self.kernels = self.ctx.native_kernels()
        self.site = site0
        for s in range(N_SLOTS):
            self.ctx.set_stream(s, stream.cuda_stream)
            self.ctx.input_buffer(s)[:] = self.gt
            self.ctx.submit(s, self.site, wl.B)          # uploads the genotypes once (untimed)
            self.ctx.sync(s)
            self.site += wl.B
        self.i = 0

    def run(self, n_launches, kern_ms=None):
        """n launches, N_SLOTS in flight; adds the per-launch device times (libvgl's CUDA events around the kernels) to kern_ms"""
        ctx, capi, B = self.ctx, self.capi, self.wl.B
        pend = []
        for _ in range(n_launches):
            s = self.i % N_SLOTS
            if len(pend) == N_SLOTS:
                d = pend.pop(0)
                ctx.sync(d)
                if kern_ms is not None:
                    kern_ms += ctx.timing(d)
            ctx.submit(s, self.site, B, flags=capi.SUBMIT_GT_ON_DEVICE)
            pend.append(s)
            self.site += B
            self.i += 1
        for d in pend:
            ctx.sync(d)
            if kern_ms is not None:
                kern_ms += ctx.timing(d)
        return d

    def roofline(self, last_slot, kern_ms_per_launch):
        """algorithmic bytes of the last launch / the kernels' average launch duration"""
        capi, ctx = self.capi, self.ctx
        b = ctx.wait(last_slot)
        ctx.copy_sites(last_slot, b)
        alg = ctx.algorithmic_bytes(b)
        fused = "+" not in self.kernels      # one kernel does the whole path; libvgl reports its time in the T_EMIT interval
        k = kern_ms_per_launch
        dev_ms = float(k[capi.T_EMIT]) if fused else float(k[capi.T_SIM] + k[capi.T_SITE] + k[capi.T_SCAN] + k[capi.T_EMIT])
        peak, peak_src = measured_peak()
        achieved = alg / (dev_ms * 1e-3) / 1e9
        traffic, traffic_src, traffic_cells = load_traffic(self.wl.name)
        cells = self.wl.B * self.wl.S
        if traffic is not None and traffic_cells and traffic_cells != cells:      # captured at another batch size: scale per cell
            traffic = int(traffic * cells / traffic_cells)
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "kernel": "%s (%s per batch; algorithmic bytes of the whole path / its average launch duration, CUDA events on the "
                          "launching stream)" % (self.kernels, "one launch" if fused else "four launches"),
                "algorithmic_bytes_per_launch": alg, "bytes_per_cell": alg / cells,
                "kernel_ms": {self.kernels: dev_ms} if fused else
                             {"k_sim": float(k[capi.T_SIM]), "k_site": float(k[capi.T_SITE]),
                              "k_scan": float(k[capi.T_SCAN]), "k_emit": float(k[capi.T_EMIT])}}
        g15 = float((b.sites["n_genotypes"] == 15).mean())
        return roof, dev_ms, alg, g15, b

    def gvcf_leg(self, slot):
        """SURVEY.md 8(f) row 3: the gVCF block merger (bcf_utils.cpp:662-942) over the batch still resident in HBM"""
        import numpy as np
        a, ctx, B, S = self.a, self.ctx, self.wl.B, self.wl.S
        if not (a.do_gvcf and a.do_unobserved in (1, 2)):
            return None
        dps = [int(x) for x in a.gvcf_dps.split(",")]
        rid0, pos0 = np.zeros(B, np.int32), np.arange(B, dtype=np.int32)
        gm = [ctx.gvcf_merge(slot, rid0, pos0, dps) for _ in range(4)]
        g_ms = min(x["ms_kernels"] for x in gm[1:])
        members = int(gm[-1]["recs"]["n_members"].sum())
        g_alg = 4 * B * S + 16 * members * S + 16 * gm[-1]["n_blocks"] * S      # DP plane in; DP + 3 PL per member cell in; per block out
        pk, pk_src = measured_peak()
        return {"what": "gVCF block merger on one batch (sites at consecutive positions of one contig)",
                "kernel_ms": g_ms, "records": int(len(gm[-1]["recs"])), "blocks": int(gm[-1]["n_blocks"]),
                "member_sites": members, "sites_per_s": B / (g_ms * 1e-3),
                "roofline": {"bound": "hbm", "achieved": g_alg / (g_ms * 1e-3) / 1e9, "peak": pk, "unit": "GB/s",
                             "frac": g_alg / (g_ms * 1e-3) / 1e9 / pk, "peak_source": pk_src, "traffic": None,
                             "algorithmic_bytes_per_launch": g_alg}}

    def close(self):
        self.ctx.close()


def sub_leg(name, local, stream):
    """one of the other BASELINE configs, kernel side (N=1): `sub` launches timed by CUDA events on the launching stream"""
    import numpy as np
    import torch
    from vcfgl_b200 import capi
    wl = Workload(name)
    leg = KernelLeg(wl, local, 0, stream, 0)
    leg.run(8)
    torch.cuda.synchronize()
    l0 = leg.ctx.launch_count()
    kern_ms = np.zeros(capi.T_COUNT)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    last = leg.run(wl.sub, kern_ms)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    launches = leg.ctx.launch_count() - l0
    roof, dev_ms, alg, g15, _ = leg.roofline(last, kern_ms / wl.sub)
    out = {"workload": wl.text, "value": wl.sub * wl.B * wl.S / (ms * 1e-3), "unit": UNIT, "launches": wl.sub, "gpu_launches": int(launches),
           "cells_per_launch": wl.B * wl.S, "ms_per_launch": ms / wl.sub, "kernel_ms": dev_ms, "kernels": leg.kernels,
           "timed_region_ms": ms, "sites_with_15_genotypes": g15, "roofline": roof}
    g = leg.gvcf_leg(last)
    if g is not None:
        out["gvcf_merge"] = g
    leg.close()
    return out


DUMP_SEED, DUMP_SITES, DUMP_SAMPLES = 20260003, 128, 256     # the sample --dump-outputs writes: <= 48 MB for any workload


def dump_outputs(leg, out_dir):
    """--dump-outputs: a fixed, seeded sample of what the timed loop computed in its last launches (the N_SLOTS batches still
    resident in HBM, oldest first), as out_dir/<name>.npy.  Per sampled site: the global site id and the vgl_site_out values a
    caller receives (`site_*`); per sampled cell (site x sample): FORMAT/DP and the tag vectors, padded with NaN to 15 genotypes /
    5 alleles (NaN throughout a skipped site).  Integers are stored as float64, GL / GP / QS / I16 as the float32 bits the
    kernels wrote."""
    import numpy as np
    import torch
    capi, ctx, B, S = leg.capi, leg.ctx, leg.wl.B, leg.wl.S
    rng = np.random.default_rng(DUMP_SEED)
    samples = np.sort(rng.choice(S, min(DUMP_SAMPLES, S), replace=False))
    fields = [f for f in capi.SITE_DTYPE.names if f not in ("_pad", "g_off", "r_off")]
    planes = (("gl", "<f4", "g", 15), ("gp", "<f4", "g", 15), ("pl", "<i4", "g", 15),
              ("ad", "<i4", "r", 5), ("adf", "<i4", "r", 5), ("adr", "<i4", "r", 5))
    out = {}

    def gather(ptr, typestr, idx):
        """plane[idx] of a device plane (torch indexes libvgl's memory through the CUDA array interface, no copy of the plane)"""
        class Plane:
            __cuda_array_interface__ = {"shape": (int(idx.max()) + 1,), "typestr": typestr, "data": (ptr, False), "version": 3}
        t = torch.as_tensor(Plane(), device="cuda")
        return t[torch.from_numpy(idx).cuda()].cpu().numpy()

    for i in range(leg.i - N_SLOTS, leg.i):
        slot, first = i % N_SLOTS, leg.site - (leg.i - i) * B
        b = ctx.wait(slot)
        recs = ctx.copy_sites(slot, b)
        sites = np.sort(rng.choice(B, min(DUMP_SITES, B), replace=False))
        part = {"site_id": (first + sites).astype(np.float64)}
        for f in fields:
            v = recs[f][sites]
            part["site_" + f] = v.astype(np.float32 if v.dtype.kind == "f" else np.float64)
        part["dp"] = gather(b.raw.dp, "<i4", (sites[:, None] * S + samples[None, :]).reshape(-1)).reshape(len(sites), -1).astype(np.float64)
        for name, typestr, kind, width in planes:
            ptr = getattr(b.raw, name)
            if not ptr:
                continue
            idx, pos = [], []
            for k, site in enumerate(sites):
                r = recs[site]
                if r["skip_code"] != 0:
                    continue
                n = int(r["n_genotypes"] if kind == "g" else r["n_alleles"])
                off = int(r["g_off"] if kind == "g" else r["r_off"])
                idx.append((off + samples[:, None] * n + np.arange(n)[None, :]).reshape(-1))
                pos.append((k * len(samples) * width + np.arange(len(samples))[:, None] * width + np.arange(n)[None, :]).reshape(-1))
            dt = np.float32 if typestr == "<f4" else np.float64
            v = np.full(len(sites) * len(samples) * width, np.nan, dt)
            if idx:
                v[np.concatenate(pos)] = gather(ptr, typestr, np.concatenate(idx))
            part[name] = v.reshape(len(sites), len(samples), width)
        for k, v in part.items():
            out.setdefault(k, []).append(v)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), np.concatenate(v))


def bind_to_gpu_numa_node(torch, local):
    """Pin this process to the CPU cores NVML lists as close to its GPU.  The pinned host buffers are first touched there, so the
    DMA of the result copies ends on the GPU's own socket instead of crossing the inter-socket link (which all ranks would share).
    Returns the number of cores bound to, or None."""
    if os.environ.get("VGL_BENCH_NUMA", "1") == "0":
        return None
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = torch.cuda.get_device_properties(local).pci_domain_id
        dev = torch.cuda.get_device_properties(local).pci_device_id
        h = pynvml.nvmlDeviceGetHandleByPciBusId(("%08x:%02x:%02x.0" % (dom, bus, dev)).encode())
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in range(64 * words) if (mask[c // 64] >> (c % 64)) & 1 and c in allowed]
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:
        return None


def gpu_arm(opt):
    import numpy as np
    import torch
    from vcfgl_b200 import capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; libvgl has no CPU path")
    torch.cuda.set_device(local)
    numa_cpus = bind_to_gpu_numa_node(torch, local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if dist is None:
            return ms
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    wl = Workload(opt.workload)
    B, S, L, K, W = wl.B, wl.S, wl.L, opt.steps, opt.warmup
    cells_per_step = B * S * L
    Le = max(2, min(L, int(opt.e2e_launches)))       # batches per e2e step
    E_SLOTS = 3
    e2e_batches_used = max(E_SLOTS, K * Le)           # every e2e mode simulates the same site range from site_next on
    # contiguous site range of this rank (weak scaling): the kernel leg's N_SLOTS + (K + W) * L batches, the e2e modes' batches
    # and spare batches (the input-path leg of a one-GPU run) -- disjoint from the other ranks' ranges
    per_rank_sites = (N_SLOTS + (K + W) * L + e2e_batches_used + 64) * B
    site0 = rank * per_rank_sites
    stream = torch.cuda.Stream()   # an explicit stream: libvgl treats a NULL stream as "use the slot's own"

    # ---------------- value: genotypes resident in HBM, results stay in HBM
    leg = KernelLeg(wl, local, rank, stream, site0)
    a, gt, hap, kernels = leg.a, leg.gt, leg.hap, leg.kernels
    leg.run(W * L)
    clocks = ClockSampler(local)
    barrier()
    if rank == 0:
        clocks.start()
    l0 = leg.ctx.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kern_ms = np.zeros(capi.T_COUNT)
    ev0.record(stream)
    last = leg.run(K * L, kern_ms)
    ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = leg.ctx.launch_count() - l0
    clk = clocks.stop() if rank == 0 else None
    roof, dev_ms, alg_bytes, g_share, _ = leg.roofline(last, kern_ms / (K * L))
    if opt.dump_outputs and rank == 0:
        dump_outputs(leg, opt.dump_outputs)
    gvcf_leg = leg.gvcf_leg(last) if rank == 0 else None
    site_next = leg.site
    leg.close()
    t_max = max_over_ranks(ms)
    value = world * K * cells_per_step / (t_max * 1e-3)

    # ---------------- e2e: host buffers, H2D + kernels + D2H inside the timed region
    if opt.skip_e2e:     # profiling runs only (ncu); such a line is not a bench result
        if rank == 0:
            print(json.dumps({"profiling_only": True, "value": value, "kernel_ms": dev_ms}))
        return
    streams = [torch.cuda.Stream() for _ in range(E_SLOTS)]

    def out_bytes(b):
        """bytes the D2H copies of one batch moved (spans as libvgl copies them)"""
        r = b.raw
        if b.bgzf is not None:      # VGL_HOST_BGZF: the compressed record stream, the record offsets, the per-site records
            return int(b.bgzf_bytes + 8 * (b.n_sites + 1) + b.n_sites * capi.SITE_DTYPE.itemsize)
        if b.bcf_off is not None or b.bcf is not None:   # VGL_HOST_BCF: the record stream, its offsets, the per-site records
            return int(b.bcf_bytes + 8 * (b.n_sites + 1) + b.n_sites * capi.SITE_DTYPE.itemsize)
        w = (b.narrow_bits // 8) if b.narrow_bits else 4          # DP / AD element width
        g_up, r_up = b.n_sites * ((S * 15 + 3) & ~3), b.n_sites * ((S * 5 + 3) & ~3)   # tile kernels: whole spans
        if "k_tile" not in kernels:
            g_up, r_up = b.g_elems, b.r_elems
        n = b.n_sites * S * w + b.n_sites * capi.SITE_DTYPE.itemsize
        n += 4 * g_up * sum(bool(x) for x in (r.gl, r.gp))
        n += g_up * (4 * bool(r.pl) + bool(r.pl_u8))
        n += w * r_up * sum(bool(x) for x in ((r.ad_n, r.adf_n, r.adr_n) if b.narrow_bits else (r.ad, r.adf, r.adr)))
        return int(n)

    def e2e_batches(ctx, bufs, n, first, bcf_in=None):
        pend, d2h = [], 0
        for i in range(n):
            s = i % E_SLOTS
            if len(pend) == E_SLOTS:
                d2h = out_bytes(ctx.wait(pend.pop(0)))
            bufs[s][:] = gt                       # the caller packs this batch's genotypes into pinned memory
            if bcf_in is not None:                # ... and the fields its input records pass through (CHROM, POS; ID ".", FILTER ".")
                sin = bcf_in[s]
                sin["pos"][:B] = np.arange(first + i * B, first + (i + 1) * B, dtype=np.int64) % (1 << 30)
                sin["qual_bits"][:B] = capi.F32_MISSING_BITS
            ctx.submit(s, first + i * B, B)
            pend.append(s)
        for s in pend:
            d2h = out_bytes(ctx.wait(s))
        return d2h

    def e2e_run(mode):
        ctx = capi.Context(capi.params_from_args(a, S, max_batch_sites=B, n_slots=E_SLOTS, device_id=local, host_output=mode,
                                                 bcf_dict=dict(DP=1, GL=2, PL=3, GP=4, AD=5, ADF=6, ADR=7, QS=8, I16=9, END=10, MIN_DP=11)))
        if a.do_gvcf and mode == capi.HOST_BCF:
            ctx.set_gvcf_dps([int(x) for x in a.gvcf_dps.split(",")])
        for s in range(E_SLOTS):
            ctx.set_stream(s, streams[s].cuda_stream)
        bufs = [ctx.input_buffer(s) for s in range(E_SLOTS)]
        bcf_in = [ctx.bcf_input(s)[0] for s in range(E_SLOTS)] if mode in (capi.HOST_BCF, capi.HOST_BGZF) else None
        e2e_batches(ctx, bufs, E_SLOTS, site_next, bcf_in)
        barrier()
        l0 = ctx.launch_count()
        t0 = time.perf_counter()
        d2h = e2e_batches(ctx, bufs, K * Le, site_next, bcf_in)
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3     # host wall clock around the user-facing calls (every wait has returned)
        barrier()
        n_launch = ctx.launch_count() - l0
        ms = max_over_ranks(ms)
        ctx.close()
        return world * K * Le * B * S / (ms * 1e-3), d2h, n_launch

    e2e_i32, d2h_i32, _ = e2e_run(capi.HOST_I32)
    e2e_nar, d2h_nar, nl_nar = e2e_run(capi.HOST_NARROW)
    e2e_narrow = {"value": e2e_nar, "d2h_bytes_per_step": d2h_nar * Le, "gpu_launches": int(nl_nar),
                  "planes": "VGL_HOST_NARROW: GL float32, PL/AD/DP narrowed on the device to the 8-bit values BCF stores"}
    e2e_value, d2h_bytes, e2e_launches = e2e_nar, d2h_nar, nl_nar
    e2e_planes = e2e_narrow["planes"]
    e2e_bcf = None
    if a.do_gvcf and a.do_unobserved in (1, 2):   # gVCF: block merger + serialisation on the device, seams stitched by vgl_wait
        v, nb, nl = e2e_run(capi.HOST_BCF)
        e2e_bcf = {"value": v, "d2h_bytes_per_step": nb * Le, "gpu_launches": int(nl),
                   "planes": "VGL_HOST_BCF with -doGVCF: regular and block records serialised on the device (k_gvcf_* + k_bcf_*), byte-identical "
                             "to the reference's -O u stream"}
        e2e_value, d2h_bytes, e2e_launches, e2e_planes = v, nb, nl, e2e_bcf["planes"]   # the headline of a gVCF workload
    if not a.do_gvcf:   # serialised BCF records
        v, nb, nl = e2e_run(capi.HOST_BCF)
        e2e_bcf = {"value": v, "d2h_bytes_per_step": nb * Le, "gpu_launches": int(nl),
                   "planes": "VGL_HOST_BCF: complete BCF records serialised on the device (k_bcf_plan/scan/emit), byte-identical to "
                             "the reference's -O u stream; the host only appends the buffer to the output"}
        # the headline: finished records as BGZF blocks (the reference's default container, -O b), compressed on the device
        e2e_value, d2h_bytes, e2e_launches = e2e_run(capi.HOST_BGZF)
        e2e_planes = ("VGL_HOST_BGZF: complete BCF records serialised and BGZF-compressed on the device (k_bcf_* + k_bgzf_*); inflating "
                      "the blocks gives the reference's -O u stream byte for byte; the host only appends the buffer to the output")

    # ---------------- the other BASELINE configs, kernel side; the input path
    configs, input_path = None, None
    if world == 1 and not opt.no_configs:
        configs = {}
        for name in ("cfg2", "cfg3a", "cfg3b", "cfg4", "cfg5"):
            if name != wl.name:
                configs[name] = sub_leg(name, local, stream)
    if world == 1 and not opt.no_input_path:
        input_path = input_path_leg(a, gt, hap, B, S, site_next + e2e_batches_used * B, local, peak_of=measured_peak)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---------------- CPU baseline: the reference binary, 1 thread, bounded sample
    cpu = None
    if world == 1 and not opt.no_cpu_baseline:
        if os.path.exists(REF_BIN):
            tmp = tempfile.mkdtemp(prefix="vgl_cpubase_")
            try:
                n_sites = wl.ref_sites * 2
                cells, wall = run_reference_shards(wl, 1, n_sites, 4242, tmp)
                cpu = {"value": cells / wall, "unit": UNIT, "cores": 1, "kind": "reference",
                       "sample": "%d sites x %d samples of the same workload, reference binary -O u, wall %.1f s" % (n_sites, S, wall)}
            finally:
                shutil.rmtree(tmp, ignore_errors=True)
        else:
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": "oracle/_ref/vcfgl_ref missing"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": t_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl.text, "batch_sites": B, "launches_per_step": L, "cells_per_step": cells_per_step,
                   "slots_in_flight": N_SLOTS,
                   "l2": "no flush: each launch writes %.2f GB of tag planes (> 126 MB L2)" % (alg_bytes / 1e9),
                   "n_samples": S, "timed_region_s": t_max * 1e-3,
                   "sites_with_15_genotypes": g_share, "sharding": "contiguous site ranges per GPU, no collective",
                   "cpus_bound_near_gpu": numa_cpus},
        "roofline": roof, "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(B * S * Le), "d2h_bytes_per_step": d2h_bytes * Le,
                "steps": K, "launches_per_step": Le, "gpu_launches": int(e2e_launches), "timer": "host wall clock, max over ranks",
                "planes": e2e_planes, "narrow_planes": e2e_narrow,
                "i32_planes": {"value": e2e_i32, "d2h_bytes_per_step": d2h_i32 * Le,
                               "planes": "VGL_HOST_I32: every plane int32/float32 as add_tags() hands them to htslib"},
                "bcf_records": e2e_bcf},
        "configs": configs, "input_path": input_path, "gvcf_merge": gvcf_leg,
        "gpu_launches": int(launches), "clocks": clk}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def input_path_leg(a, gt, hap, B, S, first_site, local, peak_of):
    """k_vcf_lines + k_vcf_gt on one step's worth of msprime-shaped VCF text (B records x S samples):
    `value`  text resident in HBM, kernels only (CUDA events on the parser's stream);
    `e2e`    host text in pinned memory -> H2D -> parse -> place -> simulate -> D2H of the narrowed planes;
    `cpu_baseline`  the oracle's single-threaded C restatement of the same parse on a bounded sample."""
    import numpy as np
    import torch
    from vcfgl_b200 import capi, synth
    pos = np.arange(1, B + 1, dtype=np.int64) * 7
    body = synth.vcf_body(hap, pos)
    n_text = len(body)
    ctx = capi.Context(capi.params_from_args(a, S, max_batch_sites=B, n_slots=2, device_id=local, host_output=capi.HOST_NARROW))
    ps = ctx.parser(n_text + 64, B)
    res = ps.parse(body, capi.SOURCE_BINARY, 0)
    assert res.n_records == B and res.n_errors == 0 and res.bytes_consumed == n_text, (res.n_records, res.n_errors)
    assert np.array_equal(ps.rows(0, 64), gt[:64]) and np.array_equal(ps.rows(B - 64, 64), gt[B - 64:])
    reps, ms = 6, []
    for _ in range(2):
        ps.parse(None, capi.SOURCE_BINARY, capi.PARSE_TEXT_ON_DEVICE, n_bytes=n_text)
    for _ in range(reps):
        ms.append(ps.parse(None, capi.SOURCE_BINARY, capi.PARSE_TEXT_ON_DEVICE, n_bytes=n_text).ms_kernels)
    k_ms = float(np.mean(ms))
    alg = n_text + B * S + B * capi.IN_SITE_DTYPE.itemsize
    peak, peak_src = peak_of()
    # end to end from text
    def step(i, slot):
        r = ps.parse(None, capi.SOURCE_BINARY, 0, n_bytes=n_text)          # H2D of the pinned text + kernels
        ctx.place_rows(slot, ps, B)
        ctx.submit(slot, first_site + i * B, B, flags=capi.SUBMIT_GT_ON_DEVICE)
        return r
    for i in range(2):
        step(i, i & 1)
    ctx.wait(0), ctx.wait(1)
    torch.cuda.synchronize()
    n_e2e = 4
    import time as _t
    t0 = _t.perf_counter()
    pend = []
    for i in range(n_e2e):
        slot = i & 1
        if len(pend) == 2:
            ctx.wait(pend.pop(0))
        step(i, slot)
        pend.append(slot)
    for slot in pend:
        ctx.wait(slot)
    torch.cuda.synchronize()
    wall = _t.perf_counter() - t0
    ps.close()
    ctx.close()
    # VCF text in -> finished BCF records out: input path + simulation + device BCF serialisation (VGL_HOST_BCF); the host only
    # copies POS from the parser's site records into the pass-through records and would append the returned bytes to the file
    def text_to_records(mode, n_slots, n_batches):
        ctx = capi.Context(capi.params_from_args(a, S, max_batch_sites=B, n_slots=n_slots, device_id=local, host_output=mode,
                                                 bcf_dict=dict(DP=1, GL=2, PL=3, GP=4, AD=5, ADF=6, ADR=7, QS=8, I16=9)))
        ps = ctx.parser(n_text + 64, B)
        ps.parse(body, capi.SOURCE_BINARY, 0)
        bcf_in = [ctx.bcf_input(k)[0] for k in range(n_slots)]

        def step_rec(i, slot):
            r = ps.parse(None, capi.SOURCE_BINARY, 0, n_bytes=n_text)
            sin = bcf_in[slot]
            sin["pos"][:B] = r.sites["pos"]
            sin["qual_bits"][:B] = capi.F32_MISSING_BITS
            ctx.place_rows(slot, ps, B)
            ctx.submit(slot, first_site + i * B, B, flags=capi.SUBMIT_GT_ON_DEVICE)

        def size_of(b):
            return b.bgzf_bytes if mode == capi.HOST_BGZF else b.bcf_bytes
        for i in range(n_slots):
            step_rec(i, i)
        for k in range(n_slots):
            ctx.wait(k)
        torch.cuda.synchronize()
        t0 = _t.perf_counter()
        pend, nbytes = [], 0
        for i in range(n_batches):
            slot = i % n_slots
            if len(pend) == n_slots:
                nbytes = size_of(ctx.wait(pend.pop(0)))
            step_rec(i, slot)
            pend.append(slot)
        for slot in pend:
            nbytes = size_of(ctx.wait(slot))
        torch.cuda.synchronize()
        wall_rec = _t.perf_counter() - t0
        ps.close()
        ctx.close()
        return n_batches * B * S / wall_rec, int(nbytes)

    text_to_bcf = text_to_bgzf = None
    if not a.do_gvcf:
        v, nbytes = text_to_records(capi.HOST_BCF, 2, n_e2e)
        text_to_bcf = {"value": v, "unit": UNIT, "h2d_bytes_per_step": n_text, "d2h_bytes_per_step": nbytes, "steps": n_e2e,
                       "note": "VCF text in pinned host memory -> BCF records in pinned host memory: k_vcf_* + k_place_rows + simulation + k_bcf_*; host wall clock"}
        v, nbytes = text_to_records(capi.HOST_BGZF, 3, 4 * n_e2e)
        text_to_bgzf = {"value": v, "unit": UNIT, "h2d_bytes_per_step": n_text, "d2h_bytes_per_step": nbytes, "steps": 4 * n_e2e,
                        "note": "the same with the records BGZF-compressed on the device (k_bgzf_*): what the reference program does from its input file "
                                "to its default (-O b) output file, minus reading and writing the files; three slots; host wall clock"}
    # CPU baseline: oracle restatement, one thread, bounded sample
    cpu = None
    try:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import vcfin_oracle as vo
        n_cpu = min(B, 32768)
        cut = 0
        for _ in range(n_cpu):
            cut = body.index(b"\n", cut) + 1
        t0 = _t.perf_counter()
        sites, rows, used = vo.parse(body[:cut], S, 0)
        dt = _t.perf_counter() - t0
        assert len(sites) == n_cpu and np.array_equal(rows, gt[:n_cpu])
        cpu = {"value": n_cpu * S / dt, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": "oracle/vcf_in_oracle.c on the first %d records (%.1f MB of text), %.3f s" % (n_cpu, cut / 1e6, dt)}
    except Exception as e:      # the oracle is test infrastructure; its absence must not break the bench line
        cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "unavailable: %s" % e}
    traffic, traffic_src = None, None
    try:    # DRAM bytes of the path's kernels from their ncu --set full captures (profiles/traffic.json), when this shape was profiled
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["input_path_%dx%d" % (B, S)]
        traffic, traffic_src = tr["dram_bytes_per_step"], tr["source"]
    except Exception:
        pass
    return {"what": "VCF text -> packed genotypes on the device (k_vcf_count, k_vcf_index, k_vcf_hdr, k_vcf_cells, k_vcf_gt), %d records x %d samples, %.1f MB of text per step" % (B, S, n_text / 1e6),
            "value": B * S / (k_ms * 1e-3), "unit": UNIT, "kernel_ms": k_ms, "gpu_launches_per_step": 5,
            "roofline": {"bound": "hbm", "achieved": alg / (k_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg / (k_ms * 1e-3) / 1e9 / peak, "peak_source": peak_src, "traffic": traffic, "traffic_source": traffic_src,
                         "algorithmic_bytes_per_step": alg, "bytes_per_cell": alg / (B * S)},
            "e2e": {"value": n_e2e * B * S / wall, "unit": UNIT, "h2d_bytes_per_step": n_text, "steps": n_e2e,
                    "note": "pinned host text -> H2D -> k_vcf_* -> k_place_rows -> simulate -> D2H (VGL_HOST_NARROW); host wall clock, two slots"},
            "text_to_bcf": text_to_bcf, "text_to_bgzf": text_to_bgzf, "cpu_baseline": cpu}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-input-path", action="store_true", help="skip the VCF-text input-path leg")
    ap.add_argument("--no-configs", action="store_true", help="skip the sub-legs of the other BASELINE configs")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling only: stop after the kernel-side loop")
    ap.add_argument("--e2e-launches", type=int, default=12, help="batches per end-to-end step (the timed region starts and ends with an empty pipeline)")
    ap.add_argument("--workload", default="cfg5", choices=sorted(WORKLOADS))
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a fixed seeded sample of what the last "
                                                          "launches computed as DIR/<name>.npy (rank 0; --impl b200 only)")
    opt = ap.parse_args()
    if opt.steps < 1:
        ap.error("--steps must be at least 1")
    if opt.dump_outputs and opt.impl != "b200":
        ap.error("--dump-outputs writes what the GPU path computed; it does not apply to --impl reference")
    opt.warmup = max(opt.warmup, 3) if opt.impl == "b200" else opt.warmup
    if opt.impl == "reference":
        reference_arm(opt)
    else:
        gpu_arm(opt)


if __name__ == "__main__":
    main()
