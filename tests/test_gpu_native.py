"""Native-RNG (Philox) simulator on the GPU.

(1) self-replay: the kernel's own draws (vgl_native_draws), fed to the CPU oracle and back through
    the replay path, must reproduce the native run's tags bit-exactly -- this checks the whole native
    pipeline at sizes where no reference capture exists, and that results do not depend on batch size.
(2) statistical parity with the reference (tests/golden/stats.json, made by
    tools/make_stats_golden.py from the instrumented reference, >= 1e6 cells per fixture): two-sample
    chi-square on the per-cell depth histogram (per group of samples with --depths-file), the true-base ->
    read-base matrix, the haplotype pick, the strand split, the tail distances and the side of a site's tail
    mass, the per-read qs histogram and the mis-called reads per site (--error-qs 1); two-sample
    Kolmogorov-Smirnov on depth, quality score and tail distance; two-proportion z-test on genotype-call
    discordance; alpha = 0.001 each.  Every fixture runs on each native kernel set that takes its flags.
"""
import json
import os

import numpy as np
import pytest
from scipy import stats

import golden_cases as gc
import oracle_lib
from vcfgl_b200 import args as vargs
from vcfgl_b200 import capi, synth

pytestmark = pytest.mark.gpu
ALPHA = 1e-3
STATS = json.load(open(os.path.join(gc.GOLD, "stats.json")))
PAIRS = [(a1, a2) for a2 in range(5) for a1 in range(a2 + 1)]


def u32(x):
    return np.ascontiguousarray(x).view(np.uint32)


SELF_CASES = {
    "gl1_fixed_alltags": "--seed 5 -d 6 -e 0.02 -GL 1 -doUnobserved 1 -addGP 1 -addPL 1 -addI16 1 -addQS 1 -addInfoDP 1 "
                         "-addFormatAD 1 -addInfoAD 1 -addFormatADF 1 -addInfoADF 1 -addFormatADR 1 -addInfoADR 1",
    "gl2_fixed": "--seed 6 -d 4 -e 0.05 -GL 2 -doUnobserved 4 -addPL 1 -addFormatAD 1 -addQS 1",
    "gl2_eq2_lut": "--seed 7 -d 4 -e 0.01 -eq 2 -bv 1e-5 -GL 2 --adjust-qs 3 -addPL 1 -addQS 1 -addI16 1 -addFormatAD 1",
    "gl1_eq2": "--seed 8 -d 5 -e 0.02 -eq 2 -bv 1e-4 -GL 1 -addPL 1 -addFormatAD 1",
    "gl2_eq1": "--seed 9 -d 3 -e 0.05 -eq 1 -bv 1e-3 -GL 2 -addPL 1 -addFormatAD 1",
    "gl1_deep": "--seed 10 -d 280 -e 0.01 -GL 1 -addPL 1 -addFormatAD 1",
    "gl2_precise": "--seed 11 -d 4 -e 0.01 -eq 2 -bv 1e-5 -GL 2 --precise-gl 1 -addPL 1",
}


@pytest.mark.parametrize("name", sorted(SELF_CASES))
def test_native_tags_match_oracle_on_own_draws(name):
    S, n_sites = (6, 40) if "deep" in name else (37, 300)
    self_replay(name, SELF_CASES[name], 1, S, n_sites)


def self_replay(name, argv, sampler, S, n_sites, kernels=None, qs_bins=None, depths=None):
    a = vargs.parse_args(argv.split(), qs_bins=qs_bins, depths=depths)
    hap = synth.sfs_genotypes(n_sites, S, 99, missing_rate=0.05) if S > 1 else \
        np.random.default_rng(1).integers(0, 2, (n_sites, 2)).astype(np.int8)
    gt = synth.pack_gt(hap)
    ctx = capi.Context(capi.params_from_args(a, S, max_batch_sites=n_sites, n_slots=1, sampler=sampler))
    if kernels:
        assert ctx.native_kernels() == kernels, ctx.native_kernels()
    ctx.input_buffer(0)[:n_sites] = gt
    first = 123456789012
    ctx.submit(0, first, n_sites)
    b = ctx.wait(0)
    native = [b.site(i) for i in range(n_sites)]
    native = [{k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in d.items()} for d in native]
    rp = ctx.native_draws(0, first, n_sites)
    assert np.array_equal(rp["depths"], b.dp)
    # (a) oracle on the kernel's draws (the oracle needs the kept-read capture for depth > 255; covered by (b) + golden d300 cases)
    if "deep" not in name:
        assert oracle_lib.check_sites_on_draws(a, S, hap, native, rp, gl_rtol=1e-6 if name == "gl2_precise" else 0.0) > 0
    # (b) replay of the kernel's draws through the C ABI, in two batches with different slots sizes
    if "deep" not in name:
        ctx.submit(0, 7, n_sites, replay=rp)
        b2 = ctx.wait(0)
        for i in range(n_sites):
            d, e = native[i], b2.site(i)
            assert d["skip_code"] == e["skip_code"]
            if d["skip_code"] == 0:
                assert np.array_equal(u32(d["gl"]), u32(e["gl"])), (name, i)
    # (c) batch-size independence: the same sites in two half batches give identical tags
    h = n_sites // 2
    ctx.input_buffer(0)[:n_sites - h] = gt[h:]
    ctx.submit(0, first + h, n_sites - h)
    b3 = ctx.wait(0)
    for i in range(h, n_sites):
        d, e = native[i], b3.site(i - h)
        assert d["skip_code"] == e["skip_code"]
        if d["skip_code"] == 0:
            assert np.array_equal(u32(d["gl"]), u32(e["gl"])), (name, i)
            assert np.array_equal(d["fmt_dp"], e["fmt_dp"])
    ctx.close()


def chi2_two_sample(a, b, min_expected=5):
    a, b = np.asarray(a, float).ravel(), np.asarray(b, float).ravel()
    keep = (a + b) > 0
    a, b = a[keep], b[keep]
    # pool sparse categories
    order = np.argsort(a + b)
    a, b = a[order], b[order]
    tot = a.sum() + b.sum()
    while len(a) > 2 and min((a[0] + b[0]) * a.sum() / tot, (a[0] + b[0]) * b.sum() / tot) < min_expected:
        a = np.concatenate([[a[0] + a[1]], a[2:]])
        b = np.concatenate([[b[0] + b[1]], b[2:]])
        order = np.argsort(a + b)
        a, b = a[order], b[order]
    return stats.chi2_contingency(np.stack([a, b]))[1]


def ks_two_sample(h1, h2):
    """two-sample Kolmogorov-Smirnov test from two histograms over the same ordered support (asymptotic p-value; for a
    discrete law the test is conservative)"""
    h1, h2 = np.asarray(h1, float).ravel(), np.asarray(h2, float).ravel()
    n1, n2 = h1.sum(), h2.sum()
    d = np.abs(np.cumsum(h1) / n1 - np.cumsum(h2) / n2).max()
    return float(stats.kstwobign.sf(d * np.sqrt(n1 * n2 / (n1 + n2))))


# every fixture runs on each native kernel set that takes its flags; the kernel set is asserted, so that a dispatch change
# in vgl_create cannot silently move a test to another kernel.  (fixture, sampler, kernels, drop the strand flags?)
PER_READ = "k_sim+k_site+k_scan+k_emit"
DIST_RUNS = [
    ("gl1_d10", 1, PER_READ, False),
    ("gl1_d10", 0, "k_tile_m1f", True),            # without FORMAT/ADF the headline kernel takes it
    ("gl1_d30", 1, PER_READ, False),
    ("gl1_d30", 0, "k_tile_m1f", False),
    ("gl1_aux", 1, PER_READ, False),
    ("gl1_aux", 0, "k_tile_m1f", False),           # the AUX variant (QS / I16 / INFO ADF, ADR)
    ("gl1_df", 1, PER_READ, False),                # --depths-file: per-sample Poisson means (k_fused_m1f: tests/test_gpu_fused.py)
    ("gl1_df", 0, "k_tile_m1f", False),            # one alias table per distinct mean
    ("gl2_d2_e02", 1, PER_READ, False),
    ("gl2_d2_e02", 0, "k_tile_m2", True),
    ("gl2_eq2", 1, PER_READ, False),
    ("gl2_eq2", 0, "k_tile_m2", False),
    ("gl2_eq2_bins", 1, PER_READ, False),
    ("gl2_eq2_bins", 0, "k_tile_m2", False),
    ("gl2_eq1", 1, PER_READ, False),
    ("gl2_eq1", 0, "k_tile_m2", False),
]


@pytest.mark.parametrize("name,sampler,kernels,drop_strand", DIST_RUNS, ids=["%s-%s" % (r[0], r[2].split("+")[0]) for r in DIST_RUNS])
def test_native_distributions_match_reference(name, sampler, kernels, drop_strand):
    distributions(name, sampler, kernels=kernels, strand=not drop_strand)


def test_fixed_depth_has_the_reference_read_laws():
    """VGL_DEPTH_FIXED (north_star: "Poisson/fixed"; the reference CLI has no such option): every cell has exactly the
    depth, the read-level laws (mis-calls, haplotype pick) are those of the reference's gl1_d10 capture"""
    distributions("gl1_d10", 0, kernels="k_tile_m1f", strand=False, fixed_depth=True)


def distributions(name, sampler, kernels=None, strand=True, fixed_depth=False, batch=2000):
    st = STATS[name]
    argv = list(st["argv"])
    if not strand:   # kernels without strand tags: drop the ADF/ADR flags of the fixture's command line
        for flag in ("-addFormatADF", "-addFormatADR"):
            while flag in argv:
                i = argv.index(flag)
                del argv[i:i + 2]
    a = vargs.parse_args(argv, qs_bins=st.get("qs_bins"), depths=st.get("depths"))
    S, n_sites = st["S"], st["n_sites"]
    hap_all = synth.sfs_genotypes(n_sites, S, st["gt_seed"])
    batch = min(batch * 100 // S, n_sites)
    ctx = capi.Context(capi.params_from_args(a, S, max_batch_sites=batch, n_slots=1, sampler=sampler, fixed_depth=fixed_depth))
    if kernels:
        assert ctx.native_kernels() == kernels, (ctx.native_kernels(), kernels)
    depth_hist = np.zeros(200, np.int64)
    depth_by_sample = np.zeros((S, 64), np.int64)
    conf = np.zeros((4, 4), np.int64)
    het_reads = np.zeros(2, np.int64)
    strand_n = np.zeros(2, np.int64)
    qs_hist = np.zeros(256, np.int64)
    tail_hist = np.zeros(32, np.int64)
    tail_side = np.zeros(2, np.int64)
    site_err_hist = np.zeros(64, np.int64)
    disc = {"hom": [0, 0], "het": [0, 0]}
    for lo in range(0, n_sites, batch):
        nb = min(batch, n_sites - lo)
        hap = hap_all[lo:lo + nb]
        ctx.input_buffer(0)[:nb] = synth.pack_gt(hap)
        ctx.submit(0, lo, nb)
        b = ctx.wait(0)
        dpl = b.dp[:nb * S].reshape(nb, S)
        depth_hist += np.bincount(np.minimum(dpl.ravel(), 199), minlength=200)
        np.add.at(depth_by_sample, (np.tile(np.arange(S), nb), np.minimum(dpl.ravel(), 63)), 1)
        dd = ctx.discordance(0)     # on-device summary (tests/test_gpu_discordance.py pins it to the definition)
        for k in ("hom", "het"):
            disc[k][0] += dd[k][0]
            disc[k][1] += dd[k][1]
        sites = b.sites[:nb]
        if a.add_i16:
            keep = (sites["skip_code"] == 0) & (sites["info_dp"] > 0)
            tail_side += [int((sites["i16"][keep][:, 12] > 0).sum()), int((sites["i16"][keep][:, 14] > 0).sum())]
        rp = ctx.native_draws(0, lo, nb)
        assert np.array_equal(rp["depths"], dpl.ravel())
        cell_of_read = np.repeat(np.arange(nb * S), np.diff(rp["read_offsets"]))
        g0 = hap.reshape(-1, 2)[cell_of_read, 0]
        g1 = hap.reshape(-1, 2)[cell_of_read, 1]
        hom = g0 == g1
        np.add.at(conf, (g0[hom], rp["bases"][hom]), 1)
        err_site = np.bincount(cell_of_read[hom] // S, weights=(rp["bases"][hom] != g0[hom]), minlength=nb).astype(np.int64)
        site_err_hist += np.bincount(np.minimum(err_site, 63), minlength=64)
        het = ~hom
        het_reads += [(rp["bases"][het] == g0[het]).sum(), (rp["bases"][het] == g1[het]).sum()]
        if strand:
            strand_n += np.bincount(rp["strands"], minlength=2)[:2]
        if a.error_qs == 2:
            qs_hist += np.bincount(rp["qs"], minlength=256)
        if a.add_i16:
            tail_hist += np.bincount(np.minimum(rp["tail_dists"], 31), minlength=32)
    ctx.close()
    pvals = {}
    if fixed_depth:
        assert depth_hist[int(a.depth)] == depth_hist.sum(), "fixed depth: every cell must hold exactly --depth reads"
    else:
        pvals["depth"] = chi2_two_sample(depth_hist, st["depth_hist"])
        pvals["depth_ks"] = ks_two_sample(depth_hist, st["depth_hist"])
        if st.get("depths") is None:
            pvals["depth_vs_poisson"] = chi2_two_sample(depth_hist, stats.poisson.pmf(np.arange(200), a.depth) * depth_hist.sum() * 1e3)
        else:   # per-sample means: each group of samples that share a mean against the reference's same group
            ref_by = np.array(st["depth_by_sample"])
            means = np.array(st["depths"])
            for m in sorted(set(means)):
                pvals["depth_mean_%g" % m] = chi2_two_sample(depth_by_sample[means == m].sum(axis=0), ref_by[means == m].sum(axis=0))
                pvals["depth_ks_mean_%g" % m] = ks_two_sample(depth_by_sample[means == m].sum(axis=0), ref_by[means == m].sum(axis=0))
    ref_conf = np.array(st["confusion"])
    for t in range(4):
        if ref_conf[t].sum() > 0:
            pvals["confusion_true%d" % t] = chi2_two_sample(conf[t], ref_conf[t])
    pvals["het_hap_pick"] = chi2_two_sample(het_reads, st["het_reads"])
    if a.error_qs == 1 and not fixed_depth:   # the per-site beta draw shows as over-dispersion of the mis-called reads per site
        pvals["site_errors"] = chi2_two_sample(site_err_hist, st["site_err_hist"])
    if strand and sum(st["strand"][1:]) > 0 and strand_n.sum() > 0:
        pvals["strand"] = chi2_two_sample(strand_n, st["strand"])
    if a.error_qs == 2:
        pvals["qs"] = chi2_two_sample(qs_hist, st["qs_hist"])
        pvals["qs_ks"] = ks_two_sample(qs_hist, st["qs_hist"])
    if a.add_i16:
        pvals["tail"] = chi2_two_sample(tail_hist, st["tail_hist"])
        pvals["tail_ks"] = ks_two_sample(tail_hist, st["tail_hist"])
        pvals["tail_side"] = chi2_two_sample(tail_side, st["tail_side"])   # the stale r_base of vcfgl.cpp:657
    if not fixed_depth:
        for k in ("hom", "het"):   # genotype-call discordance (argmax GL vs truth), misc/gtDiscordance.cpp strata
            n1, x1 = disc[k]
            n2, x2 = st["discordance"][k]
            pp = (x1 + x2) / (n1 + n2)
            if 0 < pp < 1:
                z = (x1 / n1 - x2 / n2) / np.sqrt(pp * (1 - pp) * (1 / n1 + 1 / n2))
                pvals["discordance_" + k] = 2 * stats.norm.sf(abs(z))
    bad = {k: v for k, v in pvals.items() if not (v >= ALPHA)}
    assert not bad, (name, kernels, bad, pvals)
