"""The fused single-kernel path (native RNG, GL model 1 / fixed qs, count-level sampler).

(1) every emitted tag is re-derived by the CPU oracle from the kernel's own per-cell counts
    (AD/ADF/DP are outputs; for fixed-qs model 1 all tags are functions of the counts) -> bit-exact;
(2) layout: compact, in site order, deterministic, independent of batch boundaries;
(3) the count-level sampler has the reference's distributions (same fixtures and tests as the
    per-read sampler): depth, true-base -> read-base matrix, haplotype split, strand, discordance.
"""
import numpy as np
import pytest

import oracle_lib
from test_gpu_native import ALPHA, PAIRS, STATS, chi2_two_sample, ks_two_sample, u32
from scipy import stats
from vcfgl_b200 import args as vargs
from vcfgl_b200 import capi, synth

pytestmark = pytest.mark.gpu

CASES = {
    "cfg2": ("--seed 42 -d 10 -e 0.01 -GL 1 -addGL 1 -addPL 1 -addFormatAD 1", 100, 700),
    "alltags_star": ("--seed 5 -d 6 -e 0.02 -GL 1 -doUnobserved 1 -addGP 1 -addPL 1 -addInfoDP 1 -addFormatAD 1 -addInfoAD 1 "
                     "-addFormatADF 1 -addInfoADF 1 -addFormatADR 1 -addInfoADR 1", 37, 400),
    # GP and the strand planes on k_fused_m1f itself: with --error-qs 0 the count-level sampler's GP runs go to k_tile_m1f
    "alltags_eq1": ("--seed 16 -d 6 -e 0.02 -eq 1 -bv 1e-3 -GL 1 -doUnobserved 0 -addGP 1 -addPL 1 -addFormatAD 1 -addFormatADF 1 "
                    "-addFormatADR 1", 37, 400),
    "trim_rminvar": ("--seed 6 -d 2 -e 0.1 -GL 1 -doUnobserved 0 --rm-invar-sites 4 --rm-empty-sites 1 -addPL 1 -addFormatAD 1", 5, 900),
    "explode5_nonref": ("--seed 7 -d 3 -e 0.3 -GL 1 -doUnobserved 5 -addPL 1 -addFormatAD 1 -addFormatADF 1", 3, 700),
    "explode3_lowdepth": ("--seed 8 -d 0.3 -e 0.05 -GL 1 -doUnobserved 3 -addPL 1 -addFormatAD 1", 2, 1500),
    "eq1": ("--seed 9 -d 5 -e 0.05 -eq 1 -bv 1e-3 -GL 1 -addPL 1 -addFormatAD 1 --adjust-qs 1", 64, 300),
    "s1": ("--seed 10 -d 4 -e 0.05 -GL 1 -addPL 1 -addFormatAD 1", 1, 3000),
    "s1300": ("--seed 11 -d 8 -e 0.01 -GL 1 -addPL 1 -addFormatAD 1", 1300, 40),
    "s2501_scratch": ("--seed 14 -d 3 -e 0.02 -GL 1 -addGL 1 -addPL 1 -addFormatAD 1", 2501, 12),
    "e_high": ("--seed 12 -d 12 -e 0.9 -GL 1 -addPL 1 -addFormatAD 1", 33, 300),
    "deep": ("--seed 13 -d 280 -e 0.01 -GL 1 -addPL 1 -addFormatAD 1", 6, 60),
    # every third site has no reads and is dropped; its neighbours show all four bases (+ <*>: all 15 base pairs have a slot), so
    # 32-cell chunks mix lanes of skipped sites with lanes of the unpredicated store path
    "skipped_next_to_all15": ("--seed 15 -d 6 -e 0.6 -GL 1 -doUnobserved 1 --rm-empty-sites 1 -addPL 1 -addFormatAD 1", 6, 900),
}


def run(a, S, gt, first, n, sampler=2, cap=None):
    ctx = capi.Context(capi.params_from_args(a, S, max_batch_sites=cap or n, n_slots=1, sampler=sampler))
    ctx.input_buffer(0)[:n] = gt
    ctx.submit(0, first, n)
    b = ctx.wait(0)
    assert b.status == 0
    sites = [{k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in b.site(i).items()} for i in range(n)]
    offs = b.sites["g_off"].copy(), b.sites["r_off"].copy(), b.g_elems, b.r_elems
    run.kernels = ctx.native_kernels()
    ctx.close()
    return sites, offs


@pytest.mark.parametrize("name", sorted(CASES))
def test_fused_tags_match_oracle_on_own_counts(name):
    argv, S, n_sites = CASES[name]
    a = vargs.parse_args(argv.split())
    hap = synth.sfs_genotypes(n_sites, S, 4242, missing_rate=0.04) if S > 1 else \
        np.random.default_rng(1).integers(0, 2, (n_sites, 2)).astype(np.int8)
    if name.startswith("skipped"):
        hap[::3] = -1
    gt = synth.pack_gt(hap)
    first = 987654321
    sites, (g_off, r_off, g_elems, r_elems) = run(a, S, gt, first, n_sites)
    orc = oracle_lib.Oracle(a, S)
    # (2) layout: blocks in site order, 16-byte aligned, disjoint, inside the used extent.  (The tile kernel packs
    # blocks densely within a tile of sites and starts every tile at a fixed stride; the general kernels pack all.)
    pos_g = pos_r = 0
    for i, d in enumerate(sites):
        assert g_off[i] >= pos_g and r_off[i] >= pos_r, (name, i)
        assert g_off[i] % 4 == 0 and r_off[i] % 4 == 0, (name, i)
        pos_g, pos_r = g_off[i], r_off[i]
        if d["skip_code"] == 0:
            pos_g += (S * d["n_genotypes"] + 3) // 4 * 4
            pos_r += (S * d["n_alleles"] + 3) // 4 * 4
    assert pos_g <= g_elems and pos_r <= r_elems
    assert g_elems <= n_sites * ((S * 15 + 3) // 4 * 4) and r_elems <= n_sites * ((S * 5 + 3) // 4 * 4)
    # (1) oracle on the kernel's own counts
    n_cmp = 0
    gp_share = [0, 0]
    for i, d in enumerate(sites):
        dp = d["fmt_dp"]
        miss = (hap[i, 0::2] < 0) | (hap[i, 1::2] < 0)
        assert (dp[miss] == 0).all()
        if d["skip_code"] != 0:
            assert d["skip_code"] in (-3, -4)
            continue
        A = d["n_alleles"]
        ad = d["fmt_ad"].reshape(S, A)
        adf = d["fmt_adf"].reshape(S, A) if d.get("fmt_adf") is not None else None
        a2b = d["alleles2acgt"]
        assert (ad.sum(axis=1) == dp).all(), (name, i)
        bases, strands = [], []
        for s in range(S):
            for al in range(A):
                if 0 <= a2b[al] < 4:
                    k = int(ad[s, al])
                    f = int(adf[s, al]) if adf is not None else k
                    bases += [a2b[al]] * k
                    strands += [0] * f + [1] * (k - f)
        if (dp > 255).any():
            continue   # depth > 255: the kept subset is random; AD/DP consistency checked above
        o = orc.site(hap[i], dp, np.array(bases, np.uint8), np.array(strands, np.uint8))
        assert o["ret"] == 0 and o["n_alleles"] == A and o["n_genotypes"] == d["n_genotypes"], (name, i)
        if d["info_dp"] > 0:
            assert np.array_equal(o["alleles2acgt"], a2b), (name, i)
        assert np.array_equal(u32(o["gl"]), u32(d["gl"])), (name, i, o["gl"], d["gl"])
        assert np.array_equal(o["pl"], d["pl"]), (name, i)
        for key in ("fmt_ad", "fmt_adf", "fmt_adr", "info_ad", "info_adf", "info_adr"):
            if getattr(a, "add_" + key) and d.get(key) is not None:
                assert np.array_equal(o[key], d[key]), (name, i, key)
        if a.add_gp:
            assert d.get("gp") is not None, (name, i)
            eq, n = oracle_lib.check_gp(d["gp"], o["gl"], o["gp"], dp, d["n_genotypes"])
            gp_share[0] += eq
            gp_share[1] += n
        n_cmp += 1
    assert n_cmp > 0 or name == "deep"
    if a.add_gp:
        print("%s: GP bit-equal to the oracle: %d of %d (%s)" % (name, gp_share[0], gp_share[1], run.kernels))
    # (2) determinism + batch independence: same sites, other batch boundaries and capacity
    h = n_sites // 3
    again, _ = run(a, S, gt[h:], first + h, n_sites - h, cap=n_sites + 11)
    for i in range(h, n_sites):
        d, e = sites[i], again[i - h]
        assert d["skip_code"] == e["skip_code"]
        assert np.array_equal(d["fmt_dp"], e["fmt_dp"])
        if d["skip_code"] == 0:
            assert np.array_equal(u32(d["gl"]), u32(e["gl"])) and np.array_equal(d["fmt_ad"], e["fmt_ad"])


@pytest.mark.parametrize("name,no_tile,kernels", [("gl1_d10", True, "k_fused_m1f"), ("gl1_d10", False, "k_tile_m1f"), ("gl1_d30", True, "k_fused_m1f"),
                                                  ("gl1_d30", False, "k_tile_m1f"), ("gl1_df", True, "k_fused_m1f"),
                                                  ("gl1_df", False, "k_tile_m1f")])
def test_count_sampler_distributions_match_reference(name, no_tile, kernels, monkeypatch):
    """the count-level sampler against the reference's captures (>= 1e6 cells each), from the AD / ADF planes alone (the
    fused kernel has no per-read draws to export); the kernel set is asserted"""
    st = STATS[name]
    a = vargs.parse_args(st["argv"], depths=st.get("depths"))
    S, n_sites = st["S"], st["n_sites"]
    if no_tile:
        monkeypatch.setenv("VGL_NO_TILE", "1")
    hap_all = synth.sfs_genotypes(n_sites, S, st["gt_seed"])
    batch = 2000
    ctx = capi.Context(capi.params_from_args(a, S, max_batch_sites=batch, n_slots=1, sampler=2))
    assert ctx.native_kernels() == kernels, ctx.native_kernels()
    depth_hist = np.zeros(200, np.int64)
    depth_by_sample = np.zeros((S, 64), np.int64)
    conf = np.zeros((4, 4), np.int64)
    het_reads = np.zeros(2, np.int64)
    strand = np.zeros(2, np.int64)
    disc = {"hom": [0, 0], "het": [0, 0]}
    for lo in range(0, n_sites, batch):
        nb = min(batch, n_sites - lo)
        hap = hap_all[lo:lo + nb]
        ctx.input_buffer(0)[:nb] = synth.pack_gt(hap)
        ctx.submit(0, lo, nb)
        b = ctx.wait(0)
        assert b.status == 0
        depth_hist += np.bincount(np.minimum(b.dp[:nb * S], 199), minlength=200)
        np.add.at(depth_by_sample, (np.tile(np.arange(S), nb), np.minimum(b.dp[:nb * S], 63)), 1)
        dd = ctx.discordance(0)
        for k in ("hom", "het"):
            disc[k][0] += dd[k][0]
            disc[k][1] += dd[k][1]
        for i in range(nb):
            d = b.site(i)
            if d["skip_code"] != 0 or d["info_dp"] == 0:
                continue
            A = d["n_alleles"]
            a2b = d["alleles2acgt"]
            ad = d["fmt_ad"].reshape(S, A)
            acgt = np.zeros((S, 4), np.int64)
            for al in range(A):
                if 0 <= a2b[al] < 4:
                    acgt[:, a2b[al]] = ad[:, al]
            g0, g1 = hap[i, 0::2], hap[i, 1::2]
            hom = g0 == g1
            for t in range(4):
                conf[t] += acgt[hom & (g0 == t)].sum(axis=0)
            het = ~hom
            het_reads[0] += acgt[het, g0[het]].sum()
            het_reads[1] += acgt[het, g1[het]].sum()
            if d.get("fmt_adf") is not None:
                f = int(d["fmt_adf"].sum())
                strand += [f, int(ad.sum()) - f]
    ctx.close()
    pvals = {}
    pvals["depth"] = chi2_two_sample(depth_hist, st["depth_hist"])
    pvals["depth_ks"] = ks_two_sample(depth_hist, st["depth_hist"])
    if st.get("depths") is None:
        pvals["depth_vs_poisson"] = chi2_two_sample(depth_hist, stats.poisson.pmf(np.arange(200), a.depth) * depth_hist.sum() * 1e3)
    else:   # --depths-file: each group of samples that share a mean against the reference's same group
        ref_by, means = np.array(st["depth_by_sample"]), np.array(st["depths"])
        for m in sorted(set(means)):
            pvals["depth_mean_%g" % m] = chi2_two_sample(depth_by_sample[means == m].sum(axis=0), ref_by[means == m].sum(axis=0))
            pvals["depth_ks_mean_%g" % m] = ks_two_sample(depth_by_sample[means == m].sum(axis=0), ref_by[means == m].sum(axis=0))
    ref_conf = np.array(st["confusion"])
    for t in range(4):
        if ref_conf[t].sum() > 0:
            pvals["confusion_true%d" % t] = chi2_two_sample(conf[t], ref_conf[t])
    pvals["het_hap_pick"] = chi2_two_sample(het_reads, st["het_reads"])
    if strand.sum() > 0 and sum(st["strand"][1:]) > 0:
        pvals["strand"] = chi2_two_sample(strand, st["strand"])
    for k in ("hom", "het"):
        n1, x1 = disc[k]
        n2, x2 = st["discordance"][k]
        pp = (x1 + x2) / (n1 + n2)
        if 0 < pp < 1:
            z = (x1 / n1 - x2 / n2) / np.sqrt(pp * (1 - pp) * (1 / n1 + 1 / n2))
            pvals["discordance_" + k] = 2 * stats.norm.sf(abs(z))
    bad = {k: v for k, v in pvals.items() if not (v >= ALPHA)}
    assert not bad, (name, kernels, bad, pvals)
