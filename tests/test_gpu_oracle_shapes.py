"""The tile kernels against the CPU oracle where they could go wrong unnoticed: the extra-plane pass of k_tile_m1f, the
tile-geometry edges, many tiles per CTA, and the shapes bench.py times.

Every comparison is oracle_lib.check_sites_on_draws: the plain-C oracle run on the batch's own draws (vgl_native_draws)
must give every field of the site record and every plane the arguments ask for, GP within check_gp's rounding bound.

(a) XTRA: the AUX variant of k_tile_m1f writes GP and FORMAT ADF / ADR in a second pass per chunk.  Each tag mix runs at
    S = 1, 3, 37, 2501 and 4096 (counts in global memory, an S4 / 32 chunk-mask row without a spare entry), over
    -doUnobserved 0 / 1 / 3 / 5 and three depth / error regimes: low depth (depth-0 cells), -d 30 -e 0.01 (GL < -38:
    subnormal GP) and -e 0.25 (a high error rate the kernel still takes).  Missing genotypes throughout.
(b) Geometry: T = min(32, 2048 // S4) sites per tile.  S at the steps of T (64 / 65, 512 / 513, 680 / 681), at the largest
    site held in shared memory (2045, 2048), the smallest and a 32-aligned counts row in global memory (2049, 4096, 4097) and
    the largest S the tile kernels take (60000, where the 32-bit slot arithmetic is at its limit).  2T + 1 sites, so the
    last tile is partial, then a one-site batch.
(c) Many tiles per CTA: the tile kernels run persistent CTAs (at most 8 per SM) that take tiles from a ticket; a batch of
    >= 3 x SMs x 8 tiles makes every CTA carry its shared state (site totals, AUX accumulators, chunk tickets, per-CTA
    scratch rows) from one tile into the next.  A seeded sample of sites plus the last 64 (the late tiles are the CTAs'
    second or later ones).
(d) The benched shapes: one full batch of each bench.WORKLOADS entry, in the kernel leg's context (bench.N_SLOTS slots,
    results left on the device); the first and last tile and a seeded sample, read on the device.  A sampled site's draws
    come from another slot (vgl_native_draws writes its slot's FORMAT/DP plane), with the site's genotypes in row 0.

Each case asserts its kernel set.  The share of GP values bit-equal to the oracle's is printed per case (pytest -s).
"""
import functools

import numpy as np
import pytest
import torch

import bench
import oracle_lib
from device_util import device_gather
from test_gpu_native import self_replay
from vcfgl_b200 import args as vargs
from vcfgl_b200 import capi, synth

pytestmark = pytest.mark.gpu

M1, M2 = "k_tile_m1f", "k_tile_m2"
RTA3 = [(0, 2, 2), (3, 14, 12), (15, 30, 23), (31, 63, 37)]
TILE_CELLS, TILE_MAX_SITES, CTAS_PER_SM = 2048, 32, 8      # tile_common.cuh


def sites_per_tile(S):
    return max(1, min(TILE_MAX_SITES, TILE_CELLS // ((S + 3) & ~3)))


# ---------------------------------------------------------------- (a) the XTRA variant of k_tile_m1f
XTRA_TAGS = {
    "gp": "-addGP 1 -addPL 1 -addFormatAD 1",
    "adf": "-addPL 1 -addFormatADF 1",
    "adr": "-addPL 1 -addFormatADR 1",
    "adf_adr": "-addPL 1 -addFormatAD 1 -addFormatADF 1 -addFormatADR 1",
    "gp_without_gl": "-addGL 0 -addGP 1 -addPL 1",          # GL is staged for GP only (stage_gl)
    "gp_without_pl": "-addGP 1 -addFormatAD 1",              # the GEN subset
    "all_qs_i16": "-addGP 1 -addPL 1 -addFormatAD 1 -addFormatADF 1 -addFormatADR 1 -addQS 1 -addI16 1 -addInfoDP 1 "
                  "-addInfoAD 1 -addInfoADF 1 -addInfoADR 1",
}
XTRA_S = {1: 400, 3: 300, 37: 100, 2501: 5, 4096: 4}       # S: sites
# -e 0.25: about the largest error rate k_tile_m1f takes (its scores need the fast division; -e 0.3 goes to k_fused_m1f)
REGIMES = {"low": "-d 3 -e 0.02", "subnormal": "-d 30 -e 0.01", "e025": "-d 4 -e 0.25"}
UNOBS = (0, 1, 3, 5)


def xtra_cases():
    """every tag mix at every S; -doUnobserved and the regime rotate over them; all_qs_i16 also at S = 37 in every
    (-doUnobserved, regime) pair"""
    out = {}
    for vi, tags in enumerate(sorted(XTRA_TAGS)):
        for si, S in enumerate(sorted(XTRA_S)):
            k = vi + si
            u, reg = UNOBS[k % len(UNOBS)], sorted(REGIMES)[k % len(REGIMES)]
            out["%s-S%d-u%d-%s" % (tags, S, u, reg)] = (tags, S, u, reg)
    for u in UNOBS:
        for reg in sorted(REGIMES):
            out.setdefault("all_qs_i16-S37-u%d-%s" % (u, reg), ("all_qs_i16", 37, u, reg))
    return out


XTRA_CASES = xtra_cases()


def xtra_argv(name):
    tags, S, u, reg = XTRA_CASES[name]
    return "--seed %d -GL 1 %s -doUnobserved %d %s" % (101 + sorted(XTRA_CASES).index(name), REGIMES[reg], u, XTRA_TAGS[tags])


@pytest.mark.parametrize("name", sorted(XTRA_CASES))
def test_xtra_planes_match_oracle(name):
    tags, S, u, reg = XTRA_CASES[name]
    share = [0, 0]
    self_replay(name, xtra_argv(name), 0, S, XTRA_S[S], kernels=M1, gp_share=share)
    if "-addGP 1" in XTRA_TAGS[tags]:
        assert share[1] > 0


# ---------------------------------------------------------------- shared by (b), (c): a tile-kernel family per argv
FAMILIES = {
    # name: (argv after the seed and depth, kernel set, --qs-bins)
    "m1_plain": ("-GL 1 -e 0.02 -addGL 1 -addPL 1 -addFormatAD 1", M1, None),
    "m1_gen": ("-GL 1 -e 0.02 -addGL 0 -addPL 1", M1, None),
    "m1_aux": ("-GL 1 -e 0.02 -doUnobserved 1 -addPL 1 -addI16 1 -addQS 1 -addInfoADF 1 -addInfoADR 1", M1, None),
    "m1_xtra": ("-GL 1 -e 0.02 -addPL 1 -addGP 1 -addFormatADF 1 -addFormatADR 1", M1, None),
    "m2_eq0": ("-GL 2 -e 0.01 -addGL 1 -addPL 1 -addFormatAD 1", M2, None),
    "m2_lut_bins": ("-GL 2 -e 0.01 -eq 2 -bv 1e-5 -addGL 1 -addPL 1", M2, RTA3),
}
FAM = sorted(FAMILIES)


def family_args(fam, seed, depth):
    argv, kernels, bins = FAMILIES[fam]
    return vargs.parse_args(("--seed %d -d %g %s" % (seed, depth, argv)).split(), qs_bins=bins), kernels


def own_draws_check(a, S, kernels, batches, label, pick=None):
    """each (first_site_id, haplotypes) batch through one VGL_HOST_I32 slot, then the oracle on the slot's own draws at the
    sites pick(n_sites) (default: all)"""
    B = max(len(h) for _, h in batches)
    ctx = capi.Context(capi.params_from_args(a, S, max_batch_sites=B, n_slots=1))
    assert ctx.native_kernels() == kernels, (ctx.native_kernels(), kernels)
    orc = oracle_lib.Oracle(a, S)
    share = [0, 0]
    for first, hap in batches:
        n = len(hap)
        ctx.input_buffer(0)[:n] = synth.pack_gt(hap)
        ctx.submit(0, first, n)
        b = ctx.wait(0)
        assert b.status == 0
        idx = list(range(n)) if pick is None else pick(n)
        native = {i: {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in b.site(i).items()} for i in idx}
        dp = b.dp[:n * S].copy()
        rp = ctx.native_draws(0, first, n)
        assert np.array_equal(rp["depths"], dp)
        assert oracle_lib.check_sites_on_draws(a, S, hap, native, rp, idx=idx, orc=orc, gp_share=share) > 0, (label, first)
    ctx.close()
    if a.add_gp:
        assert share[1] > 0
        print("%s: GP bit-equal to the oracle: %d of %d (%s)" % (label, share[0], share[1], kernels))


# ---------------------------------------------------------------- (b) geometry sweep
GEOM_S = [4, 63, 64, 65, 511, 512, 513, 680, 681, 2045, 2048, 2049, 4096, 4097, 60000]


def geometry_cases():
    """every family at each S >= 2045; below, three families per S in rotation (each family at five S)"""
    out = []
    for k, S in enumerate(GEOM_S):
        fams = FAM if S >= 2045 else [FAM[(k + j) % len(FAM)] for j in (0, 2, 4)]
        out += [(fam, S) for fam in fams]
    return out


GEOM_CASES = geometry_cases()


@pytest.mark.parametrize("fam,S", GEOM_CASES, ids=["%s-S%d" % c for c in GEOM_CASES])
def test_tile_geometry_edges_match_oracle(fam, S):
    a, kernels = family_args(fam, 300 + GEOM_CASES.index((fam, S)), 2)
    T = sites_per_tile(S)
    n = 2 * T + 1
    hap = synth.sfs_genotypes(n, S, 17 + S, missing_rate=0.05)
    one = synth.sfs_genotypes(1, S, 18 + S, missing_rate=0.05)
    own_draws_check(a, S, kernels, [(7 * S, hap), (10 ** 9 + S, one)], "%s-S%d" % (fam, S))


# ---------------------------------------------------------------- (c) many tiles per CTA
@functools.lru_cache(maxsize=None)
def many_tiles():
    return 3 * torch.cuda.get_device_properties(0).multi_processor_count * CTAS_PER_SM


def sample_and_tail(seed, n_sample=512, n_tail=64):
    def pick(n):
        rng = np.random.default_rng(seed)
        s = set(rng.choice(n, min(n_sample, n), replace=False).tolist()) | set(range(max(0, n - n_tail), n))
        return sorted(s)
    return pick


MANY_CASES = [(fam, S) for fam in FAM for S in (37, 2049)]


@pytest.mark.parametrize("fam,S", MANY_CASES, ids=["%s-S%d" % c for c in MANY_CASES])
def test_many_tiles_per_cta_match_oracle(fam, S):
    a, kernels = family_args(fam, 500 + MANY_CASES.index((fam, S)), 2)
    n = many_tiles() * sites_per_tile(S)
    hap = synth.sfs_genotypes(n, S, 23 + S, missing_rate=0.05)
    own_draws_check(a, S, kernels, [(31 * S, hap)], "%s-S%d-many" % (fam, S), pick=sample_and_tail(S))


# ---------------------------------------------------------------- (d) the benched shapes
BENCH_KERNELS = {"cfg5": M1, "cfg2": M1, "cfg3a": M2, "cfg3b": M2, "cfg4": M1}


def site_from_device(b, recs, i, S):
    """Batch.site(i) of a VGL_HOST_NONE batch, its blocks gathered on the device"""
    s = recs[i]
    A, G = int(s["n_alleles"]), int(s["n_genotypes"])
    raw = b.raw
    d = dict(skip_code=int(s["skip_code"]), n_alleles=A, n_alleles_observed=int(s["n_alleles_observed"]), n_genotypes=G,
             alleles2acgt=s["alleles2acgt"][:5].astype(np.int32), acgt2alleles=s["acgt2alleles"][:5].astype(np.int32),
             info_dp=int(s["info_dp"]), info_ad=s["info_ad"][:A].copy(), info_adf=s["info_adf"][:A].copy(),
             info_adr=s["info_adr"][:A].copy(), qs=s["qs"][:A].copy(), i16=s["i16"].copy(),
             fmt_dp=device_gather(raw.dp, "<i4", np.arange(i * S, (i + 1) * S)))
    if d["skip_code"] == 0:
        g = int(s["g_off"]) + np.arange(S * G)
        r = int(s["r_off"]) + np.arange(S * A)
        for k, t in (("gl", "<f4"), ("gp", "<f4"), ("pl", "<i4")):
            d[k] = device_gather(getattr(raw, k), t, g)
        for k, p in (("fmt_ad", "ad"), ("fmt_adf", "adf"), ("fmt_adr", "adr")):
            d[k] = device_gather(getattr(raw, p), "<i4", r)
    return d


@pytest.mark.parametrize("name", sorted(bench.WORKLOADS))
def test_benched_shape_matches_oracle(name):
    wl = bench.Workload(name)
    a, S, B = wl.sim_args(), wl.S, wl.B
    gt, hap = wl.genotypes(20260002)
    ctx = capi.Context(capi.params_from_args(a, S, max_batch_sites=B, n_slots=bench.N_SLOTS, host_output=False))
    assert ctx.native_kernels() == BENCH_KERNELS[name], ctx.native_kernels()
    first = 7 * B + 11
    ctx.input_buffer(0)[:B] = gt
    ctx.submit(0, first, B)
    b = ctx.wait(0)
    assert b.status == 0
    recs = ctx.copy_sites(0, b)
    T = sites_per_tile(S)
    rng = np.random.default_rng(20260004)
    n_sample = 48 if name == "cfg5" else 256
    edge = set(range(T)) | set(range((B - 1) // T * T, B))      # every site of the first and the last tile
    idx = sorted(edge | set(rng.choice(B, n_sample, replace=False).tolist()))
    orc = oracle_lib.Oracle(a, S)
    share, n_cmp = [0, 0], 0
    for i in idx:
        d = site_from_device(b, recs, i, S)
        ctx.input_buffer(1)[0] = gt[i]
        rp = ctx.native_draws(1, first + i, 1)
        assert np.array_equal(rp["depths"], d["fmt_dp"]), i
        n_cmp += oracle_lib.check_sites_on_draws(a, S, hap[i:i + 1], [d], rp, orc=orc, gp_share=share)
    assert n_cmp > 0
    if a.add_gp:
        print("%s: GP bit-equal to the oracle: %d of %d (%s)" % (name, share[0], share[1], BENCH_KERNELS[name]))
    ctx.close()
