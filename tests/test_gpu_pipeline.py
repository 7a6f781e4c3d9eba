"""Batches in flight: a context with K slots, up to K batches submitted before the first wait and waited in submission order
(the schedule bench.py and host/vgl_host.hpp run), against the same batches through one VGL_HOST_I32 slot, submit then wait.
Bit for bit: every named vgl_site_out field, the used plane extents, every plane (float planes as their uint32 bits, which
also covers the NaN payloads of missing values).

The batches are small (a few tiles of the tile kernels) and many, so that most CTAs of a launch exit early and the next
batch's kernels could start while the first CTAs still hold their per-CTA scratch rows.  The list holds full batches, B - 1,
one site, a batch of missing genotypes only, and first_site_id values with gaps.

Each kernel set runs in VGL_HOST_NONE (planes gathered on the device through __cuda_array_interface__, as bench.py's
--dump-outputs does, plus vgl_copy_sites and vgl_discordance), VGL_HOST_I32 and VGL_HOST_NARROW at K = 2 and 8, and once with
every slot on one torch stream (bench.py).  One batch of each K = 8 VGL_HOST_NONE run is also checked against the CPU oracle
on that slot's own draws, so that the reference run is not the only anchor.

Record modes: VGL_HOST_BCF / VGL_HOST_BGZF streams of three slots in flight against the one-slot record stream, the
benched shape (10 000 samples), a batch whose pass-through bytes make more BGZF blocks than its share of sites predicts, and
-doGVCF waits out of submission order."""
import functools
import math
from collections import deque

import numpy as np
import pytest
import torch

import oracle_lib
from bcf_util import bo
import truth_util as tu
from test_gpu_bgzf import inflate_all, split_blocks
from vcfgl_b200 import args as vargs
from vcfgl_b200 import capi, synth

pytestmark = pytest.mark.gpu

PER_READ = "k_sim+k_site+k_scan+k_emit"
TRUTH = "k_truth_site+k_scan+k_truth_emit"
CFG2 = "--seed 42 -d 10 -e 0.01 -GL 1 -addGL 1 -addPL 1 -addFormatAD 1"
RTA3 = [(0, 2, 2), (3, 14, 12), (15, 30, 23), (31, 63, 37)]
CASES = {
    # name: (argv, S, B, kernel set, qs_bins)
    "tile_m1f": (CFG2, 37, 150, "k_tile_m1f", None),
    "tile_m1f_pure": ("--seed 3 -d 1 -e 0.01 -GL 1 -addPL 1 -addFormatAD 1", 37, 150, "k_tile_m1f", None),      # 32 d e < 0.5
    "tile_m1f_aux": ("--seed 5 -d 6 -e 0.02 -GL 1 -addI16 1 -addQS 1 -doUnobserved 1 -addPL 1 -addFormatAD 1", 37, 150, "k_tile_m1f", None),
    "tile_m1f_big": (CFG2, 2501, 3, "k_tile_m1f", None),                                                          # S > 2048
    "tile_m2_eq0": ("--seed 4 -d 6 -e 0.01 -GL 2 -addGL 1 -addPL 1 -addFormatAD 1", 37, 150, "k_tile_m2", None),
    "tile_m2_eq1": ("--seed 9 -d 3 -e 0.05 -eq 1 -bv 1e-3 -GL 2 -addPL 1 -addFormatAD 1", 37, 150, "k_tile_m2", None),
    "tile_m2_eq2": ("--seed 7 -d 4 -e 0.01 -eq 2 -bv 1e-5 -GL 2 -addPL 1 -addFormatAD 1", 37, 150, "k_tile_m2", None),
    "tile_m2_eq2_bins": ("--seed 4 -d 10 -e 0.01 -GL 2 -eq 2 -bv 1e-5 -addGL 1 -addPL 1", 37, 150, "k_tile_m2", RTA3),
    "tile_m2_big": ("--seed 14 -d 3 -e 0.02 -GL 2 -addGL 1 -addPL 1 -addFormatAD 1", 2501, 3, "k_tile_m2", None),
    "fused_m1f": ("--seed 9 -d 5 -e 0.05 -eq 1 -bv 1e-3 -GL 1 -addPL 1 -addFormatAD 1", 37, 150, "k_fused_m1f", None),
    "per_read": ("--seed 8 -d 5 -e 0.02 -eq 2 -bv 1e-4 -GL 1 -addPL 1 -addFormatAD 1", 37, 150, PER_READ, None),
    "truth": ("--seed 1 --depth inf -e 0 -GL 1 -addGL 1 -addPL 1 -addFormatDP 0", 37, 150, TRUTH, None),
}
PLANES = ("dp", "gl", "gp", "pl", "ad", "adf", "adr")
SITE_FIELDS = [f for f in capi.SITE_DTYPE.names if f != "_pad"]


def batch_list(S, B, seed, truth=False, reps=4):
    """[(first_site_id, packed genotypes [n, S], haplotypes int8 [n, 2S])]: >= 32 batches of the shapes listed above"""
    sizes = [B, B - 1, 1, B, B, 2, B, B // 2 + 1]
    out, first = [], 17
    for r in range(reps):
        for j, n in enumerate(sizes):
            n = max(n, 1)
            hap = synth.sfs_genotypes(n, S, seed + 8 * r + j, missing_rate=0.0 if truth else 0.05)
            if j == 4 and not truth:           # a truth run refuses a missing genotype (VGL_EMISSING)
                hap[:] = -1
            out.append((first, synth.pack_gt(hap), hap))
            first += n + (0 if j % 3 else 1000003 * (r + 1))      # gaps between the site ids of some batches
    return out


def device_plane(ptr, typestr, n):
    """a copy of n elements of a device plane, taken through its CUDA array interface"""
    if not ptr:
        return None
    dt = np.dtype(typestr)
    if n == 0:
        return np.zeros(0, dt)

    class Plane:
        __cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (ptr, False), "version": 3}
    return torch.as_tensor(Plane(), device="cuda").clone().cpu().numpy()


def collect(ctx, slot, mode, disc):
    """the waited slot's results, copied out of pinned / device memory before the slot is submitted again"""
    b = ctx.wait(slot)
    assert b.status == 0
    n, S = b.n_sites, b.S
    r = dict(g=b.g_elems, r=b.r_elems)
    if mode == capi.HOST_NONE:
        r["sites"] = ctx.copy_sites(slot, b).copy()
        raw = b.raw
        r["dp"] = device_plane(raw.dp, "<i4", n * S)
        for k, t in (("gl", "<f4"), ("gp", "<f4"), ("pl", "<i4")):
            r[k] = device_plane(getattr(raw, k), t, b.g_elems)
        for k in ("ad", "adf", "adr"):
            r[k] = device_plane(getattr(raw, k), "<i4", b.r_elems)
    else:
        r["sites"] = b.sites.copy()
        for k in PLANES:
            v = getattr(b, k)
            r[k] = None if v is None else v.copy()
        if mode == capi.HOST_NARROW:
            r["pl"] = None if b.pl_u8 is None else b.pl_u8.copy()
    if not ctx.params.tag_mask & vargs.TAG_FMT_DP:   # the plane exists but holds no tag (--depth inf writes no depths)
        r["dp"] = None
    if disc:
        r["disc"] = ctx.discordance(slot)
    return r


def run(a, S, B, batches, mode, K, kernels, one_stream=False, disc=False, anchor=False):
    ctx = capi.Context(capi.params_from_args(a, S, max_batch_sites=B, n_slots=K, host_output=mode))
    assert ctx.native_kernels() == kernels
    if one_stream:
        stream = torch.cuda.Stream()
        for k in range(K):
            ctx.set_stream(k, stream.cuda_stream)
    res = [None] * len(batches)
    pending = deque()
    for i, (first, gt, _) in enumerate(batches):
        if len(pending) == K:
            j = pending.popleft()
            res[j] = collect(ctx, j % K, mode, disc)
        ctx.input_buffer(i % K)[:len(gt)] = gt
        ctx.submit(i % K, first, len(gt))
        pending.append(i)
    while pending:
        j = pending.popleft()
        res[j] = collect(ctx, j % K, mode, disc)
    if anchor:      # the last batch's slot still holds its genotypes
        check_anchor(ctx, a, S, (len(batches) - 1) % K, batches[-1], res[-1], kernels)
    ctx.close()
    return res


def site_dicts(r, S):
    """Batch.site() of every site of a collected result"""
    out = []
    for i, s in enumerate(r["sites"]):
        A, G = int(s["n_alleles"]), int(s["n_genotypes"])
        d = dict(skip_code=int(s["skip_code"]), n_alleles=A, n_genotypes=G, alleles2acgt=s["alleles2acgt"][:5].astype(np.int32),
                 info_ad=s["info_ad"][:A], info_adf=s["info_adf"][:A], info_adr=s["info_adr"][:A], qs=s["qs"][:A], i16=s["i16"],
                 fmt_dp=None if r["dp"] is None else r["dp"][i * S:(i + 1) * S])
        if d["skip_code"] == 0:
            g0, r0 = int(s["g_off"]), int(s["r_off"])
            for k in ("gl", "pl", "gp"):
                d[k] = None if r[k] is None else r[k][g0:g0 + S * G]
            for k, p in (("fmt_ad", "ad"), ("fmt_adf", "adf"), ("fmt_adr", "adr")):
                d[k] = None if r[p] is None else r[p][r0:r0 + S * A]
        out.append(d)
    return out


def check_anchor(ctx, a, S, slot, batch, r, kernels):
    """one batch against the CPU oracle: on the slot's own draws (vgl_native_draws), on the kernel's own counts where the
    sampler draws no reads one by one (k_fused_m1f), on the true genotypes under --depth inf"""
    first, gt, hap = batch
    sites = site_dicts(r, S)
    if kernels == TRUTH:
        for i, d in enumerate(sites):
            w = tu.to.site(hap[i], a.do_unobserved)
            assert d["n_genotypes"] == w["n_genotypes"] and d["alleles2acgt"].tolist() == w["alleles2acgt"], i
            assert np.array_equal(d["gl"].view(np.uint32), w["gl"].view(np.uint32)) and np.array_equal(d["pl"], w["pl"]), i
        return
    if kernels == "k_fused_m1f":    # every tag is a function of the counts: the oracle on reads rebuilt from AD
        orc = oracle_lib.Oracle(a, S)
        n_cmp = 0
        for i, d in enumerate(sites):
            if d["skip_code"] != 0:
                continue
            ad = d["fmt_ad"].reshape(S, d["n_alleles"])
            bases = [int(d["alleles2acgt"][al]) for s in range(S) for al in range(d["n_alleles"]) if 0 <= d["alleles2acgt"][al] < 4
                     for _ in range(int(ad[s, al]))]
            o = orc.site(hap[i], d["fmt_dp"], np.array(bases, np.uint8))
            assert np.array_equal(o["pl"], d["pl"]) and np.array_equal(o["fmt_ad"], d["fmt_ad"]), i
            assert np.array_equal(o["gl"].view(np.uint32), bits(d["gl"])), i
            n_cmp += 1
        assert n_cmp > 0
        return
    rp = ctx.native_draws(slot, first, len(gt))
    assert np.array_equal(rp["depths"], r["dp"])
    assert oracle_lib.check_sites_on_draws(a, S, hap, sites, rp) > 0


def bits(x):
    return None if x is None else np.ascontiguousarray(x).view(np.uint32)


def site_blocks(w, S):
    """element masks of the sites' blocks in the genotype and allele planes (VGL_HOST_NONE leaves the tile kernels' holes
    between them as they were: only VGL_HOST_I32 / VGL_HOST_NARROW copy whole spans, so only there are the holes zeroed)"""
    mg, mr = np.zeros(w["g"], bool), np.zeros(w["r"], bool)
    for s in w["sites"]:
        if s["skip_code"] == 0:
            mg[s["g_off"]:s["g_off"] + S * s["n_genotypes"]] = True
            mr[s["r_off"]:s["r_off"] + S * s["n_alleles"]] = True
    return mg, mr


def assert_same(got, want, mode, S):
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert (g["g"], g["r"]) == (w["g"], w["r"]), i
        mg, mr = site_blocks(w, S)
        for f in SITE_FIELDS:
            x, y = g["sites"][f], w["sites"][f]
            if x.dtype.kind == "f":
                x, y = bits(x), bits(y)
            assert np.array_equal(x, y), (i, f)
        for k in PLANES:
            x, y = g[k], w[k]
            assert (x is None) == (y is None), (i, k)
            if x is None:
                continue
            if mode == capi.HOST_NARROW and k == "pl":    # 8-bit PL: the int32 values where FORMAT/DP > 0 (missing elsewhere)
                have = y[:w["g"]] != capi.I32_MISSING
                assert np.array_equal(x[:w["g"]][have].astype(np.int32), y[:w["g"]][have]), (i, k)
                continue
            n = len(y) if k == "dp" else (w["g"] if k in ("gl", "gp", "pl") else w["r"])
            x, y = bits(x[:n].astype(y.dtype)), bits(y[:n])
            if mode == capi.HOST_NONE and k != "dp":
                x, y = x[mg if k in ("gl", "gp", "pl") else mr], y[mg if k in ("gl", "gp", "pl") else mr]
            assert np.array_equal(x, y), (i, k)
        if "disc" in g:
            assert g["disc"]["hom"] == w["disc"]["hom"] and g["disc"]["het"] == w["disc"]["het"], i


@functools.lru_cache(maxsize=None)
def case_inputs(name):
    argv, S, B, kernels, bins = CASES[name]
    a = vargs.parse_args(argv.split(), qs_bins=bins)
    batches = batch_list(S, B, 1000 + sorted(CASES).index(name), truth=kernels == TRUTH)
    disc = bool(a.add_gl and a.add_fmt_dp)
    return a, S, B, kernels, batches, disc, run(a, S, B, batches, capi.HOST_I32, 1, kernels, disc=disc)


RUNS = [(n, m, k) for n in sorted(CASES) for m in ("none", "i32", "narrow") for k in (2, 8) if not (n == "truth" and m == "narrow")]
MODES = dict(none=capi.HOST_NONE, i32=capi.HOST_I32, narrow=capi.HOST_NARROW)


@pytest.mark.parametrize("name,mode,K", RUNS, ids=["%s-%s-%s-K%d" % (CASES[n][3].split("+")[0], n, m, k) for n, m, k in RUNS])
def test_batches_in_flight_equal_one_slot(name, mode, K):
    a, S, B, kernels, batches, disc, want = case_inputs(name)
    m = MODES[mode]
    got = run(a, S, B, batches, m, K, kernels, disc=disc and m == capi.HOST_NONE, anchor=m == capi.HOST_NONE and K == 8)
    assert_same(got, want, m, S)


@pytest.mark.parametrize("name", sorted(CASES), ids=["%s-%s" % (CASES[n][3].split("+")[0], n) for n in sorted(CASES)])
def test_slots_on_one_torch_stream_equal_one_slot(name):
    a, S, B, kernels, batches, disc, want = case_inputs(name)
    got = run(a, S, B, batches, capi.HOST_NONE, 4, kernels, one_stream=True, disc=disc)
    assert_same(got, want, capi.HOST_NONE, S)


# ---------------------------------------------------------------- record modes
IDS = dict(DP=1, GL=2, PL=3, GP=4, AD=5, ADF=6, ADR=7, QS=8, I16=9)


def fill_bcf_input(ctx, slot, first, m, info=None):
    sin, blob = ctx.bcf_input(slot)
    sin[:m] = 0
    sin["pos"][:m] = (np.arange(first, first + m) * 3 + 1) % (1 << 30)
    sin["qual_bits"][:m] = capi.F32_MISSING_BITS
    o = 0
    for k, pt in (info or {}).items():    # FILTER + INFO bytes of the input record (one INFO field each)
        sin[k]["flt_info_off"], sin[k]["flt_info_len"], sin[k]["n_info"] = o, len(pt), 1
        blob[o:o + len(pt)] = np.frombuffer(pt, np.uint8)
        o += len(pt)


def record_run(a, S, B, batches, mode, K, blob_per_site=16, infos=None):
    """-> per batch: the record stream (HOST_BCF) or its BGZF blocks inflated (HOST_BGZF), and the BGZF block count"""
    ctx = capi.Context(capi.params_from_args(a, S, max_batch_sites=B, n_slots=K, host_output=mode, bcf_dict=IDS,
                                             bcf_blob_bytes_per_site=blob_per_site))
    res = [None] * len(batches)
    pending = deque()

    def take(j):
        b = ctx.wait(j % K)
        assert b.status == 0
        if mode == capi.HOST_BGZF:
            raw, _ = inflate_all(bytes(b.bgzf))       # CRC and ISIZE of every block checked
            assert len(split_blocks(bytes(b.bgzf))) == b.bgzf_blocks
            assert len(raw) == b.bcf_bytes
            res[j] = (raw, b.bgzf_blocks)
        else:
            res[j] = (bytes(b.bcf), 0)
    for i, (first, gt) in enumerate(batches):
        if len(pending) == K:
            take(pending.popleft())
        ctx.input_buffer(i % K)[:len(gt)] = gt
        fill_bcf_input(ctx, i % K, first, len(gt), (infos or {}).get(i))
        ctx.submit(i % K, first, len(gt))
        pending.append(i)
    while pending:
        take(pending.popleft())
    ctx.close()
    return res


@pytest.mark.parametrize("mode", ["bcf", "bgzf"])
@pytest.mark.parametrize("shape", ["irregular", "bench"])
def test_record_streams_in_flight_equal_one_slot(mode, shape):
    if shape == "irregular":
        S, B, sizes = 37, 64, [64, 7, 1, 63, 33, 64, 2, 64, 17, 64, 40, 5, 64, 64, 1, 30]
        argv = "--seed 6 -d 6 -e 0.02 -GL 1 -doUnobserved 1 -addGL 1 -addPL 1 -addFormatAD 1 -addInfoDP 1"
    else:     # bench.py's record legs: 10 000 samples x 64 sites in batches of 16
        S, B, sizes, argv = 10000, 16, [16] * 4, CFG2
    a = vargs.parse_args(argv.split())
    batches, first = [], 5
    for j, n in enumerate(sizes):
        hap = synth.sfs_genotypes(n, S, 77 + j, missing_rate=0.03)
        batches.append((first, synth.pack_gt(hap)))
        first += n + (1000 if j % 4 == 3 else 0)
    want = record_run(a, S, B, batches, capi.HOST_BCF, 1)
    got = record_run(a, S, B, batches, capi.HOST_BCF if mode == "bcf" else capi.HOST_BGZF, 3)
    assert b"".join(g for g, _ in got) == b"".join(w for w, _ in want)
    assert sum(len(w) for w, _ in want) > 0


def test_bgzf_batch_that_carries_most_of_the_blob():
    """a 2-site batch whose INFO pass-through fills most of the context's 1 MiB blob makes far more BGZF blocks than its share
    of sites predicts: every block must still be compressed from ranges made for it"""
    S, B, per_site = 4, 4096, 256
    a = vargs.parse_args(CFG2.split())
    first_batch = synth.pack_gt(synth.sfs_genotypes(2000, S, 5, missing_rate=0.0))      # builds the context's Huffman code
    second = synth.pack_gt(synth.sfs_genotypes(2, S, 6, missing_rate=0.0))
    vals = np.random.default_rng(3).random(125000).astype(np.float32)
    pt = b"\x00" + bo.enc_int1(11) + bo.enc_vfloat(vals)                  # empty FILTER, INFO key 11: 125 000 floats
    assert 2 * len(pt) <= B * per_site
    batches = [(0, first_batch), (5000, second)]
    infos = {1: {0: pt, 1: pt}}
    # blocks the launch of k_bgzf_ranges covered before it looped over the real count (capi.cu: nb_max from the site share)
    t = a.tag_mask
    wc = 2        # depth law bounded by 255 reads: 16-bit depths
    per_cell = (wc if t & vargs.TAG_FMT_DP else 0) + (60 if t & vargs.TAG_GL else 0) + (60 if t & vargs.TAG_GP else 0) + \
        (30 if t & vargs.TAG_PL else 0) + 5 * wc * sum(bool(t & x) for x in (vargs.TAG_FMT_AD, vargs.TAG_FMT_ADF, vargs.TAG_FMT_ADR))
    bcf_cap = (B * S * per_cell + B * (512 + per_site) + 15) & ~15
    nb_max = min(math.ceil(bcf_cap / 32768), math.ceil((int(bcf_cap * 2 / B) + 65536) / 32768))
    old_cover = 8 * math.ceil(nb_max / 8)
    want = record_run(a, S, B, [(f, g) for f, g in batches], capi.HOST_BCF, 1, per_site, infos)
    got = record_run(a, S, B, [(f, g) for f, g in batches], capi.HOST_BGZF, 1, per_site, infos)
    assert got[1][1] > old_cover, (got[1][1], old_cover)
    assert got[1][0] == want[1][0] and got[0][0] == want[0][0]
    assert len(want[1][0]) > 2 * len(pt)


def test_gvcf_waits_out_of_submission_order_are_refused():
    a = vargs.parse_args("--seed 1 -d 10 -e 0.001 -GL 1 -doUnobserved 1 -doGVCF 1 --gvcf-dps 1,5,10 -addPL 1".split())
    S, B = 4, 16
    ctx = capi.Context(capi.params_from_args(a, S, B, n_slots=3, host_output=capi.HOST_BCF,
                                             bcf_dict=dict(DP=1, GL=2, PL=3, END=4, MIN_DP=5)))
    ctx.set_gvcf_dps([1, 5, 10])
    for slot in range(3):
        ctx.input_buffer(slot)[:B] = synth.pack_gt(synth.sfs_genotypes(B, S, slot))
        fill_bcf_input(ctx, slot, slot * B, B)
        ctx.submit(slot, slot * B, B)
    for slot in (1, 2):
        with pytest.raises(capi.VglError) as e:
            ctx.wait(slot)
        assert e.value.code == capi.VGL_ESTATE
    for slot in range(3):
        assert ctx.wait(slot).status == 0
    assert ctx.wait(0).status == 0      # a slot already waited may be read again
    ctx.close()
