"""GPU parity of the OUTPUT path (VGL_HOST_BCF, csrc/bcf.cu): the records serialised on the device must be the bytes
the reference writes.

(1) replay: every non-gVCF golden case is replayed through the C ABI with the reference's own draws and the device's
    record stream is compared with the file the UNMODIFIED reference binary wrote with `-O u` (tests/golden/bcf/):
    byte-identical, except inside float FORMAT blocks of runs whose floats may differ in the last place from glibc's
    (GP, --precise-gl 1; see test_gpu_replay_parity.py), where 1e-6 relative applies and everything else must be equal.
(2) native: the record stream of a native batch equals the CPU oracle's encoding (oracle/bcf_oracle.py, pinned on the
    reference's bytes by test_bcf_oracle.py) of the arrays the same seed yields through VGL_HOST_I32 -- at sizes and
    value ranges the reference captures do not reach (int16 / int32 vectors, long pass-through fields, odd alignments)."""
import struct

import numpy as np
import pytest

import bcf_util as bu
import golden_cases as gc
import replay_util
from vcfgl_b200 import args as vargs
from vcfgl_b200 import capi, synth

pytestmark = pytest.mark.gpu
bo = bu.bo
REL_TOL = 1e-6


def dict_from_ids(ids):
    d = {}
    for k, v in ids.items():
        kind, name = k.split("/")
        if kind in ("FORMAT", "INFO"):
            d[name] = v
    return {k: v for k, v in d.items() if k.lower() in ("dp", "gl", "pl", "gp", "ad", "adf", "adr", "qs", "i16")}


def assert_records_close(got, want, where):
    """identical bytes, or identical in everything but float FORMAT payloads, which agree to REL_TOL"""
    if got == want:
        return True
    g, w = bo.split_record(got), bo.split_record(want)
    for k in ("rid", "pos", "rlen", "qual_bits", "n_info", "n_allele", "n_sample", "n_fmt", "id_bytes", "alleles", "filter_bytes"):
        assert g[k] == w[k], (where, k, g[k], w[k])
    assert [k for k, _ in g["infos"]] == [k for k, _ in w["infos"]]
    for (kg, bg), (kw, bw) in zip(g["infos"], w["infos"]):
        if bg != bw:   # INFO floats (QS) of the inexact cases
            assert len(bg) == len(bw) and bg[:3] == bw[:3], (where, "info", kg)
    for (kg, ng, tg, bg), (kw, nw, tw, bw) in zip(g["fmts"], w["fmts"]):
        assert (kg, ng, tg, len(bg)) == (kw, nw, tw, len(bw)), (where, "fmt", kg)
        if bg == bw:
            continue
        assert tg == bo.BT_FLOAT, (where, "integer FORMAT block differs", kg)
        n = ng * g["n_sample"]
        x = np.frombuffer(bg[-4 * n:], "<f4").astype(np.float64)
        y = np.frombuffer(bw[-4 * n:], "<f4").astype(np.float64)
        same = np.frombuffer(bg[-4 * n:], "<u4") == np.frombuffer(bw[-4 * n:], "<u4")
        with np.errstate(invalid="ignore"):
            near = np.isfinite(x) & np.isfinite(y) & (np.abs(x - y) <= REL_TOL * np.maximum(np.abs(y), 1e-30))
        assert (same | near).all(), (where, "float FORMAT block", kg)
    return False


@pytest.mark.parametrize("cid", bu.BCF_CASES + gc.FUZZ_IDS)
def test_replay_records_equal_the_reference_file(cid):
    a = bu.any_args(cid)
    sites = bu.any_sites(cid)
    S = sites[0].S
    _, ids, recs = bu.reference_bcf(cid)
    gt, rp = replay_util.batch_from_dump(sites, a)
    n = len(sites)
    prm = capi.params_from_args(a, S, max_batch_sites=n, n_slots=1, host_output=capi.HOST_BCF, bcf_dict=dict_from_ids(ids))
    ctx = capi.Context(prm)
    ctx.input_buffer(0)[:n] = gt
    sin, blob = ctx.bcf_input(0)
    # pass-through fields: what the reference kept of each INPUT record = the ID / FILTER (+ the input's own INFO) bytes of its
    # output record; skipped sites have no record and keep the "." defaults
    _, itags = bu.enabled_tags(a)
    kept = [k for k, d in enumerate(sites) if d.ret == 0]
    assert len(kept) == len(recs)
    o = 0
    sin[:n] = 0
    for k, d in enumerate(sites):
        sin[k]["rid"], sin[k]["pos"], sin[k]["qual_bits"] = d.rid, d.pos, capi.F32_MISSING_BITS
    for k, rec in zip(kept, recs):
        r = bo.split_record(rec)
        n_in = r["n_info"] - len(itags)
        pt = r["filter_bytes"] + b"".join(b for _, b in r["infos"][:n_in])
        sin[k]["qual_bits"], sin[k]["n_info"] = r["qual_bits"], n_in
        if r["id_bytes"] != b"\x07":
            sin[k]["id_off"], sin[k]["id_len"] = o, len(r["id_bytes"])
            blob[o:o + len(r["id_bytes"])] = np.frombuffer(r["id_bytes"], np.uint8)
            o += len(r["id_bytes"])
        if pt != b"\x00":
            sin[k]["flt_info_off"], sin[k]["flt_info_len"] = o, len(pt)
            blob[o:o + len(pt)] = np.frombuffer(pt, np.uint8)
            o += len(pt)
    ctx.submit(0, 1000, n, replay=rp)
    b = ctx.wait(0)
    assert b.status == 0
    exact = not (a.add_gp or (a.precise_gl and a.error_qs == 2))
    n_same = 0
    for j, (k, want) in enumerate(zip(kept, recs)):
        lo, hi = int(b.bcf_off[k]), int(b.bcf_off[k + 1])
        got = bytes(b.bcf[lo:hi])
        if exact:
            assert got == want, (cid, k, sites[k].pos)
            n_same += 1
        else:
            n_same += assert_records_close(got, want, (cid, k))
    for k, d in enumerate(sites):
        if d.ret != 0:
            assert b.bcf_off[k] == b.bcf_off[k + 1] and b.sites[k]["skip_code"] == d.ret
    assert b.bcf_bytes == int(b.bcf_off[n]) == sum(len(r) for r in recs)
    if exact:   # the whole stream is what the reference wrote after its header
        assert bytes(b.bcf) == b"".join(recs)
    assert n_same >= 0.5 * len(recs)
    ctx.close()


def _native_pair(argv, S, n_sites, batch, passthrough_seed=None, missing=0.0, fixed_depth=False, in_fmt_seed=None):
    """run the same native batch through VGL_HOST_I32 and VGL_HOST_BCF; returns (expected stream from the oracle, got)"""
    a = vargs.parse_args(argv.split())
    hap = synth.sfs_genotypes(n_sites, S, 4242, missing)
    gt = synth.pack_gt(hap)
    ids = dict(DP=1, GL=2, PL=3, GP=4, AD=5, ADF=200, ADR=7, QS=40000, I16=9)   # ADF: 16-bit key, QS: 32-bit key
    dict_ids = {"FORMAT/" + k: v for k, v in ids.items()}
    dict_ids.update({"INFO/" + k: v for k, v in ids.items()})
    rng = np.random.default_rng(passthrough_seed or 0)
    ref = capi.Context(capi.params_from_args(a, S, max_batch_sites=batch, n_slots=1, host_output=capi.HOST_I32, fixed_depth=fixed_depth))
    dev = capi.Context(capi.params_from_args(a, S, max_batch_sites=batch, n_slots=2, host_output=capi.HOST_BCF, bcf_dict=ids,
                                             bcf_blob_bytes_per_site=64 + (12 * S + 32 if in_fmt_seed is not None else 0), fixed_depth=fixed_depth))
    frng = np.random.default_rng(in_fmt_seed or 0)
    ftags, itags = bu.enabled_tags(a)
    want, got = [], []
    slot = 0
    for s0 in range(0, n_sites, batch):
        m = min(batch, n_sites - s0)
        ref.input_buffer(0)[:m] = gt[s0:s0 + m]
        ref.submit(0, s0, m)
        rb = ref.wait(0)
        dev.input_buffer(slot)[:m] = gt[s0:s0 + m]
        sin, blob = dev.bcf_input(slot)
        sin[:m] = 0
        pts = []
        o = 0
        for k in range(m):
            sin[k]["rid"], sin[k]["pos"], sin[k]["qual_bits"] = (s0 + k) % 3, 10 * (s0 + k) + 7, capi.F32_MISSING_BITS
            idb, pt, n_in = b"\x07", b"\x00", 0
            if passthrough_seed is not None and rng.random() < 0.7:
                name = ("rs%d" % rng.integers(1, 10 ** int(rng.integers(1, 9)))).encode()
                idb = bo.enc_vchar(name)
                pt = bo.enc_vint([0] if rng.random() < 0.5 else [3, 5])
                if rng.random() < 0.5:   # one INFO field of the input record: key 11, a float vector
                    pt += bo.enc_int1(11) + bo.enc_vfloat(rng.random(int(rng.integers(1, 4))).astype(np.float32))
                    n_in = 1
                sin[k]["qual_bits"] = int(np.float32(rng.random() * 100).view(np.uint32))
                sin[k]["id_off"], sin[k]["id_len"] = o, len(idb)
                blob[o:o + len(idb)] = np.frombuffer(idb, np.uint8)
                o += len(idb)
                sin[k]["flt_info_off"], sin[k]["flt_info_len"] = o, len(pt)
                blob[o:o + len(pt)] = np.frombuffer(pt, np.uint8)
                o += len(pt)
                sin[k]["n_info"] = n_in
            in_fmt = []
            if in_fmt_seed is not None and frng.random() < 0.8:
                # FORMAT blocks of the input record besides GT (the reference keeps them, vcfgl.cpp:793): an input DP (key of the
                # simulated DP: replaced in place), GQ (int8 / int16), a float vector, a per-sample string -- in random order
                cand = [(ids["DP"], bo.enc_int1(ids["DP"]) + bo.enc_vint(frng.integers(0, 90, S), 1)),
                        (60, bo.enc_int1(60) + bo.enc_vint(frng.integers(0, 300 if frng.random() < 0.5 else 99, S), 1)),
                        (61, bo.enc_int1(61) + bo.enc_size(2, bo.BT_FLOAT) + frng.random(2 * S).astype("<f4").tobytes()),
                        (300, bo.enc_int1(300) + bo.enc_size(3, bo.BT_CHAR) + bytes(frng.integers(65, 90, 3 * S).astype(np.uint8)))]
                pick = [cand[j] for j in frng.permutation(4)[:int(frng.integers(1, 5))]]
                in_fmt = pick
                fb = b"".join(x[1] for x in pick)
                sin[k]["fmt_off"], sin[k]["fmt_len"], sin[k]["n_fmt"] = o, len(fb), len(pick)
                blob[o:o + len(fb)] = np.frombuffer(fb, np.uint8)
                o += len(fb)
            pts.append((idb, pt, n_in, int(sin[k]["qual_bits"]), in_fmt))
        dev.submit(slot, s0, m)
        db = dev.wait(slot)
        assert db.status == 0 and rb.status == 0
        for k in range(m):
            o_ = rb.site(k)
            lo, hi = int(db.bcf_off[k]), int(db.bcf_off[k + 1])
            assert db.sites[k]["skip_code"] == o_["skip_code"]
            if o_["skip_code"] != 0:
                assert lo == hi
                continue
            fmt = {t: {"DP": o_["fmt_dp"], "GL": o_.get("gl"), "PL": o_.get("pl"), "GP": o_.get("gp"), "AD": o_.get("fmt_ad"),
                       "ADF": o_.get("fmt_adf"), "ADR": o_.get("fmt_adr")}[t] for t in ftags}
            info = {t: {"DP": np.array([o_["info_dp"]]), "QS": o_["qs"], "I16": o_["i16"], "AD": o_["info_ad"], "ADF": o_["info_adf"],
                        "ADR": o_["info_adr"]}[t] for t in itags}
            alleles = bo.alleles_of_site(o_["n_alleles"], o_["alleles2acgt"], o_["info_dp"], a.do_unobserved, a.do_gvcf)
            idb, pt, n_in, qb, in_fmt = pts[k]
            want.append(bo.encode_record((s0 + k) % 3, 10 * (s0 + k) + 7, qb, idb, pt, n_in, alleles, S, dict_ids, fmt, info, in_fmt=in_fmt))
            got.append(bytes(db.bcf[lo:hi]))
        assert db.bcf_bytes == int(db.bcf_off[m])
        slot ^= 1
    ref.close()
    dev.close()
    return want, got


def _check(want, got):
    assert len(want) == len(got) and len(want) > 0
    for k, (w, g) in enumerate(zip(want, got)):
        assert g == w, (k, len(g), len(w), next((i for i in range(min(len(g), len(w))) if g[i] != w[i]), None))


def test_native_cfg2_stream_equals_oracle():
    want, got = _native_pair("--seed 42 -d 10 -e 0.01 -GL 1 -addGL 1 -addPL 1 -addFormatAD 1", 100, 3000, 1024)
    _check(want, got)
    kinds = {bo.split_record(g)["fmts"][2][2] for g in got}     # PL comes as int8 where max <= 127, else int16
    assert kinds == {bo.BT_INT8, bo.BT_INT16} or kinds == {bo.BT_INT16}


def test_native_all_tags_wide_vectors_and_passthrough():
    # depth 300 -> FORMAT AD / DP need int16, 150 samples x 300 reads -> INFO AD / DP need int32; 16- and 32-bit dictionary keys;
    # IDs, QUAL, FILTER lists and an INFO field of the input record ride along at every byte alignment
    tags = "-addGP 1 -addPL 1 -addI16 1 -addQS 1 -addInfoDP 1 -addFormatAD 1 -addInfoAD 1 -addFormatADF 1 -addInfoADF 1 -addFormatADR 1 -addInfoADR 1"
    want, got = _native_pair("--seed 7 -d 300 -e 0.02 -GL 2 -doUnobserved 2 " + tags, 150, 96, 40, passthrough_seed=5)
    _check(want, got)
    r = bo.split_record(got[0])
    assert {t for _, _, t, _ in r["fmts"]} >= {bo.BT_INT16, bo.BT_FLOAT}


@pytest.mark.parametrize("S,tags", [(7, "-addPL 1 -addFormatAD 1"), (33, "-addGP 1 -addPL 1 -addFormatAD 1 -addFormatADF 1 -addInfoDP 1"),
                                    (120, "-addGL 1 -addPL 1 -addFormatDP 0")])
def test_native_input_records_with_other_format_keys(S, tags):
    # the input record carries FORMAT blocks besides GT (GT:DP:GQ ...): the reference keeps them in front of the simulated tags and
    # replaces an input DP in place (layout pinned on the reference by tests/test_bcf_live_reference.py through the same oracle)
    want, got = _native_pair("--seed 21 -d 6 -e 0.02 -GL 1 -doUnobserved 1 " + tags, S, 400, 128, passthrough_seed=3, in_fmt_seed=9)
    _check(want, got)
    assert any(len(bo.split_record(g)["fmts"]) > 4 for g in got)


@pytest.mark.parametrize("S", [1, 2, 3, 5, 33])
def test_native_small_sample_counts_missing_and_empty_sites(S):
    # tiny records (every word straddles segments), missing genotypes, sites without reads kept (--rm-empty-sites 0) in every
    # -doUnobserved mode, one sample (bcf_enc_vint's n == 1 form)
    for unobs in range(6):
        want, got = _native_pair("--seed %d -d 0.4 -e 0.05 -GL 1 -doUnobserved %d -addPL 1 -addFormatAD 1 -addInfoAD 1 -addInfoDP 1 -addQS 1"
                                 % (11 + unobs, unobs), S, 300, 128, passthrough_seed=unobs + 1, missing=0.2)
        _check(want, got)


def test_native_ten_thousand_samples():
    want, got = _native_pair("--seed 42 -d 30 -e 0.01 -GL 1 -addPL 1 -addFormatAD 1", 10000, 24, 16)
    _check(want, got)


def test_gvcf_record_modes_that_are_rejected():
    # -doGVCF through VGL_HOST_BCF needs the block merger's requirements (-doUnobserved 1|2: tests/test_gpu_gvcf_bcf.py covers the mode);
    # the BGZF stream cannot be spliced at batch seams, and a submit without the thresholds is a state error
    a = vargs.parse_args("--seed 1 -d 10 -e 0.001 -GL 1 -doUnobserved 4 -doGVCF 1 --gvcf-dps 1,5,10 -addPL 1".split())
    with pytest.raises(capi.VglError) as e:
        capi.Context(capi.params_from_args(a, 4, 16, host_output=capi.HOST_BCF))
    assert e.value.code == capi.VGL_EINVAL
    a = vargs.parse_args("--seed 1 -d 10 -e 0.001 -GL 1 -doUnobserved 1 -doGVCF 1 --gvcf-dps 1,5,10 -addPL 1".split())
    with pytest.raises(capi.VglError) as e:
        capi.Context(capi.params_from_args(a, 4, 16, host_output=capi.HOST_BGZF))
    assert e.value.code == capi.VGL_EINVAL
    ctx = capi.Context(capi.params_from_args(a, 4, 16, n_slots=1, host_output=capi.HOST_BCF, bcf_dict=dict(DP=1, GL=2, PL=3, END=4, MIN_DP=5)))
    ctx.input_buffer(0)[:] = 0
    with pytest.raises(capi.VglError) as e:
        ctx.submit(0, 0, 16)
    assert e.value.code == capi.VGL_ESTATE
    ctx.close()


def test_cpp_host_stream_writes_a_bcf_file_the_oracle_reads(tmp_path):
    """vcfgl_b200/host/vgl_host.hpp BcfStreamSimulator (C++ host mirror over the C ABI): the file the example driver writes
    parses as BCF and its records equal the oracle's encoding of the arrays the same parameters give through Python."""
    import os
    import subprocess
    exe = os.path.join(bu.ROOT, "vcfgl_b200", "host", "example_driver")
    if not os.path.exists(exe):
        pytest.skip("example_driver not built")
    out = str(tmp_path / "x.bcf")
    n_sites, S = 11, 4
    subprocess.check_call([exe, str(n_sites)], env=dict(os.environ, VGL_BCF_OUT=out))
    _, ids, recs = bo.read_bcf(out)
    a = vargs.parse_args("--seed 42 -d 4 -e 0.01 -GL 1 -doUnobserved 1 -addGL 1 -addPL 1 -addFormatAD 1 -addInfoDP 1".split())
    gts = np.zeros((n_sites, 2 * S), np.int8)
    for i in range(n_sites):
        for s in range(S):
            gts[i, 2 * s] = 1 if (i + s) % 3 == 2 else 0
            gts[i, 2 * s + 1] = 1 if (i + s) % 3 >= 1 else 0
    ctx = capi.Context(capi.params_from_args(a, S, max_batch_sites=16, n_slots=1))
    ctx.input_buffer(0)[:n_sites] = synth.pack_gt(gts)
    ctx.submit(0, 0, n_sites)
    b = ctx.wait(0)
    want = []
    for k in range(n_sites):
        o = b.site(k)
        if o["skip_code"] != 0:
            continue
        fmt = {"DP": o["fmt_dp"], "GL": o["gl"], "PL": o["pl"], "AD": o["fmt_ad"]}
        alleles = bo.alleles_of_site(o["n_alleles"], o["alleles2acgt"], o["info_dp"], 1, 0)
        want.append(bo.encode_record(0, 10 * k + 1, capi.F32_MISSING_BITS, b"\x07", b"\x11\x00", 0, alleles, S, ids, fmt,
                                     {"DP": np.array([o["info_dp"]])}))
    ctx.close()
    assert recs == want


def test_cpp_host_stream_writes_a_bgzf_file(tmp_path):
    """the same driver with VGL_BGZF_OUT: a complete BGZF-compressed BCF file (stored header block written by the host, the
    record blocks compressed on the device, the EOF block) -- it must gunzip to the -O u file byte for byte"""
    import gzip
    import os
    import subprocess
    exe = os.path.join(bu.ROOT, "vcfgl_b200", "host", "example_driver")
    if not os.path.exists(exe):
        pytest.skip("example_driver not built")
    plain, packed = str(tmp_path / "u.bcf"), str(tmp_path / "b.bcf")
    for n_sites, batch in ((11, 4), (3000, 1024)):
        subprocess.check_call([exe, str(n_sites)], env=dict(os.environ, VGL_BCF_OUT=plain, VGL_BATCH=str(batch)))
        subprocess.check_call([exe, str(n_sites)], env=dict(os.environ, VGL_BGZF_OUT=packed, VGL_BATCH=str(batch)))
        raw = open(packed, "rb").read()
        assert raw[:4] == b"\x1f\x8b\x08\x04" and raw[-28:] == bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
        assert gzip.open(packed, "rb").read() == open(plain, "rb").read()
        # the reference's own htslib (oracle/_ref/hts_read_bcf: hts_open / bcf_hdr_read / bcf_read) reads the file as BGZF-compressed
        # BCF and sees the records of the uncompressed one
        reader = os.path.join(bu.ROOT, "oracle", "_ref", "hts_read_bcf")
        if os.path.exists(reader):
            a_, b_ = (subprocess.check_output([reader, f]).decode().splitlines() for f in (plain, packed))
            assert a_[0].split()[:4] == ["format", "9", "compression", "0"] and b_[0].split()[:4] == ["format", "9", "compression", "2"]   # bcf; none / bgzf
            assert a_[1:] == b_[1:] and a_[-1] == "records %d" % n_sites


def test_input_record_with_fewer_format_blocks_than_n_fmt_is_rejected():
    # two blocks fill fmt_len exactly but the record promises three: vgl_submit refuses it before any copy or launch
    # (the host check: tests/test_bcf_input_check.py), and the slot takes the corrected record afterwards
    a = vargs.parse_args("--seed 1 -d 4 -e 0.01 -GL 1 -addPL 1".split())
    S = 3
    ctx = capi.Context(capi.params_from_args(a, S, 4, n_slots=1, host_output=capi.HOST_BCF, bcf_dict=dict(DP=1, GL=2, PL=3),
                                             bcf_blob_bytes_per_site=64))
    ctx.input_buffer(0)[:1] = 0
    sin, blob = ctx.bcf_input(0)
    sin[:1] = 0
    fb = bo.enc_int1(60) + bo.enc_vint([10, 20, 30], 1) + bo.enc_int1(61) + bo.enc_size(1, bo.BT_FLOAT) + np.ones(S, "<f4").tobytes()
    blob[:len(fb)] = np.frombuffer(fb, np.uint8)
    sin[0]["fmt_off"], sin[0]["fmt_len"], sin[0]["n_fmt"] = 0, len(fb), 3
    launches = ctx.launch_count()
    with pytest.raises(capi.VglError) as e:
        ctx.submit(0, 0, 1)
    assert e.value.code == capi.VGL_EINVAL and ctx.launch_count() == launches
    sin[0]["n_fmt"] = 2
    ctx.submit(0, 0, 1)
    assert ctx.wait(0).status == 0
    ctx.close()
