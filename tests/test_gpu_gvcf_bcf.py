"""-doGVCF 1 through VGL_HOST_BCF: the block merger AND the record serialisation on the device, the seam between batches
stitched inside vgl_wait (csrc/capi.cu gvcf_seam: a block open at a batch's end is held back, merged with the next batch's
first block when that continues it -- the one record encoded on the host -- and the last one comes from vgl_gvcf_flush).

The reference's own -doGVCF runs (three of its golden tests + five more, tests/golden/gvcf, tools/make_golden_gvcf.py) are
replayed on the device from the captures, cut into batches of several sizes; the concatenated output must be the record
stream of the file the UNMODIFIED reference wrote (-O u), byte for byte: regular records, block records with END / MIN_DP /
QS / PL / DP, in order."""
import numpy as np
import pytest

import bcf_util as bu
import golden_cases as gc
import gvcf_util as gu
import replay_util
from vcfgl_b200 import capi

pytestmark = pytest.mark.gpu
bo, go = gu.bo, gu.go


def all_sites(cid):
    return gc.case_sites(cid) if cid in gu.MAIN_GVCF else gu.vgl_dump.read_dump(gu.os.path.join(gu.GVCF_DIR, cid + ".vgld.gz"))


# (batch size, slots): with three slots, up to three batches are in flight before the first wait (the seam is stitched in
# vgl_wait, in submission order)
BATCHES = [pytest.param(0, 1, id="0"), pytest.param(1, 1, id="1"), pytest.param(7, 1, id="7"), pytest.param(13, 1, id="13"),
           pytest.param(7, 3, id="7-slots3"), pytest.param(13, 3, id="13-slots3")]


@pytest.mark.parametrize("batch,n_slots", BATCHES)
@pytest.mark.parametrize("cid", gu.CASES)
def test_gvcf_record_stream_equals_the_reference_file(cid, batch, n_slots):
    a, kept, (_, ids, recs) = gu.load(cid)
    if a.do_unobserved not in (1, 2):
        pytest.skip("the reference itself stops at the second member of a block with -doUnobserved 4|5")
    sites = all_sites(cid)
    S, n = sites[0].S, len(sites)
    batch = batch or n
    want = go.merge(gu.oracle_input(kept), gu.dps_of(a))
    assert len(want) == len(recs)
    idx = [i for i, d in enumerate(sites) if d.ret == 0]      # written sites -> capture indices
    d_ids = {k.split("/")[1].lower(): v for k, v in ids.items() if k.split("/")[0] in ("FORMAT", "INFO")}
    bcf_dict = {k: d_ids[k] for k in ("dp", "gl", "pl", "gp", "ad", "adf", "adr", "qs", "i16", "end", "min_dp") if k in d_ids}
    ctx = capi.Context(capi.params_from_args(a, S, max_batch_sites=batch, n_slots=n_slots, host_output=capi.HOST_BCF, bcf_dict=bcf_dict,
                                             bcf_blob_bytes_per_site=96))
    ctx.set_gvcf_dps(gu.dps_of(a))
    # pass-through fields of the regular records (block records are cleared records): from the reference's own output
    _, itags = bu.enabled_tags(a)
    pt = {}
    for o, rec in zip(want, recs):
        if o["kind"] == "site":
            r = bo.split_record(rec)
            n_in = r["n_info"] - len(itags)
            pt[idx[o["site"]]] = (r["qual_bits"], n_in, r["id_bytes"], r["filter_bytes"] + b"".join(b for _, b in r["infos"][:n_in]))
    got = bytearray()
    n_out = 0
    pending = []

    def take():
        nonlocal n_out
        b = ctx.wait(pending.pop(0))
        assert b.status == 0 and b.bcf_off is None
        got.extend(bytes(b.bcf) if b.bcf is not None else b"")
        n_out += b.n_recs
    for j, lo in enumerate(range(0, n, batch)):
        slot = j % n_slots
        if len(pending) == n_slots:
            take()
        part = sites[lo:lo + batch]
        m = len(part)
        gt, rp = replay_util.batch_from_dump(part, a)
        ctx.input_buffer(slot)[:m] = gt
        sin, blob = ctx.bcf_input(slot)
        sin[:m] = 0
        o_ = 0
        for k, d in enumerate(part):
            sin[k]["rid"], sin[k]["pos"], sin[k]["qual_bits"] = d.rid, d.pos, capi.F32_MISSING_BITS
            if lo + k in pt:
                qb, n_in, idb, fi = pt[lo + k]
                sin[k]["qual_bits"], sin[k]["n_info"] = qb, n_in
                if idb != b"\x07":
                    sin[k]["id_off"], sin[k]["id_len"] = o_, len(idb)
                    blob[o_:o_ + len(idb)] = np.frombuffer(idb, np.uint8)
                    o_ += len(idb)
                if fi != b"\x00":
                    sin[k]["flt_info_off"], sin[k]["flt_info_len"] = o_, len(fi)
                    blob[o_:o_ + len(fi)] = np.frombuffer(fi, np.uint8)
                    o_ += len(fi)
        ctx.submit(slot, lo, m, replay=rp)
        pending.append(slot)
    while pending:
        take()
    tail = ctx.gvcf_flush()
    got += tail
    n_out += 1 if tail else 0
    assert ctx.gvcf_flush() == b""
    ctx.close()
    assert n_out == len(recs)
    assert bytes(got) == b"".join(recs), (cid, batch)
