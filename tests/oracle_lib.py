"""ctypes access to oracle/libvgl_oracle.so (the plain-C CPU restatement) --
test infrastructure; never imported by the product package."""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIB = os.path.join(ORACLE_DIR, "libvgl_oracle.so")


class VgoParams(C.Structure):
    _fields_ = [("n_samples", C.c_int32), ("error_rate", C.c_double), ("error_qs", C.c_int32),
                ("gl_model", C.c_int32), ("gl1_theta", C.c_double), ("precise_gl", C.c_int32),
                ("adjust_qs", C.c_int32), ("adjust_by", C.c_double), ("n_qs_bins", C.c_int32),
                ("qs_bins", (C.c_uint8 * 3) * 255), ("do_unobserved", C.c_int32),
                ("rm_invar_sites", C.c_int32), ("rm_empty_sites", C.c_int32), ("do_gvcf", C.c_int32),
                ("i16_mapq", C.c_int32),
                ("add_gl", C.c_int32), ("add_gp", C.c_int32), ("add_pl", C.c_int32),
                ("add_i16", C.c_int32), ("add_qs", C.c_int32),
                ("add_fmt_dp", C.c_int32), ("add_info_dp", C.c_int32),
                ("add_fmt_ad", C.c_int32), ("add_info_ad", C.c_int32),
                ("add_fmt_adf", C.c_int32), ("add_info_adf", C.c_int32),
                ("add_fmt_adr", C.c_int32), ("add_info_adr", C.c_int32)]


class VgoSiteIn(C.Structure):
    _fields_ = [("gts", C.c_void_p), ("depths", C.c_void_p), ("n_reads", C.c_int32),
                ("bases", C.c_void_p), ("strands", C.c_void_p), ("qs", C.c_void_p),
                ("adj_qs", C.c_void_p), ("eprob", C.c_void_p), ("n_tails", C.c_int32),
                ("tails", C.c_void_p), ("n_em", C.c_int32), ("em_sample", C.c_void_p),
                ("em_n", C.c_void_p), ("em_codes", C.c_void_p)]


class VgoSiteOut(C.Structure):
    _fields_ = [("ret", C.c_int32), ("n_alleles", C.c_int32), ("n_alleles_observed", C.c_int32),
                ("n_genotypes", C.c_int32), ("allele_unobserved", C.c_int32),
                ("alleles2acgt", C.c_int32 * 5), ("acgt2alleles", C.c_int32 * 5),
                ("info_dp", C.c_int32), ("fmt_dp", C.c_void_p), ("gl", C.c_void_p),
                ("pl", C.c_void_p), ("gp", C.c_void_p), ("fmt_ad", C.c_void_p),
                ("fmt_adf", C.c_void_p), ("fmt_adr", C.c_void_p),
                ("info_ad", C.c_int32 * 5), ("info_adf", C.c_int32 * 5), ("info_adr", C.c_int32 * 5),
                ("qs", C.c_float * 5), ("i16", C.c_float * 16)]


def build_oracle(force=False):
    src = os.path.join(ORACLE_DIR, "vgl_oracle.c")
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "libvgl_oracle.so"], stdout=subprocess.DEVNULL)
    return LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build_oracle())
        _lib.vgo_create.restype = C.c_void_p
        _lib.vgo_create.argtypes = [C.POINTER(VgoParams)]
        _lib.vgo_destroy.argtypes = [C.c_void_p]
        _lib.vgo_site.argtypes = [C.c_void_p, C.POINTER(VgoSiteIn), C.POINTER(VgoSiteOut)]
        _lib.vgo_site.restype = C.c_int
        _lib.vgo_precalc_qs.argtypes = [C.c_void_p]
        _lib.vgo_precalc_adj_qs.argtypes = [C.c_void_p]
        _lib.vgo_precalc_gl2.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        _lib.vgo_lut_log10_gl.restype = C.POINTER(C.c_double)
        for f in ("vgo_errmod_fk", "vgo_errmod_beta", "vgo_errmod_lhet"):
            getattr(_lib, f).restype = C.POINTER(C.c_double)
            getattr(_lib, f).argtypes = [C.c_void_p]
        _lib.vgo_errmod_cal.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    return _lib


def params_from_args(a, n_samples) -> VgoParams:
    """vcfgl_b200.args.SimArgs -> vgo_params"""
    p = VgoParams()
    p.n_samples = n_samples
    p.error_rate = a.error_rate
    p.error_qs = a.error_qs
    p.gl_model = a.gl_model
    p.gl1_theta = a.gl1_theta
    p.precise_gl = a.precise_gl
    p.adjust_qs = a.adjust_qs
    p.adjust_by = a.adjust_by
    bins = a.qs_bins or []
    p.n_qs_bins = len(bins)
    for i, (s, e, q) in enumerate(bins):
        p.qs_bins[i][0], p.qs_bins[i][1], p.qs_bins[i][2] = s, e, q
    p.do_unobserved = a.do_unobserved
    p.rm_invar_sites = a.rm_invar_sites
    p.rm_empty_sites = a.rm_empty_sites
    p.do_gvcf = a.do_gvcf
    p.i16_mapq = a.i16_mapq
    for f in ("add_gl", "add_gp", "add_pl", "add_i16", "add_qs", "add_fmt_dp", "add_info_dp",
              "add_fmt_ad", "add_info_ad", "add_fmt_adf", "add_info_adf", "add_fmt_adr", "add_info_adr"):
        setattr(p, f, getattr(a, f))
    return p


class Oracle:
    """One oracle context (fixed params); `site()` maps draws -> tags."""

    def __init__(self, args, n_samples):
        self.S = n_samples
        self.args = args
        self.p = params_from_args(args, n_samples)
        self.ctx = lib().vgo_create(C.byref(self.p))
        assert self.ctx

    def __del__(self):
        try:
            if self.ctx:
                lib().vgo_destroy(self.ctx)
                self.ctx = None
        except Exception:
            pass

    def precalc(self):
        g = (C.c_double * 3)()
        lib().vgo_precalc_gl2(self.ctx, g)
        return lib().vgo_precalc_qs(self.ctx), lib().vgo_precalc_adj_qs(self.ctx), list(g)

    def site(self, gts, depths, bases, strands=None, qs=None, adj_qs=None, eprob=None, tails=None,
             em_sample=None, em_n=None, em_codes=None):
        S = self.S
        keep = []

        def arr(x, dt):
            if x is None:
                x = np.zeros(0, dtype=dt)
            x = np.ascontiguousarray(x, dtype=dt)
            keep.append(x)
            return x.ctypes.data

        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        n = len(bases)
        zi = np.zeros(n, np.int32)
        i = VgoSiteIn()
        i.gts = arr(gts, np.int8)
        i.depths = arr(depths, np.int32)
        i.n_reads = n
        i.bases = arr(bases, np.uint8)
        i.strands = arr(strands if strands is not None else np.zeros(n, np.uint8), np.uint8)
        i.qs = arr(qs if qs is not None else zi, np.int32)
        i.adj_qs = arr(adj_qs if adj_qs is not None else zi, np.int32)
        i.eprob = arr(eprob if eprob is not None else np.zeros(n), np.float64)
        tails = np.zeros(0, np.int32) if tails is None else np.asarray(tails, np.int32)
        i.n_tails = len(tails)
        i.tails = arr(tails, np.int32)
        em_sample = np.zeros(0, np.int32) if em_sample is None else em_sample
        i.n_em = len(em_sample)
        i.em_sample = arr(em_sample, np.int32)
        i.em_n = arr(em_n, np.int32)
        i.em_codes = arr(em_codes, np.uint16)
        o = VgoSiteOut()
        res = dict(fmt_dp=np.zeros(S, np.int32), gl=np.zeros(S * 15, np.float32),
                   pl=np.zeros(S * 15, np.int32), gp=np.zeros(S * 15, np.float32),
                   fmt_ad=np.zeros(S * 5, np.int32), fmt_adf=np.zeros(S * 5, np.int32),
                   fmt_adr=np.zeros(S * 5, np.int32))
        for k, v in res.items():
            setattr(o, k, v.ctypes.data)
        ret = lib().vgo_site(self.ctx, C.byref(i), C.byref(o))
        G, A = o.n_genotypes, o.n_alleles
        out = dict(ret=ret, n_alleles=A, n_alleles_observed=o.n_alleles_observed, n_genotypes=G,
                   allele_unobserved=o.allele_unobserved,
                   alleles2acgt=np.array(o.alleles2acgt[:], np.int32),
                   acgt2alleles=np.array(o.acgt2alleles[:], np.int32),
                   info_dp=o.info_dp, fmt_dp=res["fmt_dp"],
                   gl=res["gl"][:S * G], pl=res["pl"][:S * G], gp=res["gp"][:S * G],
                   fmt_ad=res["fmt_ad"][:S * A], fmt_adf=res["fmt_adf"][:S * A], fmt_adr=res["fmt_adr"][:S * A],
                   info_ad=np.array(o.info_ad[:A], np.int32), info_adf=np.array(o.info_adf[:A], np.int32),
                   info_adr=np.array(o.info_adr[:A], np.int32),
                   qs=np.array(o.qs[:A], np.float32), i16=np.array(o.i16[:], np.float32))
        return out

    def site_from_dump(self, d):
        """d: tests.vgl_dump.SiteDump"""
        return self.site(d.gts, d.depths, d.r_base, d.r_strand, d.r_qs, d.r_adjqs, d.r_eprob, d.tails,
                         d.em_sample, d.em_n, d.em_codes)


F32_MISSING_BITS = 0x7F800001      # VGO_MISSING_F32_BITS (bcf_float_missing)


def _bits(x):
    return np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)


def check_gp(gp, gl_oracle, gp_oracle, fmt_dp, G):
    """FORMAT/GP of one site ([S * G] float32) against
    (a) a float64 reference made from the oracle's GL, independent of the float order of oracle and kernel:
        ref = 10^gl / sum(10^gl) per sample, |gp - ref| <= (G + 2) 2^-24 ref + 2^-149 -- the float rounding of each term,
        of the float sum of G positive terms and of the division; 2^-149 covers a subnormal GP (GL < -38);
    (b) the oracle's GP: bit-equal or 1 float ulp apart (the device takes exp10 in double, the oracle libm pow: the two may
        round to different floats);
    (c) the missing value exactly in the samples with FORMAT/DP == 0.
    Returns (values bit-equal to the oracle, values compared)."""
    gp = _bits(gp).reshape(-1, G)
    want = _bits(gp_oracle).reshape(-1, G)
    assert gp.shape == want.shape, (gp.shape, want.shape)
    dp0 = np.asarray(fmt_dp) == 0
    miss = gp == F32_MISSING_BITS
    assert (miss == dp0[:, None]).all(), ("GP missing where FORMAT/DP > 0, or set where FORMAT/DP == 0", np.nonzero(miss != dp0[:, None]))
    have = ~dp0
    got = gp[have].view(np.float32).astype(np.float64)
    e = 10.0 ** np.asarray(gl_oracle, np.float32).reshape(-1, G)[have].astype(np.float64)
    ref = e / e.sum(axis=1, keepdims=True)
    bound = (G + 2) * 2.0 ** -24 * ref + 2.0 ** -149
    bad = ~(np.abs(got - ref) <= bound)
    assert not bad.any(), ("GP off the float64 reference", got[bad], ref[bad])
    ulps = np.abs(gp[have].astype(np.int64) - want[have].astype(np.int64))     # both non-negative floats: bits are monotonic
    assert (ulps <= 1).all(), ("GP more than 1 ulp from the oracle", got[ulps > 1], want[have][ulps > 1].view(np.float32))
    return int((ulps == 0).sum()), int(ulps.size)


def check_sites_on_draws(a, S, hap, native, rp, gl_rtol=0.0, idx=None, orc=None, gp_share=None):
    """The oracle run on a batch's own draws (vgl_native_draws: `rp`) must give the tags the kernels emitted for that batch:
    native[i] = Batch.site(i) of site i, hap = int8 [n_sites, 2S] true genotypes.  Every field of the record (n_alleles*,
    INFO/DP, INFO AD family, QS, I16; the allele maps where INFO/DP > 0) and every plane asked for (FORMAT/DP, GL, PL, the
    FORMAT AD family; GP through check_gp).  A plane the arguments ask for that the batch does not return is a failure.  GL bit
    for bit, or (gl_rtol > 0) within that relative tolerance where the bits differ.  `idx`: the sites to compare (default:
    all); `orc`: an Oracle of (a, S) to reuse; `gp_share`: a [bit-equal, compared] pair the GP counts are added to.
    Returns the number of written sites compared."""
    orc = orc or Oracle(a, S)
    off = rp["read_offsets"]
    n_cmp = 0
    for i in (range(len(native)) if idx is None else idx):
        d = native[i]
        sl = slice(off[i * S], off[(i + 1) * S])
        o = orc.site(hap[i], rp["depths"][i * S:(i + 1) * S], rp["bases"][sl], rp["strands"][sl],
                     None if rp["qs"] is None else rp["qs"][sl].astype(np.int32),
                     None if rp["adj_qs"] is None else rp["adj_qs"][sl].astype(np.int32),
                     None if rp["error_probs"] is None else rp["error_probs"][sl],
                     rp["tail_dists"][sl].astype(np.int32) if a.add_i16 else None)
        assert o["ret"] == d["skip_code"], i
        if a.add_fmt_dp:
            assert d.get("fmt_dp") is not None, (i, "fmt_dp")
            assert np.array_equal(o["fmt_dp"], d["fmt_dp"]), (i, "fmt_dp")
        if o["ret"] != 0:
            continue
        assert o["n_alleles"] == d["n_alleles"] and o["n_genotypes"] == d["n_genotypes"], i
        assert o["n_alleles_observed"] == d["n_alleles_observed"], (i, o["n_alleles_observed"], d["n_alleles_observed"])
        assert o["info_dp"] == d["info_dp"], (i, o["info_dp"], d["info_dp"])
        if o["info_dp"] > 0:
            assert np.array_equal(o["alleles2acgt"], d["alleles2acgt"]), (i, o["alleles2acgt"], d["alleles2acgt"])
            assert np.array_equal(o["acgt2alleles"], d["acgt2alleles"]), (i, o["acgt2alleles"], d["acgt2alleles"])
        for key in ("pl", "fmt_ad", "fmt_adf", "fmt_adr", "info_ad", "info_adf", "info_adr"):
            if not getattr(a, "add_" + key):
                continue
            assert d.get(key) is not None, (i, key, "asked for, not returned")
            assert np.array_equal(o[key], d[key]), (i, key, o[key], d[key])
        if a.add_gl:
            assert d.get("gl") is not None, (i, "gl", "asked for, not returned")
            same = o["gl"].view(np.uint32) == _bits(d["gl"])   # missing (a NaN payload) compares by bits
            if gl_rtol > 0:
                with np.errstate(invalid="ignore"):
                    same |= np.abs(o["gl"].astype(np.float64) - d["gl"]) <= gl_rtol * np.abs(d["gl"].astype(np.float64))
            assert same.all(), i
        if a.add_gp:
            assert d.get("gp") is not None, (i, "gp", "asked for, not returned")
            eq, n = check_gp(d["gp"], o["gl"], o["gp"], o["fmt_dp"], o["n_genotypes"])
            if gp_share is not None:
                gp_share[0] += eq
                gp_share[1] += n
        if a.add_qs:
            assert np.array_equal(o["qs"].view(np.uint32), _bits(d["qs"])), i
        if a.add_i16:
            assert np.array_equal(o["i16"].view(np.uint32), _bits(d["i16"])), (i, o["i16"], d["i16"])
        n_cmp += 1
    return n_cmp
