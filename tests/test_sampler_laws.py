"""The count-level samplers' host tables and draw keying against exact laws, on the CPU through the tables shim.

The chi-square / KS tests of tests/test_gpu_native.py cannot see a defect rarer than about 1e-4 per cell, or one that moves
mass inside a histogram bin.  These tests pin the pieces the samplers are built from instead:
- Philox4x32-10 (csrc/philox.cuh) against the Random123 known answers;
- the depth law the 256-column Walker alias table induces under the kernels' decode (tile_m1f.cu tile_sample_cell, tile_m2.cu
  m2_depth), in integers, against the Poisson pmf in 40-digit arithmetic;
- the guide table k_fused_m1f builds over the Poisson CDF (fused.cu): a lower bound of the inversion for every top byte;
- the error-count thresholds floor(P(E <= j | n) * 2^32) (binomial_cdf4_u32) against 40-digit binomial CDFs;
- the uniform maps u01_32 / u01_53 at their extreme words.
"""
import ctypes as C
import os
import subprocess

import mpmath
import numpy as np
import pytest

from vcfgl_b200 import args as vargs
from vcfgl_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, "tests", "_tables_shim.so")
CSRC = os.path.join(ROOT, "vcfgl_b200", "csrc")
TWO64 = 1 << 64
mpmath.mp.dps = 40


@pytest.fixture(scope="module")
def laws_shim():
    srcs = [os.path.join(ROOT, "tests", "tables_shim.cpp"), os.path.join(CSRC, "tables.cpp")]
    deps = srcs + [os.path.join(CSRC, "tables.h"), os.path.join(CSRC, "philox.cuh")]
    if not os.path.exists(SHIM) or os.path.getmtime(SHIM) < max(os.path.getmtime(s) for s in deps):
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-std=c++17", "-o", SHIM] + srcs)
    L = C.CDLL(SHIM)
    P = C.c_void_p
    L.shim_philox.argtypes = [C.c_uint32, C.c_uint32, P, C.c_int64, P]
    L.shim_counts_b01.argtypes = [C.c_uint64, C.c_int64, C.c_int64, C.c_int64, P]
    L.shim_draws.argtypes = [C.c_uint64, P, P, P, C.c_uint32, P, C.c_int64, P]
    L.shim_scan_counts_word.argtypes = [C.c_uint64, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_uint32, P, C.c_int64]
    L.shim_scan_counts_word.restype = C.c_int64
    L.shim_u01_32.argtypes = [C.c_uint32]
    L.shim_u01_32.restype = C.c_double
    L.shim_u01_53.argtypes = [C.c_uint32, C.c_uint32]
    L.shim_u01_53.restype = C.c_double
    L.shim_poisson_cdf_u64.argtypes = [C.c_double, C.c_int, P, C.c_int]
    L.shim_poisson_alias_u64.argtypes = [P, C.c_int, P]
    L.shim_binomial_cdf4_u32.argtypes = [C.c_double, P]
    L.shim_plan_tables.argtypes = [C.POINTER(capi.VglParams), P, C.c_int, P, P, C.POINTER(C.c_int), C.POINTER(C.c_double)]
    L.shim_kernel_set.argtypes = [C.POINTER(capi.VglParams), C.c_int, C.POINTER(C.c_int)]
    L.shim_kernel_set.restype = C.c_char_p
    return L


def philox(L, ctr, k0, k1):
    c = np.ascontiguousarray(ctr, np.uint32).reshape(-1, 4)
    out = np.zeros_like(c)
    L.shim_philox(k0, k1, c.ctypes.data, len(c), out.ctypes.data)
    return out


def pois_cdf(L, lam):
    out = np.zeros(1024, np.uint64)
    n = L.shim_poisson_cdf_u64(lam, 1024, out.ctypes.data, 1024)
    return out[:n]


def pois_alias(L, cdf):
    cdf = np.ascontiguousarray(cdf, np.uint64)
    out = np.zeros(256, np.uint64)
    return out if L.shim_poisson_alias_u64(cdf.ctypes.data, len(cdf), out.ctypes.data) == 256 else None


def binom_cdf4(L, e):
    out = np.zeros(1024, np.uint32)
    L.shim_binomial_cdf4_u32(e, out.ctypes.data)
    return out.reshape(256, 4)


def plan_tables(L, argv, S, depths=None, qs_bins=None, fixed_depth=False):
    """alias rows [rows][256], each sample's row (--depths-file), qs class words [768], dominant class, P(minor class)"""
    a = vargs.parse_args(argv.split(), qs_bins=qs_bins, depths=depths)
    p = capi.params_from_args(a, S, max_batch_sites=1, n_slots=1, fixed_depth=fixed_depth)
    alias = np.zeros((max(S, 1), 256), np.uint64)
    rows = np.zeros(S, np.uint16)
    qcls = np.zeros(768, np.uint32)
    qd, qm = C.c_int(0), C.c_double(0.0)
    n = L.shim_plan_tables(C.byref(p), alias.ctypes.data, len(alias), rows.ctypes.data, qcls.ctypes.data, C.byref(qd), C.byref(qm))
    assert n >= 0
    return alias[:n], rows, qcls, qd.value, qm.value


def kernel_set(L, argv, S, depths=None):
    a = vargs.parse_args(argv.split(), depths=depths)
    p = capi.params_from_args(a, S, max_batch_sites=100, n_slots=1)
    rc = C.c_int(1)
    name = L.shim_kernel_set(C.byref(p), 1, C.byref(rc)).decode()
    assert rc.value == capi.VGL_OK
    return name


# ---- Philox4x32-10: the Random123 known-answer vectors (kat_vectors, philox4x32 10)
@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(laws_shim, ctr, key, want):
    assert tuple(int(x) for x in philox(laws_shim, ctr, *key)[0]) == want


def test_counts_blocks_follow_the_counter_layout(laws_shim):
    """block b of the P_COUNTS counter of (site, sample) = philox((site_lo, site_hi8, sample, 5 << 24 | b), seed_lo, seed_hi)"""
    seed, site0, S = (7 << 32) | 0x89ABCDEF, (0x5A << 32) | 0xFFFFFFF0, 5
    got = np.zeros((3 * S, 8), np.uint32)
    laws_shim.shim_counts_b01(seed, site0, 3, S, got.ctypes.data)
    for i in range(3 * S):
        site, sample = site0 + i // S, i % S
        for b in (0, 1):
            ctr = (site & 0xFFFFFFFF, (site >> 32) & 0xFF, sample, (5 << 24) | b)
            assert np.array_equal(got[i, 4 * b:4 * b + 4], philox(laws_shim, ctr, seed & 0xFFFFFFFF, seed >> 32)[0])


# ---- the depth law of the tile kernels' alias table
def induced_law(alias):
    """P(n = k) * 2^64 under the kernels' decode: column = top byte of the 64-bit uniform, kept when its low 56 bits are below
    t56 = entry >> 8, else the alias entry & 0xFF (the kernels compare frac56 << 8 with (entry & ~0xFF) in 64 bits)"""
    m = [0] * 256
    for col in range(256):
        e = int(alias[col])
        t56, al = e >> 8, e & 0xFF
        m[col] += t56
        m[al] += (1 << 56) - t56
    return m


def pmf_exact(lam, K):
    lam = mpmath.mpf(lam)
    return [mpmath.exp(-lam) * lam ** k / mpmath.factorial(k) for k in range(K)]


def largest_tile_mean(L):
    """the largest same-mean Poisson depth (to 1e-9) that k_tile_m1f takes: beyond it the law no longer fits 256 outcomes"""
    argv = "--seed 3 -d %r -e 0.01 -GL 1 -addPL 1 -addFormatAD 1"
    lo, hi = 100.0, 200.0
    assert kernel_set(L, argv % lo, 4) == "k_tile_m1f" and kernel_set(L, argv % hi, 4) != "k_tile_m1f"
    while hi - lo > 1e-9:
        mid = 0.5 * (lo + hi)
        if kernel_set(L, argv % mid, 4) == "k_tile_m1f":
            lo = mid
        else:
            hi = mid
    return lo, hi


def check_alias_law(alias, lam, bound=2.0 ** -56, tail_bound=2.0 ** -60):
    m = induced_law(alias)
    assert sum(m) == TWO64
    last = max(k for k in range(256) if m[k])
    pmf = pmf_exact(lam, 256)
    tail = 1 - mpmath.fsum(pmf[:last + 1])
    assert tail <= tail_bound, (lam, last, tail)
    dev = max(abs(mpmath.mpf(m[k]) / TWO64 - pmf[k]) for k in range(256))
    assert dev <= bound, (lam, dev)
    return float(dev), last, float(tail)


@pytest.mark.parametrize("lam", [1e-3, 0.5, 1.0, 2.0, 4.5, 10.0, 30.0, 80.0, "largest"])
def test_alias_table_induces_the_poisson_law(laws_shim, lam):
    # Near the cutoff (about 144) the long double sums of poisson_cdf_u64 carry an error of ~3e-17: its table can end while
    # ~2e-17 of mass lies beyond it, which the last entry takes.  There the bounds are 2^-54 for both.
    bound, tail_bound = 2.0 ** -56, 2.0 ** -60
    if lam == "largest":
        lam, _ = largest_tile_mean(laws_shim)
        bound = tail_bound = 2.0 ** -54
    alias = pois_alias(laws_shim, pois_cdf(laws_shim, lam))
    assert alias is not None
    dev, last, tail = check_alias_law(alias, lam, bound, tail_bound)
    print("lambda %.10g: max |P(k) - pmf(k)| = %.3g (bound %.3g), last outcome %d, tail %.3g (bound %.3g)"
          % (lam, dev, bound, last, tail, tail_bound))


def test_alias_tables_of_a_depths_file(laws_shim):
    """--depths-file: one alias row per distinct mean; every sample's row induces its own mean's law"""
    means = [0.5 + (i % 5) * 2.0 for i in range(37)] + [55.25, 0.5]
    S = len(means)
    alias, rows, _, _, _ = plan_tables(laws_shim, "--seed 3 -e 0.01 -GL 1 -addPL 1 -addFormatAD 1", S, depths=means)
    distinct = list(dict.fromkeys(means))
    assert len(alias) == len(distinct)
    checked = set()
    for s, m in enumerate(means):
        r = int(rows[s])
        assert r == distinct.index(m)
        if r not in checked:
            dev, _, _ = check_alias_law(alias[r], m)
            print("depths-file mean %g (row %d): max deviation %.3g" % (m, r, dev))
            checked.add(r)


# ---- the guide table of k_fused_m1f (fused.cu): guide[j] = first k whose CDF entry exceeds j << 56
def inversion(cdf, u):
    """the count-level sampler's Poisson draw: smallest k with u < cdf[k], at most len(cdf) - 1"""
    k = int(np.searchsorted(cdf, np.uint64(u), side="right"))
    return min(k, len(cdf) - 1)


@pytest.mark.parametrize("lam", [1e-3, 0.5, 1.0, 4.5, 10.0, 30.0, 80.0, 280.0, 600.0])
def test_fused_guide_is_a_lower_bound_of_the_inversion(laws_shim, lam):
    cdf = pois_cdf(laws_shim, lam)
    n = len(cdf)
    tight = 0
    for j in range(256):
        k = 0
        while k < n - 1 and int(cdf[k]) <= (j << 56):
            k += 1
        # the inversion is non-decreasing in u: its least value over top byte j is at u = j << 56
        lo = inversion(cdf, j << 56)
        assert k <= lo, (lam, j, k, lo)
        tight += k == lo
        # and the guided walk (counts_sampler.cuh) ends at the inversion's answer at both ends of the byte
        for u in (j << 56, ((j + 1) << 56) - 1):
            g = k
            while g < n - 1 and u >= int(cdf[g]):
                g += 1
            assert g == inversion(cdf, u)
    print("lambda %g: %d CDF entries, guide equal to the inversion at the low end of %d of 256 top bytes" % (lam, n, tight))


# ---- the error-count thresholds
@pytest.mark.parametrize("e", [1e-6, 1e-3, 0.01, 0.02, 0.05, 0.25, 0.5])
def test_binomial_thresholds_are_floors_of_the_exact_cdf(laws_shim, e):
    t = binom_cdf4(laws_shim, e)
    E = mpmath.mpf(e)
    two32 = mpmath.mpf(2) ** 32
    worst = mpmath.mpf(0)
    for n in range(256):
        cdf = mpmath.mpf(0)
        for j in range(4):
            if j <= n:
                cdf += mpmath.binomial(n, j) * E ** j * (1 - E) ** (n - j)
            sc = cdf * two32 if j <= n else two32
            want = int(mpmath.floor(sc))
            want = 0xFFFFFFFF if want >= 0xFFFFFFFF else want
            assert int(t[n, j]) == want, (e, n, j, int(t[n, j]), want, sc)
            if want < 0xFFFFFFFF:
                worst = max(worst, sc - want)
    print("e %g: every threshold is floor(P(E <= j | n) * 2^32); largest fractional part dropped %.6f" % (e, float(worst)))


# ---- the uniform maps
def test_uniform_maps_stay_inside_the_open_interval(laws_shim):
    L = laws_shim
    for w in (0, 1, 0x7FFFFFFF, 0xFFFFFFFE, 0xFFFFFFFF):
        u = L.shim_u01_32(w)
        assert 0.0 < u < 1.0 and u == (w + 0.5) * 2.0 ** -32
    top = L.shim_u01_53(0xFFFFFFFF, 0xFFFFFFFF)
    assert 0.0 < L.shim_u01_53(0, 0) < top < 1.0
    assert top == 1.0 - 2.0 ** -53
    # every other word keeps its value: ((v + 0.5) rounded to double) * 2^-53
    rng = np.random.default_rng(5)
    words = [(0, 0), (0xFFFFFFFF, 0xFFFFF7FF), (0xFFFFFFFF, 0xFFFFF000), (0xFFFFFFFE, 0xFFFFFFFF)] + \
        [tuple(int(x) for x in rng.integers(0, 1 << 32, 2)) for _ in range(1000)]
    for hi, lo in words:
        v = (hi << 21) ^ (lo >> 11)
        if v == (1 << 53) - 1:
            continue
        want = (float(v) + 0.5) * 1.1102230246251565e-16
        assert want < 1.0 and L.shim_u01_53(hi, lo) == want, (hi, lo)
