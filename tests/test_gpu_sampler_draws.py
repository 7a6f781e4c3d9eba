"""The count-level samplers' draws on the device against their exact quantile maps, cell by cell.

Every draw is a pure function of (seed, site, sample).  The CPU restates from each cell's Philox words (tables shim) and the host
tables what the cell must draw -- its depth, its number of mis-called reads E, its haplotype split and the placement of its
errors -- and the device's draws must match:
- integer paths exactly: the alias decode of the depth, the threshold comparisons of E, the haplotype popcounts (blocks 2+ for
  heterozygous cells deeper than 64 reads), the placement of errors (with the model-2 re-draws of occupied positions), the
  model-2 minor quality-class count and classes;
- floating-point walks (binom_inversion, the float CDF walk of sample_counts and of k_tile_m2 under --error-qs 1): E must be the
  exact quantile of Binomial(n, e) at the uniform the kernel consumed, taken as its exact grid value.  The one exception is a
  uniform within EPS of a CDF step (n * 2^-22 for the float walks, n * 2^-44 for the double ones); such cells are counted.
Rare branches are reached by steering: the CPU scans site ids for cells that take them and submits those sites as one-site
batches.  Each case also checks one unsteered batch of at least 2 M cells in full.
"""
import mpmath
import numpy as np
import pytest
from scipy import stats

from test_sampler_laws import binom_cdf4, laws_shim, plan_tables, pois_cdf  # noqa: F401  (laws_shim: the shim fixture)
from vcfgl_b200 import args as vargs
from vcfgl_b200 import capi

pytestmark = pytest.mark.gpu
P_READ, P_QS, P_COUNTS = 1, 3, 5
RTA3 = [(0, 2, 2), (3, 14, 12), (15, 30, 23), (31, 63, 37)]
MIN_BRANCH = 16
S = 1000
UNSTEERED_SITES = 2048                  # x 1000 samples: the full batch of each case
UF_TOP = 0xFFFFFF00                     # b0.z >> 8 == 0xFFFFFF: the 24-bit uniform rounds to 1.0f

CASES = {
    # name: argv, kernel set, sampler model, steered branches
    "m1f_d10": ("--seed 101 -d 10 -e 0.02 -GL 1 -addPL 1 -addFormatAD 1", "k_tile_m1f", "m1f", ["z_beyond_table", "E>3"]),
    "m1f_d80": ("--seed 102 -d 80 -e 0.02 -GL 1 -addPL 1 -addFormatAD 1", "k_tile_m1f", "m1f", ["het_n>64", "z_beyond_table", "E>3"]),
    "m1f_depths_file": ("--seed 103 -e 0.05 -GL 1 -addPL 1 -addFormatAD 1", "k_tile_m1f", "m1f", ["z_beyond_table", "E>3"]),
    "m1f_fixed": ("--seed 104 -d 70 -e 0.05 -GL 1 -addPL 1 -addFormatAD 1", "k_tile_m1f", "m1f", ["het_n>64", "z_beyond_table", "E>3"]),
    "m2_eq0": ("--seed 105 -d 50 -e 0.05 -GL 2 -addPL 1 -addFormatAD 1", "k_tile_m2", "m2", ["n>64", "redraw", "z_beyond_table", "E>3"]),
    "m2_eq1_cfg3i": ("--seed 42 -d 10 -e 0.01 -GL 2 -eq 1 -bv 1e-5 -addGL 1 -addPL 1", "k_tile_m2", "m2",
                     ["uf_top", "uf_exact", "E>3", "redraw"]),
    "m2_eq2_rta3": ("--seed 107 -d 10 -e 0.01 -GL 2 -eq 2 -bv 1e-5 -addGL 1 -addPL 1", "k_tile_m2", "m2",
                    ["z_beyond_table", "E>3", "redraw", "minor_qs"]),
    "fused_eq1": ("--seed 108 -d 10 -e 0.02 -eq 1 -bv 1e-4 -GL 1 -doUnobserved 3 -addPL 1 -addFormatAD 1", "k_fused_m1f", "fused",
                  ["uf_top", "uf_exact", "E>3"]),
}
DF_MEANS = [0.5 + (i % 7) * 9.0 for i in range(S)]


def case_args(name, argv):
    a = vargs.parse_args(argv.split(), qs_bins=RTA3 if "rta3" in name else None,
                         depths=DF_MEANS if "depths_file" in name else None)
    return a, "fixed" in name


def genotypes(site, mixed):
    """the genotype row of a site, a function of its id: hom-only rows (E is observable), or mixed rows with 2% missing"""
    rng = np.random.default_rng([site & 0xFFFFFFFF, site >> 32, int(mixed)])
    g0 = rng.integers(0, 4, S)
    if not mixed:
        return (g0 | (g0 << 4)).astype(np.uint8)
    g1 = np.where(rng.random(S) < 0.5, g0, rng.integers(0, 4, S))
    gt = (g0 | (g1 << 4)).astype(np.uint8)
    gt[rng.random(S) < 0.02] = 0xFF
    return gt


def popcount(x):
    x = np.asarray(x, np.uint64)
    return np.array([bin(int(v)).count("1") for v in x], np.int64) if x.size < 64 else \
        np.unpackbits(x.view(np.uint8).reshape(-1, 8), axis=1).sum(axis=1).astype(np.int64)


def low_bits(k):
    k = np.clip(np.asarray(k, np.int64), 0, 32)
    return ((np.uint64(1) << k.astype(np.uint64)) - np.uint64(1)).astype(np.uint64)


def mulhi(a, b):
    return (np.asarray(a, np.uint64) * np.asarray(b, np.uint64)) >> np.uint64(32)


class Draws:
    """Philox words of cells, through the shim"""

    def __init__(self, L, seed):
        self.L, self.seed = L, seed

    def b01(self, site0, n_sites):
        out = np.zeros((n_sites * S, 8), np.uint32)
        self.L.shim_counts_b01(self.seed, site0, n_sites, S, out.ctypes.data)
        return out.astype(np.uint64)

    def blocks(self, site, sample, purpose, block, read=None):
        n = len(site)
        site = np.ascontiguousarray(site, np.int64)
        sample = np.ascontiguousarray(sample, np.uint32)
        block = np.ascontiguousarray(np.broadcast_to(block, (n,)), np.uint32)
        read = np.ascontiguousarray(np.zeros(n) if read is None else np.broadcast_to(read, (n,)), np.uint32)
        out = np.zeros((n, 4), np.uint32)
        if n:
            self.L.shim_draws(self.seed, site.ctypes.data, sample.ctypes.data, read.ctypes.data, purpose, block.ctypes.data, n,
                              out.ctypes.data)
        return out.astype(np.uint64)

    def word(self, site, sample, purpose, ptr):
        """word `ptr` of the stream of blocks 0, 1, ... (ptr = 4 * block + word)"""
        ptr = np.asarray(ptr, np.int64)
        b = self.blocks(site, sample, purpose, ptr // 4)
        return b[np.arange(len(ptr)), ptr % 4]


# ---- the exact quantile of Binomial(n, e)
def quantile(n, e, u, eps):
    """smallest k with u <= F(k), and whether u lies within eps of a CDF step (then k or k + 1 are both accepted).  F in double
    (scipy) decides where u is further than 1e-9 from every step; the rest is decided in 40-digit arithmetic."""
    n = np.asarray(n, np.int64)
    k = np.zeros(len(n), np.int64)
    if not len(n):
        return k, np.zeros(0, bool)
    F = stats.binom.cdf(0, n, e)
    active = u > F
    while active.any():
        k[active] += 1
        F = np.where(active, stats.binom.cdf(k, n, e), F)
        active = active & (u > F) & (k < n)
    F_lo = np.where(k > 0, stats.binom.cdf(k - 1, n, e), 0.0)
    margin = np.minimum(np.abs(u - F), np.where(k > 0, np.abs(u - F_lo), 1.0))
    near = margin < eps
    for i in np.nonzero(~near & (margin < 1e-9))[0]:
        uu = mpmath.mpf(float(u[i])) if not isinstance(u, list) else u[i]
        E = mpmath.mpf(float(np.broadcast_to(e, n.shape)[i]))
        cdf, kk = mpmath.mpf(0), 0
        while True:
            cdf += mpmath.binomial(int(n[i]), kk) * E ** kk * (1 - E) ** (int(n[i]) - kk)
            if uu <= cdf or kk == n[i]:
                break
            kk += 1
        k[i] = kk
    return k, near


# ---- the samplers, restated
def alias_depth(b, alias, rows, sample):
    col = (b[:, 0] >> np.uint64(24)).astype(np.int64)
    frac56 = ((b[:, 0] & np.uint64(0xFFFFFF)) << np.uint64(32)) | b[:, 1]
    ent = alias[rows[sample].astype(np.int64) if rows is not None else 0, col] if alias.ndim == 2 else alias[col]
    return np.where(frac56 < (ent >> np.uint64(8)), col, (ent & np.uint64(0xFF)).astype(np.int64))


def table_E(z, cdf4, n, e, eps_n):
    """E of the threshold tables, exact inversion at u01_32(z) beyond the last one"""
    c = cdf4[np.minimum(n, 255)].astype(np.uint64)
    E = (z >= c[:, 0]).astype(np.int64) + (z >= c[:, 1]) + (z >= c[:, 2])
    inv = z >= c[:, 3]
    near = np.zeros(len(z), bool)
    if inv.any():
        u = (z[inv].astype(np.float64) + 0.5) * 2.0 ** -32
        E[inv], near[inv] = quantile(n[inv], e, u, n[inv] * eps_n)
    return E, inv, near


def walk_E(z, n, e, flt):
    """--error-qs 1 under k_tile_m2: the float CDF walk on the 24-bit grid (flt), exact inversion at u01_32(z) where e > 1/2 or
    where the walk ends with its float CDF still below uf (at the top of the walk; the 24-bit uniform of the top word is 1.0f).
    Returns E, whether the cell is near a step, and where uf > 0.998f the exact inversion's E and nearness as an alternative
    (-1 elsewhere): which of the two such a cell takes depends on the last bits of the device's exp2f."""
    ufi = (z >> np.uint64(8)).astype(np.float64)
    uf32 = (ufi.astype(np.float32) + np.float32(0.5)) * np.float32(5.9604645e-08)
    top = (uf32 > np.float32(0.998)) & flt
    u_grid, u_32 = (ufi + 0.5) * 2.0 ** -24, (z.astype(np.float64) + 0.5) * 2.0 ** -32
    E, near = quantile(n, e, np.where(flt, u_grid, u_32), np.where(flt, n * 2.0 ** -22, n * 2.0 ** -44))
    alt, near_alt = np.full(len(n), -1, np.int64), np.zeros(len(n), bool)
    if top.any():
        alt[top], near_alt[top] = quantile(n[top], e[top], u_32[top], n[top] * 2.0 ** -44)
    return E, uf32 > np.float32(0.998), near, alt, near_alt


class Case:
    def __init__(self, L, name, entry):
        self.name = name
        argv, self.kernels, self.model, self.branches = entry
        self.a, self.fixed = case_args(name, argv)
        self.mixed_ok = True
        self.draws = Draws(L, self.a.seed)
        alias, rows, qcls, q_dom, q_minor = plan_tables(L, argv, S, depths=self.a.depths, qs_bins=self.a.qs_bins, fixed_depth=self.fixed)
        self.alias, self.rows = alias, (rows if self.a.depths else None)
        self.qcls, self.q_dom, self.q_minor = qcls, q_dom, q_minor
        self.cdf4 = binom_cdf4(L, self.a.error_rate)
        self.qm_cdf4 = binom_cdf4(L, q_minor) if self.a.error_qs == 2 else None
        self.pois = pois_cdf(L, self.a.depth) if self.model == "fused" else None
        self.site_e = {}

    # -- expected draws of the cells of the sites [site0, site0 + n_sites) with genotype rows gts; dev: the device's draws
    def expect(self, site0, n_sites, gts, dev=None):
        N = n_sites * S
        site = site0 + np.repeat(np.arange(n_sites, dtype=np.int64), S)
        sample = np.tile(np.arange(S, dtype=np.int64), n_sites)
        gt = gts.reshape(-1).astype(np.int64)
        b = self.draws.b01(site0, n_sites)
        g0, g1 = gt & 3, (gt >> 4) & 3
        miss = (gt & 0x88) != 0
        het = (g0 != g1) & ~miss
        if self.model == "fused":
            u64 = (b[:, 0] << np.uint64(32)) | b[:, 1]
            n = np.minimum(np.searchsorted(self.pois, u64, side="right"), len(self.pois) - 1).astype(np.int64)
        elif self.fixed:
            n = np.full(N, int(self.a.depth), np.int64)
        else:
            n = alias_depth(b, self.alias, self.rows, sample)
        n[miss] = 0
        z = b[:, 2]
        if self.a.error_qs == 1:
            e = np.repeat([self.site_e[s] for s in range(site0, site0 + n_sites)], S)
        else:
            e = np.full(N, self.a.error_rate)
        x = dict(site=site, sample=sample, g0=g0, g1=g1, het=het, n=n, e=e, b=b, miss=miss, E_alt=np.full(N, -1, np.int64),
                 near_alt=np.zeros(N, bool))
        flags = {}
        if self.model == "m1f":
            E, inv, near = table_E(z, self.cdf4, n, self.a.error_rate, 2.0 ** -44)
            flags["z_beyond_table"] = inv & (n > 0)
        elif self.model == "m2":
            if self.a.error_qs == 1:
                flt = (e > 0) & (e <= 0.5) & ((1.0 - e).astype(np.float32) != np.float32(1.0))
                E, exact, near, alt, near_alt = walk_E(z, n, e, flt)
                E[n > 64] = 0
                x.update(E_alt=alt, near_alt=near_alt)
                flags["uf_top"] = (z >= UF_TOP) & (n > 0) & (n <= 64)
                flags["uf_exact"] = exact & (n > 0) & (n <= 64)
            else:
                E, inv, near = table_E(z, self.cdf4, n, self.a.error_rate, 2.0 ** -44)
                flags["z_beyond_table"] = inv & (n > 0) & (n <= 64)
            flags["n>64"] = n > 64
            E[n > 64] = 0
        else:
            E = np.zeros(N, np.int64)
            near = np.zeros(N, bool)
            l2ok = (e > 0) & (e <= 0.5) & ((1.0 - e).astype(np.float32) != np.float32(1.0))
            ufi = (z >> np.uint64(8)).astype(np.float64)
            uf32 = (ufi.astype(np.float32) + np.float32(0.5)) * np.float32(5.9604645e-08)
            top = (uf32 > np.float32(0.998)) & (n > 0)
            ptr = np.full(N, 4, np.int64)  # the cell's stream: block 1 word 0 on
            if top.any():
                w2 = self.draws.word(site[top], sample[top], P_COUNTS, ptr[top])
                ptr[top] += 1
                u = [(mpmath.mpf(int(zz)) * 2 ** 32 + int(ww) + mpmath.mpf(0.5)) / mpmath.mpf(2) ** 64 for zz, ww in zip(z[top], w2)]
                uf = np.array([float(v) for v in u])
                E[top], near[top] = quantile(n[top], e[top], uf, n[top] * 2.0 ** -44)
            rest = ~top & (n > 0) & (e > 0)
            uu = np.where(l2ok, (ufi + 0.5) * 2.0 ** -24, (z.astype(np.float64) + 0.5) * 2.0 ** -32)
            E[rest], near[rest] = quantile(n[rest], e[rest], uu[rest], np.where(l2ok, n * 2.0 ** -22, n * 2.0 ** -44)[rest])
            flags["uf_top"] = (z >= UF_TOP) & (n > 0)
            flags["uf_exact"] = top
            x["ptr"] = ptr
        flags["E>3"] = E > 3
        flags["het_n>64"] = het & (n > 64)
        x.update(E=E, near=near)
        # the device's E where it is observable decides near-step cells; elsewhere they are left out of the full comparison
        x["E_dev"] = None
        return x, flags

    # -- the read counts (m1f, fused) of every cell given E
    def counts(self, x, E):
        N = len(E)
        n, g0, g1, het, b = x["n"], x["g0"], x["g1"], x["het"], x["b"]
        site, sample = x["site"], x["sample"]
        cnt = np.zeros((N, 4), np.int64)
        if self.model == "m1f":
            kh = popcount(b[:, 3] & low_bits(np.minimum(n, 32))) + popcount(b[:, 4] & low_bits(n - 32))
            deep = np.nonzero(het & (n > 64))[0]
            t = 0
            while len(deep):
                left = n[deep] - 64 - 32 * t
                deep = deep[left > 0]
                left = left[left > 0]
                if not len(deep):
                    break
                w = self.draws.word(site[deep], sample[deep], P_COUNTS, np.full(len(deep), 8 + t))
                kh[deep] += popcount(w & low_bits(np.minimum(left, 32)))
                t += 1
        else:  # sample_counts: binom_half over b0.w, then the stream
            ptr = x["ptr"].copy()
            kh = popcount(b[:, 3] & low_bits(np.minimum(n, 32)))
            more = np.nonzero(het & (n > 32))[0]
            left = n[more] - 32
            while len(more):
                w = self.draws.word(site[more], sample[more], P_COUNTS, ptr[more])
                ptr[more] += 1
                kh[more] += popcount(w & low_bits(np.minimum(left, 32)))
                left -= 32
                keep = left > 0
                more, left = more[keep], left[keep]
        k0 = np.where(het, kh, n)
        cnt[np.arange(N), g0] += k0
        cnt[np.arange(N), g1] += n - k0
        rem0, rem = k0.copy(), np.maximum(n, 1)
        for j in range(int(E.max(initial=0))):
            act = np.nonzero(E > j)[0]
            if self.model == "m1f":
                r = b[act, 5 + j] if j < 3 else self.draws.word(site[act], sample[act], P_COUNTS, np.full(len(act), 40 + j - 3))
                q = mulhi(r, 3 * rem[act]).astype(np.int64)
                which, woff = q // 3, q % 3
                from0 = which < rem0[act]
            else:
                r = self.draws.word(site[act], sample[act], P_COUNTS, ptr[act])
                r2 = self.draws.word(site[act], sample[act], P_COUNTS, ptr[act] + 1)
                ptr[act] += 2
                from0 = mulhi(r, rem[act]).astype(np.int64) < rem0[act]
                woff = mulhi(r2, 3).astype(np.int64)
            truth = np.where(from0, g0[act], g1[act])
            rem0[act] -= from0
            rem[act] -= 1
            wrong = (truth + 1 + woff) & 3
            cnt[act, truth] -= 1
            cnt[act, wrong] += 1
        return cnt

    # -- the read sequences (m2) of every cell of at most 64 reads given E; deep cells per read
    def sequences(self, x, E):
        N = len(E)
        n, g0, g1, het, b = x["n"], x["g0"], x["g1"], x["het"], x["b"]
        site, sample = x["site"], x["sample"]
        h = (b[:, 4] << np.uint64(32)) | b[:, 3]
        bits = ((h[:, None] >> np.arange(64, dtype=np.uint64)[None, :]) & np.uint64(1)).astype(bool)
        seq = np.where(bits & het[:, None], g0[:, None], np.where(het[:, None], g1[:, None], g0[:, None])).astype(np.int64)
        orig = seq.copy()
        hit = np.zeros((N, 64), bool)
        ptr = np.full(N, 40, np.int64)
        redraws = np.zeros(N, np.int64)
        for j in range(int(E.max(initial=0))):
            act = np.nonzero(E > j)[0]
            r = b[act, 5 + j] if j < 3 else self.draws.word(site[act], sample[act], P_COUNTS, ptr[act])
            if j >= 3:
                ptr[act] += 1
            pend = np.arange(len(act))
            pos = np.zeros(len(act), np.int64)
            woff = np.zeros(len(act), np.int64)
            while len(pend):
                c = act[pend]
                q = mulhi(r[pend], 3 * n[c]).astype(np.int64)
                pos[pend], woff[pend] = q // 3, q % 3
                busy = hit[c, pos[pend]]
                redraws[c[busy]] += 1
                pend = pend[busy]
                if len(pend):
                    c = act[pend]
                    r[pend] = self.draws.word(site[c], sample[c], P_COUNTS, ptr[c])
                    ptr[c] += 1
            hit[act, pos] = True
            seq[act, pos] = (orig[act, pos] + 1 + woff) & 3
        return seq, orig, redraws

    def deep_reads(self, x, i_cells):
        """cells deeper than 64 reads: one P_READ block per read"""
        out = {}
        for c in i_cells:
            nn = int(x["n"][c])
            w = self.draws.blocks(np.full(nn, x["site"][c]), np.full(nn, x["sample"][c]), P_READ, 0, read=np.arange(nn))
            truth = np.where((w[:, 1] >> np.uint64(31)) != 0, x["g1"][c], x["g0"][c])
            err = (w[:, 0].astype(np.float64) + 0.5) * 2.3283064365386963e-10 < x["e"][c]
            out[c] = np.where(err, (truth + 1 + mulhi(w[:, 2], 3).astype(np.int64)) & 3, truth)
        return out

    def qs_reads(self, x):
        """--error-qs 2, cells of 1..64 reads: the dominant class's score, then M minor reads (position with re-draws, class) from
        the cell's P_QS stream; returns the scores [cells][64] and M"""
        info = self.qcls[256:512].astype(np.int64)
        n, site, sample = x["n"], x["site"], x["sample"]
        N = len(n)
        cells = (n > 0) & (n <= 64)
        u = self.draws.word(site, sample, P_QS, np.zeros(N, np.int64))
        t = self.qm_cdf4[np.minimum(n, 255)].astype(np.uint64)
        M = (u >= t[:, 0]).astype(np.int64) + (u >= t[:, 1]) + (u >= t[:, 2])
        inv = cells & (u >= t[:, 3])
        if inv.any():
            M[inv], _ = quantile(n[inv], self.q_minor, (u[inv].astype(np.float64) + 0.5) * 2.0 ** -32, n[inv] * 2.0 ** -44)
        M[~cells] = 0
        q = np.full((N, 64), info[self.q_dom] & 0xFF, np.int64)
        hit = np.zeros((N, 64), bool)
        ptr = np.ones(N, np.int64)
        for j in range(int(M.max(initial=0))):
            act = np.nonzero(M > j)[0]
            pend = np.arange(len(act))
            pos = np.zeros(len(act), np.int64)
            while len(pend):
                c = act[pend]
                pos[pend] = mulhi(self.draws.word(site[c], sample[c], P_QS, ptr[c]), n[c]).astype(np.int64)
                ptr[c] += 1
                pend = pend[hit[c, pos[pend]]]
            r = self.draws.word(site[act], sample[act], P_QS, ptr[act])
            ptr[act] += 1
            col = (r >> np.uint64(24)).astype(np.int64)
            en = self.qcls[512 + col].astype(np.uint64)
            cls = np.where((r & np.uint64(0xFFFFFF)) < (en >> np.uint64(8)), col, (en & np.uint64(0xFF)).astype(np.int64))
            hit[act, pos] = True
            q[act, pos] = info[cls] & 0xFF
        return q, M


def run_case(L, name, entry, only_sites=None):
    """checks the case's steered and unsteered batches, or only the one-site batches of `only_sites` (homozygous rows)"""
    case = Case(L, name, entry)
    a = case.a
    ctx = capi.Context(capi.params_from_args(a, S, max_batch_sites=UNSTEERED_SITES, n_slots=1, fixed_depth=case.fixed))
    assert ctx.native_kernels() == case.kernels, ctx.native_kernels()
    e_ctx = None
    if a.error_qs == 1 and case.model == "fused":  # the site's e: the same P_SITE draw, exported by the model-2 kernel's draws
        ea = vargs.parse_args(entry[0].replace("-GL 1", "-GL 2").replace("-doUnobserved 3", "").split())
        e_ctx = capi.Context(capi.params_from_args(ea, S, max_batch_sites=UNSTEERED_SITES, n_slots=1))
        assert e_ctx.native_kernels() == "k_tile_m2"

    def device(site0, n_sites, gts):
        ctx.input_buffer(0)[:n_sites] = gts
        rp = None if case.model == "fused" else ctx.native_draws(0, site0, n_sites)
        if a.error_qs == 1:
            erp = rp
            if e_ctx is not None:
                e_ctx.input_buffer(0)[:n_sites] = 0  # A/A everywhere: every site has reads
                erp = e_ctx.native_draws(0, site0, n_sites)
            ep, off = erp["error_probs"], erp["read_offsets"]
            for sl in range(n_sites):
                lo, hi = off[sl * S], off[(sl + 1) * S]
                assert hi > lo, "no read at site %d" % (site0 + sl)
                assert np.all(ep[lo:hi] == ep[lo]) and 0.0 < ep[lo] < 1.0
                case.site_e[site0 + sl] = float(ep[lo])
        if case.model == "fused":
            ctx.submit(0, site0, n_sites)
            bt = ctx.wait(0)
            cnt = np.zeros((n_sites * S, 4), np.int64)
            for sl in range(n_sites):
                o = bt.site(sl)
                A = o["n_alleles"]
                ad = o["fmt_ad"].reshape(S, A)
                for al in range(A):
                    base = int(o["alleles2acgt"][al])
                    if 0 <= base < 4:
                        cnt[sl * S:(sl + 1) * S, base] = ad[:, al]
            return dict(depths=bt.dp.copy(), counts=cnt)
        return rp

    seen = {k: 0 for k in case.branches}
    tot = dict(cells=0, near=0, near_skipped=0)

    def check(site0, n_sites, mixed):
        gts = np.stack([genotypes(s, mixed) for s in range(site0, site0 + n_sites)])
        d = device(site0, n_sites, gts)
        for k in range(0, n_sites, 64):  # the model in parts of 64 sites
            m = min(64, n_sites - k)
            check_part(site0 + k, m, gts[k:k + m], cell_range(d, k * S, (k + m) * S))

    def cell_range(d, c0, c1):
        if "counts" in d:
            return dict(depths=d["depths"][c0:c1], counts=d["counts"][c0:c1])
        off = d["read_offsets"]
        lo, hi = off[c0], off[c1]
        r = dict(depths=d["depths"][c0:c1], read_offsets=off[c0:c1 + 1] - lo, bases=d["bases"][lo:hi])
        if d.get("qs") is not None:
            r["qs"] = d["qs"][lo:hi]
        return r

    def check_part(site0, n_sites, gts, d):
        x, flags = case.expect(site0, n_sites, gts)
        n, E, near = x["n"], x["E"].copy(), x["near"]
        where = "%s sites %d..%d" % (name, site0, site0 + n_sites - 1)
        bad = np.nonzero(d["depths"] != n)[0]
        assert not len(bad), "%s: depth of cell %d: device %d, exact %d" % (where, bad[0], d["depths"][bad[0]], n[bad[0]])
        keep = np.ones(len(n), bool)
        if case.model in ("m1f", "fused"):
            cnt_dev = d["counts"] if case.model == "fused" else None
            if cnt_dev is None:
                off = d["read_offsets"]
                cell = np.repeat(np.arange(len(n)), np.diff(off))
                cnt_dev = np.zeros((len(n), 4), np.int64)
                np.add.at(cnt_dev, (cell, d["bases"].astype(np.int64)), 1)
            hom = ~x["het"] & ~x["miss"]
            E_dev = n - cnt_dev[np.arange(len(n)), x["g0"]]
            # E: where the device's E is observable (homozygous cells) it must be the exact quantile, or a neighbour at a step
            badE = hom & (E_dev != E) & ~(near & (np.abs(E_dev - E) <= 1))
            i = np.nonzero(badE)[0]
            assert not len(i), "%s: cell %d (n %d, e %r, z %#x): device E %d, exact quantile %d" % (
                where, i[0], n[i[0]], x["e"][i[0]], int(x["b"][i[0], 2]), E_dev[i[0]], E[i[0]])
            E = np.where(hom, E_dev, E)
            keep = ~(near & ~hom)
            want = case.counts(x, E)
            bad = np.nonzero(keep & np.any(want != cnt_dev, axis=1))[0]
            assert not len(bad), "%s: cell %d (gt %#x, n %d, E %d): device counts %s, exact %s" % (
                where, bad[0], int(x["g0"][bad[0]] | x["g1"][bad[0]] << 4), n[bad[0]], E[bad[0]], cnt_dev[bad[0]], want[bad[0]])
        else:
            off = d["read_offsets"]
            bases = d["bases"].astype(np.int64)
            small = np.nonzero((n > 0) & (n <= 64))[0]
            dev_seq = np.zeros((len(n), 64), np.int64)
            for c in small:
                dev_seq[c, :n[c]] = bases[off[c]:off[c] + n[c]]
            # the device's E: its reads that differ from the haplotype sequence
            seq0, orig, _ = case.sequences(x, np.zeros(len(n), np.int64))
            mask = np.arange(64)[None, :] < n[:, None]
            E_dev = np.where(n <= 64, ((dev_seq != orig) & mask).sum(axis=1), 0)
            alt, near_alt = x["E_alt"], x["near_alt"]
            badE = (n <= 64) & (E_dev != E) & ~(near & (np.abs(E_dev - E) <= 1)) & \
                (E_dev != alt) & ~(near_alt & (np.abs(E_dev - alt) <= 1))
            i = np.nonzero(badE)[0]
            assert not len(i), "%s: cell %d (n %d, e %r, b0.z %#x): device E %d, exact quantile %d" % (
                where, i[0], n[i[0]], x["e"][i[0]], int(x["b"][i[0], 2]), E_dev[i[0]], E[i[0]])
            E = E_dev
            seq, _, redraws = case.sequences(x, E)
            flags["redraw"] = redraws > 0
            bad = np.nonzero(np.any((seq != dev_seq) & mask, axis=1) & (n <= 64))[0]
            assert not len(bad), "%s: cell %d (n %d, E %d): device reads %s, exact %s" % (
                where, bad[0], n[bad[0]], E[bad[0]], dev_seq[bad[0], :n[bad[0]]], seq[bad[0], :n[bad[0]]])
            deep = np.nonzero(n > 64)[0]
            for c, want in case.deep_reads(x, deep).items():
                assert np.array_equal(bases[off[c]:off[c] + n[c]], want), "%s: deep cell %d" % (where, c)
            if a.error_qs == 2:
                qs = d["qs"].astype(np.int64)
                want, M = case.qs_reads(x)
                flags["minor_qs"] = M > 0
                dev_q = np.zeros((len(n), 64), np.int64)
                for c in small:
                    dev_q[c, :n[c]] = qs[off[c]:off[c] + n[c]]
                bad = np.nonzero(np.any((want != dev_q) & mask, axis=1) & (n <= 64))[0]
                assert not len(bad), "%s: cell %d (n %d, M %d): device qs %s, exact %s" % (
                    where, bad[0], n[bad[0]], M[bad[0]], dev_q[bad[0], :n[bad[0]]], want[bad[0], :n[bad[0]]])
        tot["cells"] += len(n)
        tot["near"] += int(near.sum())
        tot["near_skipped"] += int((~keep).sum())
        for k in seen:
            seen[k] += int(flags[k].sum())

    if only_sites is not None:
        for s in only_sites:
            check(s, 1, False)
        ctx.close()
        return
    # steered one-site batches: scan site ids on the CPU for cells that take each rare branch
    rng_base = 1 << 33
    for br in case.branches:
        mixed = br in ("het_n>64", "redraw", "n>64") or case.model == "m2"
        found, site = 0, rng_base + 10 ** 7 * (case.branches.index(br) + 1)
        while seen[br] < MIN_BRANCH:
            if br == "uf_top":  # 2^-24 per cell: scan in C for some sample's b0.z >> 8 == 0xFFFFFF
                hits = np.zeros(4, np.int64)
                k = L.shim_scan_counts_word(a.seed, site, 200000, S, 2, UF_TOP, hits.ctypes.data, 4)
                cand = [int(s) for s in hits[:min(k, 4)]]
                site = (cand[-1] + 1) if k >= 4 else site + 200000
            else:
                cand = []
                while not cand:
                    chunk = 64
                    gts = np.stack([genotypes(s, mixed) for s in range(site, site + chunk)])
                    if a.error_qs == 1:
                        for s in range(site, site + chunk):
                            case.site_e.setdefault(s, a.error_rate)  # scan with the mean rate; the batch uses the site's own
                    x, flags = case.expect(site, chunk, gts) if br != "redraw" else (None, None)
                    if br == "redraw":
                        x, _ = case.expect(site, chunk, gts)
                        f = case.sequences(x, x["E"])[2] > 0
                    elif br == "minor_qs":
                        b = case.draws.blocks(x["site"], x["sample"], P_QS, 0)
                        t = case.qm_cdf4[np.minimum(x["n"], 255)]
                        f = (b[:, 0] >= t[:, 0]) & (x["n"] > 0) & (x["n"] <= 64)
                    else:
                        f = flags[br]
                    cells = np.nonzero(f)[0]
                    cand = sorted(set(int(site + c // S) for c in cells))[:8]
                    if a.error_qs == 1:
                        for s in range(site, site + chunk):
                            case.site_e.pop(s, None)
                    site += chunk
            for s in cand:
                check(s, 1, mixed)
            found += len(cand)
    # one unsteered batch in full, homozygous rows (E observable) for the E branches, mixed rows for the rest
    check(rng_base, UNSTEERED_SITES, case.model == "m2")
    if case.model != "m2":
        check(rng_base + UNSTEERED_SITES, UNSTEERED_SITES, True)
    ctx.close()
    if e_ctx is not None:
        e_ctx.close()
    print("%s (%s): %d cells checked; per steered branch %s; %d cells within EPS of a CDF step (%d of them left out of the full "
          "comparison)" % (name, case.kernels, tot["cells"], seen, tot["near"], tot["near_skipped"]))
    for k, v in seen.items():
        assert v >= MIN_BRANCH, (name, k, v)


@pytest.mark.parametrize("name", sorted(CASES))
def test_device_draws_follow_the_exact_quantile_maps(laws_shim, name):  # noqa: F811
    run_case(laws_shim, name, CASES[name])


# ---- the threshold comparisons at their boundaries.  A word equal to a threshold has probability 2^-32 per cell, so no batch
# meets one by chance: instead the error rate is chosen so that threshold j of the cell's depth equals the cell's own word.
EDGE_ARGV = {"k_tile_m1f": ("m1f", "--seed 111 -d 10 -e %r -GL 1 -addPL 1 -addFormatAD 1"),
             "k_tile_m2": ("m2", "--seed 112 -d 10 -e %r -GL 2 -addPL 1 -addFormatAD 1")}
EDGE_P = {0: (0.80, 0.85), 1: (0.975, 0.99), 2: (0.9985, 0.9995)}  # P(E <= j | 10) for e about 0.01 .. 0.02


@pytest.mark.parametrize("kernels", sorted(EDGE_ARGV))
@pytest.mark.parametrize("j", sorted(EDGE_P))
def test_error_count_threshold_equal_to_the_word(laws_shim, kernels, j):  # noqa: F811
    """fixed depth 10: sample 0 of a site whose b0.z lies where P(E <= j | 10) does for e near 0.01; e is bisected until
    binomial_cdf4_u32(e)[10][j] == b0.z.  The table says E > j there (E counts the thresholds u >= t); the device must agree."""
    model, argv = EDGE_ARGV[kernels]
    seed = int(argv.split()[1])
    draws = Draws(laws_shim, seed)
    lo_p, hi_p = EDGE_P[j]
    site = 3 << 32
    while True:
        z = int(draws.b01(site, 1)[0, 2])
        if lo_p * 2 ** 32 <= z <= hi_p * 2 ** 32:
            lo, hi = 1e-4, 0.2  # threshold j of depth 10 falls from above z to below it across [lo, hi]
            t = lambda e: int(binom_cdf4(laws_shim, e)[10, j])  # noqa: E731
            assert t(lo) > z > t(hi)
            e = None
            while e is None:
                mid = 0.5 * (lo + hi)
                if mid in (lo, hi):
                    break  # no double puts the threshold on this word: next site
                tm = t(mid)
                if tm == z:
                    e = mid
                elif tm > z:
                    lo = mid
                else:
                    hi = mid
            if e is not None:
                break
        site += 1
    print("%s: site %d, b0.z = %#x = threshold %d of depth 10 at e = %r" % (kernels, site, z, j, e))
    name = "edge_fixed_%s_%d" % (model, j)
    run_case(laws_shim, name, (argv % e, kernels, model, []), only_sites=[site])
