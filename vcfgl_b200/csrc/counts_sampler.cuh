// Count-level cell sampler (VGL_SAMPLER_COUNTS).
//
// For GL model 1 with one quality score for all reads, every output of a cell (AD/ADF/ADR, GL, PL,
// QS, I16 counts) depends on the reads only through per-base (x strand) COUNTS, and the reference's
// reads within a cell are exchangeable (iid haplotype pick, iid error, iid strand; vcfgl.cpp:469-610).
// So instead of one Philox block per read we draw the counts directly:
//   n        ~ Poisson(lambda)                    table inversion of a 64-bit uniform (or generic sampler)
//   E        ~ Binomial(n, e)                     number of mis-called reads, CDF inversion
//   k0       ~ Binomial(n, 1/2)                   reads from haplotype 0 = popcount of n random bits
//   each error: which haplotype it hits (sequential hypergeometric), wrong base uniform over the other 3
//   fwd[b]   ~ Binomial(c_b, 1/2)                 forward-strand reads per observed base
// which is the same joint distribution of counts as the per-read simulation (checked by the same
// chi-square tests against the reference, tests/test_gpu_native.py).
#pragma once
#include "cell_source.cuh"

namespace vgl {

struct CellCounts {
    int n;        // depth
    uint64_t ad;  // 4 x u16 reads per observed base
    uint64_t fwd; // 4 x u16 forward reads per observed base (0 if the strand is not sampled)
};

// smallest k with u < cdf[k]; cdf is non-decreasing u64 fixed point, cdf[m-1] = 2^64-1
__device__ __forceinline__ int cdf_search(const unsigned long long* cdf, int m, unsigned long long u)
{
    int lo = 0, hi = m - 1;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (u < cdf[mid]) hi = mid; else lo = mid + 1;
    }
    return lo;
}

// Binomial(n, 1/2) from random bits
__device__ __forceinline__ int binom_half(int n, uint32_t first_word, Stream& st)
{
    int k = 0, left = n;
    uint32_t w = first_word;
    for (;;) {
        if (left >= 32) { k += __popc(w); left -= 32; }
        else { k += __popc(w & ((1u << left) - 1u)); left = 0; }
        if (left == 0) break;
        w = st.next();
    }
    return k;
}

// Binomial(n, e) by CDF inversion, non-decreasing in u (callers combine it with threshold tables of the same CDF for the
// first few outcomes); u in (0,1).  For e > 1/2 the walk runs over the mirrored law from the other end (n - K', K' ~
// Binomial(n, 1 - e) at 1 - u), which keeps the map monotone and the starting term away from underflow.
__device__ __forceinline__ int binom_inversion(int n, double e, double u)
{
    if (e <= 0.0) return 0;
    const bool flip = e > 0.5;
    const double pe = flip ? 1.0 - e : e;
    const double uu = flip ? 1.0 - u : u;
    const double ratio = pe / (1.0 - pe);
    double p = exp2((double)n * log2(1.0 - pe)), cdf = p;
    int k = 0;
    while (uu > cdf && k < n) {
        p *= (double)(n - k) / (double)(k + 1) * ratio;
        cdf += p;
        ++k;
    }
    return flip ? n - k : k;
}

struct CountsParams {
    Key key;
    int depth_mode;
    double depth_mean;
    const double* depth_means;
    const unsigned long long* pois_cdf; // shared memory
    const unsigned short* pois_guide;    // shared memory: [256] lower bound of the answer by the top byte of u
    int pois_n;
    int sample_strand;
    float l2_1me_fast;  // log2(1-e) when e <= 0.5 and p0 does not underflow in float (fast path), else 0
};

// e: base-picking error probability of the site; l2 = log2(1 - e) (float), er = e / (1 - e) (float)
__device__ __forceinline__ CellCounts sample_counts(const CountsParams& cp, int64_t site, uint32_t sample, uint8_t gt,
                                                    double e, float l2, float er)
{
    CellCounts out;
    out.n = 0;
    out.ad = out.fwd = 0;
    const int g0 = gt & 0xF, g1 = gt >> 4;
    if (g0 == VGL_GT_MISSING || g1 == VGL_GT_MISSING) return out; // depth is drawn but discarded (vcfgl.cpp:371-379)
    const u32x4 w = draw(cp.key, site, sample, 0, P_COUNTS, 0);
    Stream st; // further words, only touched by cells that need them
    st.init(cp.key, site, sample, 0, P_COUNTS);
    st.block = 1;
    int n;
    if (cp.depth_mode == VGL_DEPTH_POISSON) {
        // guided inversion: the top byte of u gives a lower bound, then a short linear walk (exact to 2^-64)
        const unsigned long long u = ((unsigned long long)w.x << 32) | w.y;
        n = cp.pois_guide[w.x >> 24];
        while (n < cp.pois_n - 1 && u >= cp.pois_cdf[n]) ++n;
    } else if (cp.depth_mode == VGL_DEPTH_FIXED) {
        n = (int)cp.depth_mean;
    } else {
        Stream sd;
        sd.init(cp.key, site, sample, 0, P_DEPTH);
        n = poisson(sd, cp.depth_means[sample]);
    }
    if (n > 65535) n = 65535;
    out.n = n;
    if (n == 0) return out;
    // number of mis-called reads
    int E = 0;
    if (e > 0.0) {
        const float p0 = exp2f((float)n * l2);
        const float uf = ((float)(w.z >> 8) + 0.5f) * 5.9604645e-08f; // 24-bit uniform in (0,1]: the top word rounds to 1.0f
        if (uf > 0.998f) {
            // the upper tail: a float CDF saturates at 1.0f and a 24-bit uniform cannot fall into events rarer than 6e-8 per cell
            // (five errors in ten reads at e = 0.01) -- exact inversion in double with 64 random bits
            const double u = ((double)w.z + ((double)st.next() + 0.5) * 2.3283064365386963e-10) * 2.3283064365386963e-10;
            E = binom_inversion(n, e, u);
        } else if (l2 != 0.0f && p0 > 1e-30f) {
            // fast path: float CDF walk (e <= 0.5, no underflow); P(E=0) = p0 ends most cells here
            float p = p0, cdf = p0;
            while (uf > cdf && E < n) {
                p *= (float)(n - E) / (float)(E + 1) * er;
                cdf += p;
                ++E;
            }
        } else {
            E = binom_inversion(n, e, u01_32(w.z));
        }
    }
    // haplotype split
    const int k0 = (g0 == g1) ? n : binom_half(n, w.w, st);
    uint64_t ad = ((uint64_t)k0 << (16 * g0)) + ((uint64_t)(n - k0) << (16 * g1));
    // place the errors: each hits haplotype 0's reads w.p. rem0/rem (without replacement)
    int rem0 = k0, rem = n;
    for (int i = 0; i < E; ++i) {
        const uint32_t r = st.next();
        const bool from0 = mulhi32(r, (uint32_t)rem) < (uint32_t)rem0;
        const int truth = from0 ? g0 : g1;
        rem0 -= from0;
        --rem;
        const int wrong = (truth + 1 + (int)mulhi32(st.next(), 3u)) & 3;
        ad -= 1ull << (16 * truth);
        ad += 1ull << (16 * wrong);
    }
    out.ad = ad;
    if (cp.sample_strand) {
        uint64_t fwd = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int c = (int)((ad >> (16 * b)) & 0xFFFF);
            if (c) fwd |= (uint64_t)binom_half(c, st.next(), st) << (16 * b);
        }
        out.fwd = fwd;
    }
    return out;
}

// which 255 of a deep cell's reads errmod keeps (htslib/errmod.c:156-159), at count level: an urn draw
__device__ __forceinline__ uint64_t subsample_counts_255(const CountsParams& cp, int64_t site, uint32_t sample, uint64_t ad, int n)
{
    Stream st;
    st.init(cp.key, site, sample, 0, P_SUBSAMPLE);
    int c[4], k[4] = {0, 0, 0, 0};
#pragma unroll
    for (int b = 0; b < 4; ++b) c[b] = (int)((ad >> (16 * b)) & 0xFFFF);
    int rem = n;
    for (int i = 0; i < 255; ++i) {
        int r = (int)mulhi32(st.next(), (uint32_t)rem);
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const bool hit = r >= 0 && r < c[b];
            if (hit) { --c[b]; ++k[b]; r = -1; }
            else if (r >= 0) r -= c[b];
        }
        --rem;
    }
    return (uint64_t)k[0] | ((uint64_t)k[1] << 16) | ((uint64_t)k[2] << 32) | ((uint64_t)k[3] << 48);
}

} // namespace vgl
