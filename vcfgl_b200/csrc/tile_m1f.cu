// k_tile_m1f -- the headline path in one kernel, built for a low instruction count per cell:
// native RNG, GL model 1 with one run-constant quality score and error rate (--error-qs 0),
// same-mean Poisson or fixed depth (<= 255 reads per cell), no strand / GP / QS / I16 tags.
// Everything else runs through k_fused_m1f (fused.cu) or the unfused kernels (kernels.cu).
//
// Persistent CTAs pull TILES of whole sites from an atomic ticket.  A tile is a run of "virtual
// cells": every site occupies S4 = ceil4(S) slots, so that any run of 32 slots starts at a sample
// index that is a multiple of 4 -> its span in every [S][G] / [S][A] output block starts and ends
// on a 16-byte boundary (blocks themselves are padded to 16 B).
//   phase A  thread per cell: two Philox blocks -> depth (alias table), number of mis-called reads
//            (threshold table), haplotype split (popcount), error placement -> four 8-bit base
//            counts kept in shared memory; FORMAT/DP written
//   phase A2 warp per site (or site part): per-site base totals from the count cache (IDP.4A + REDUX)
//   phase B  thread per site: allele order, unobserved allele, skip code, INFO tags
//            (vcfgl.cpp:396-404, 665-782); decoupled look-back gives the tile's base offsets
//   phase C  warp per 32 cells: errmod scores from the counts (m1f.cuh), GL / PL (packed fp32x2 math)
//            and AD scattered into the warp's own shared-memory slice in allele order, then ONE bulk
//            async copy (cp.async.bulk shared -> global) per plane writes the 16-byte aligned span.
// HBM traffic = 1 B/cell in, the tag planes out.
#include "tile_common.cuh"

namespace vgl {

// BIG variant: words of a CTA's global row = counts [S4] | AUX chunk masks [S4 / 32 + 1][8]
__host__ __device__ inline size_t tile_m1f_row_words(int S4) { return (size_t)S4 + (size_t)8 * (S4 / 32 + 1); }

// One cell of the count-level sampler: returns the four 8-bit base counts (A | C << 8 | G << 16 | T << 24).
// Draws (same counter layout as draw() in philox.cuh, purpose P_COUNTS): block 0 = {x,y: depth; z: number of
// errors; w: haplotype bits 0..31}, block 1 = {x: haplotype bits 32..63; y,z,w: placement of errors 1..3};
// rarer needs (depth > 64, > 3 errors) continue with later blocks of the same (site, sample) counter.
struct TileRng {
    uint32_t s_alias;    // shared address: [256] (t56 << 8 | alias) as {lo, hi}
    uint32_t s_cdf_e;    // shared address: [256] uint4 P(E <= j | n) * 2^32, j = 0..3
    int fixed_depth;     // >= 0: every cell has this depth; < 0: Poisson via the alias table
    bool has_err;
};

// one mis-called read: read j of the `rem` left is hit; it belongs to haplotype 0 w.p. rem0/rem; the wrong base
// is uniform over the other three
__device__ __forceinline__ uint32_t tile_place_error(uint32_t ad, uint32_t r, int g0, int g1, int& rem0, int& rem)
{
    const uint32_t j = mulhi32(r, 3u * (uint32_t)rem);
    const uint32_t which = (j * 0xAAABu) >> 17; // j / 3 for j < 2^15 (rem <= 255)
    const uint32_t woff = j - 3u * which;
    const bool from0 = (int)which < rem0;
    const int truth = from0 ? g0 : g1;
    rem0 -= from0;
    --rem;
    const int wrong = (truth + 1 + (int)woff) & 3;
    return ad + (1u << (8 * wrong)) - (1u << (8 * truth));
}

__device__ __forceinline__ uint32_t tile_sample_cell(const DevParams& p, const TileRng& R, unsigned long long site, uint32_t sample, uint32_t gt)
{
    const int g0 = gt & 0x3, g1 = (gt >> 4) & 0x3;
    const uint32_t c0 = (uint32_t)site, c1 = (uint32_t)(site >> 32) & 0xFFu;
    const u32x4 b0 = philox_rk(p, c0, c1, sample, (uint32_t)P_COUNTS << 24);
    const u32x4 b1 = philox_rk(p, c0, c1, sample, ((uint32_t)P_COUNTS << 24) | 1u);
    int n;
    if (R.fixed_depth >= 0) {
        n = R.fixed_depth;
    } else { // Walker alias over 256 columns, 64-bit uniform: column = top byte, 56 bits against the column's threshold
        const uint32_t col = b0.x >> 24;
        uint2 en;
        if (p.alias_row) en = __ldg(reinterpret_cast<const uint2*>(p.pois_alias) + (size_t)__ldg(p.alias_row + min(sample, (uint32_t)p.S - 1u)) * 256u + col); // the sample's own mean (padding lanes: any row, their depth is dropped)
        else en = lds64(R.s_alias + col * 8u);
        const unsigned long long frac = ((unsigned long long)__funnelshift_l(b0.y, b0.x, 8) << 32) | (b0.y << 8);
        const unsigned long long thr = ((unsigned long long)en.y << 32) | (en.x & 0xFFFFFF00u);
        n = frac < thr ? (int)col : (int)(en.x & 0xFFu);
    }
    if (gt & 0x88u) n = 0; // a missing allele (0xF; valid alleles are 0..3): depth is drawn but discarded (vcfgl.cpp:371-379)
    const bool het = ((gt ^ (gt >> 4)) & 0x3u) != 0u;
    // haplotype split: reads from haplotype 0 = popcount of the first n random bits
    const int kh = __popc(b0.w & low_bits(min(n, 32))) + __popc(b1.x & low_bits(min(max(n - 32, 0), 32)));
    int k0 = het ? kh : n;
    int E = 0;
    bool rare = het && n > 64;
    if (R.has_err) { // number of mis-called reads: two thresholds decide 0 / 1 / 2, more is rare
        const uint4 c = lds128(R.s_cdf_e + (uint32_t)n * 16u);
        E = (b0.z >= c.x) + (b0.z >= c.y);
        rare = rare || b0.z >= c.z;
    }
    if (rare) {
        Key key;
        key.k0 = p.k0; key.k1 = p.k1;
        if (het && n > 64) {
            Stream st;
            st.init(key, (int64_t)site, sample, 0, P_COUNTS);
            st.block = 2;
            for (int left = n - 64; left > 0; left -= 32) k0 += __popc(st.next() & low_bits(min(left, 32)));
        }
        if (R.has_err) {
            const uint4 c = lds128(R.s_cdf_e + (uint32_t)n * 16u);
            if (b0.z >= c.z) E = b0.z >= c.w ? binom_inversion(n, p.error_rate, u01_32(b0.z)) : 3; // beyond the table: exact inversion
        }
    }
    uint32_t ad = ((uint32_t)k0 << (8 * g0)) + ((uint32_t)(n - k0) << (8 * g1));
    int rem0 = k0, rem = max(n, 1);
    const uint32_t ad1 = tile_place_error(ad, b1.y, g0, g1, rem0, rem); // straight-line first error (nearly every warp has one)
    if (E > 0) ad = ad1;
    if (E > 1) {
        ad = tile_place_error(ad, b1.z, g0, g1, rem0, rem);
        if (E > 2) {
            ad = tile_place_error(ad, b1.w, g0, g1, rem0, rem);
            if (E > 3) {
                Key key;
                key.k0 = p.k0; key.k1 = p.k1;
                Stream st;
                st.init(key, (int64_t)site, sample, 0, P_COUNTS);
                st.block = 10;
                for (int i = 3; i < E; ++i) ad = tile_place_error(ad, st.next(), g0, g1, rem0, rem);
            }
        }
    }
    return ad;
}

// ---------------------------------------------------------------------------------------------------------------
// AUX variant (QS, I16, INFO/ADF, INFO/ADR): the extra per-cell draws of the count-level sampler.
//   strands        the reads of a cell are grouped A.., C.., G.., T..; read r is on the forward strand when bit r of the
//                  cell's P_STRAND stream is 1 (iid fair coins, vcfgl.cpp:581-586) -> forward reads per base = popcounts
//   tail distances read r draws 1 + U{0..49} capped at 25 (vcfgl.cpp:653-656) from digit r % 3 of word (r % 12) / 3 of
//                  block r / 12 of the cell's P_TAIL stream: j = floor(word * 125000 / 2^32), digits of j in base 50
//                  (relative bias of a value's probability <= 125000 / 2^32 = 2.9e-5)
//   last read      all tail distances of a site are credited to the base of the site's LAST simulated read (the stale
//                  r_base of vcfgl.cpp:647-663): a uniformly chosen read of the last cell that has reads (P_LAST)
// vgl_native_draws() (k_tile_m1f_draws below) lists the same draws read by read.
__device__ __forceinline__ uint32_t tile_word(const u32x4& b, int j) { return j == 0 ? b.x : (j == 1 ? b.y : (j == 2 ? b.z : b.w)); }

// forward reads per base as four packed bytes; nmax = largest depth in the warp (uniform)
__device__ __forceinline__ uint32_t tile_strand_counts(const DevParams& p, unsigned long long site, uint32_t sample, uint32_t c4, int nmax)
{
    const int e0 = (int)(c4 & 0xFFu), e1 = e0 + (int)((c4 >> 8) & 0xFFu), e2 = e1 + (int)((c4 >> 16) & 0xFFu), e3 = e2 + (int)(c4 >> 24);
    const uint32_t c0 = (uint32_t)site, c1 = (uint32_t)(site >> 32) & 0xFFu;
    uint32_t f0 = 0, f1 = 0, f2 = 0, f3 = 0;
    for (int kb = 0; kb * 128 < nmax; ++kb) {
        const u32x4 blk = philox_rk(p, c0, c1, sample, ((uint32_t)P_STRAND << 24) | (uint32_t)kb);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int base = kb * 128 + j * 32;
            if (base < nmax) {
                const uint32_t w = tile_word(blk, j);
                const uint32_t m0 = low_bits(min(max(e0 - base, 0), 32)), m1 = low_bits(min(max(e1 - base, 0), 32));
                const uint32_t m2 = low_bits(min(max(e2 - base, 0), 32)), m3 = low_bits(min(max(e3 - base, 0), 32));
                f0 += __popc(w & m0);
                f1 += __popc(w & (m1 ^ m0));
                f2 += __popc(w & (m2 ^ m1));
                f3 += __popc(w & (m3 ^ m2));
            }
        }
    }
    return f0 | (f1 << 8) | (f2 << 16) | (f3 << 24);
}

// the three tail distances of one 32-bit word
__device__ __forceinline__ void tile_tail3(uint32_t w, int& t0, int& t1, int& t2)
{
    const uint32_t j = mulhi32(w, 125000u);
    const uint32_t hi = j / 2500u, r = j - hi * 2500u, mid = r / 50u, lo = r - mid * 50u;
    t0 = min((int)lo + 1, 25);
    t1 = min((int)mid + 1, 25);
    t2 = min((int)hi + 1, 25);
}

// sum and sum of squares of the tail distances of a cell's n reads; nmax = largest depth in the warp (uniform)
__device__ __forceinline__ void tile_tail_sums(const DevParams& p, unsigned long long site, uint32_t sample, int n, int nmax, uint32_t& tsum,
                                               uint32_t& tsq)
{
    const uint32_t c0 = (uint32_t)site, c1 = (uint32_t)(site >> 32) & 0xFFu;
    tsum = tsq = 0u;
    for (int kb = 0; kb * 12 < nmax; ++kb) {
        const u32x4 blk = philox_rk(p, c0, c1, sample, ((uint32_t)P_TAIL << 24) | (uint32_t)kb);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = kb * 12 + j * 3;
            if (r >= nmax) break; // uniform: no cell of the warp has a read left for this word
            int t0, t1, t2;
            tile_tail3(tile_word(blk, j), t0, t1, t2);
            t0 = r < n ? t0 : 0;
            t1 = r + 1 < n ? t1 : 0;
            t2 = r + 2 < n ? t2 : 0;
            tsum += (uint32_t)(t0 + t1 + t2);
            tsq += (uint32_t)(t0 * t0 + t1 * t1 + t2 * t2);
        }
    }
}

// tail distance of read r of a cell (sequential fall-back and the draws export)
__device__ __forceinline__ int tile_tail_of_read(const DevParams& p, unsigned long long site, uint32_t sample, int r)
{
    const u32x4 blk = philox_rk(p, (uint32_t)site, (uint32_t)(site >> 32) & 0xFFu, sample, ((uint32_t)P_TAIL << 24) | (uint32_t)(r / 12));
    int t[3];
    tile_tail3(tile_word(blk, (r % 12) / 3), t[0], t[1], t[2]);
    return t[r % 3];
}

// index (in the grouped order A.., C.., G.., T..) of the read of cell (site, sample) that counts as the site's last read
__device__ __forceinline__ int tile_last_read(const DevParams& p, unsigned long long site, uint32_t sample, int n)
{
    const u32x4 blk = philox_rk(p, (uint32_t)site, (uint32_t)(site >> 32) & 0xFFu, sample, (uint32_t)P_LAST << 24);
    return (int)mulhi32(blk.x, (uint32_t)n);
}
__device__ __forceinline__ int tile_base_of_read(uint32_t c4, int j)
{
    const int e0 = (int)(c4 & 0xFFu), e1 = e0 + (int)((c4 >> 8) & 0xFFu), e2 = e1 + (int)((c4 >> 16) & 0xFFu);
    return j < e0 ? 0 : (j < e1 ? 1 : (j < e2 ? 2 : 3));
}

// v += c, k times, as the reference's float accumulator would (vcfgl.cpp:1009-1022)
__device__ __forceinline__ float tile_add_const_times(float v, int c, int k)
{
    const float cf = (float)c;
    if (v + (float)k * cf < 16777216.0f && v == truncf(v)) return v + (float)(k * c);
    for (int i = 0; i < k; ++i) v = __fadd_rn(v, cf);
    return v;
}

// acc + 1.0f, k times, as the reference's float accumulator would round it (vcfgl.cpp:845-898: a cell whose reads all show the
// base adds the term 1.0f).  Within a binade adding 1 is exact (acc sits on the binade's grid, ulp <= 1), so the run jumps
// to the last value below the next power of two in one exact step and takes only the crossing add through the rounder.
__device__ __forceinline__ float tile_add_ones(float acc, int k)
{
    while (k > 0) {
        if (acc < 1.0f || acc >= 8388608.0f) { // below 1 the grid is finer than the result's; above 2^23 every add may round
            acc = __fadd_rn(acc, 1.0f);
            --k;
            continue;
        }
        const float top = __uint_as_float((__float_as_uint(acc) & 0x7F800000u) + 0x00800000u); // next power of two above acc
        const float d = __fsub_rn(top, acc);                                                  // exact (Sterbenz)
        const int m = min(k, (int)ceilf(d) - 1);                                              // adds that stay below `top`
        acc = __fadd_rn(acc, (float)m);                                                       // exact: same binade, on the grid
        k -= m;
        if (k > 0) { acc = __fadd_rn(acc, 1.0f); --k; }                                       // the crossing add rounds like the reference's
    }
    return acc;
}

// I16 of one site when a float accumulator overflows its exact range (vcfgl.cpp:982-1074; deep sites with many samples): the
// sums are redone in the reference's order from the cached counts.  One thread, rare and slow, but exact.
template <bool BIG>
__device__ __noinline__ void tile_site_i16_seq(const DevParams& p, const TAux& ax, const unsigned long long site, const int S, const uint32_t s_cnt_site,
                                               const uint32_t* cnt_g, float* out)
{
    float v[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = 0.0f;
    const int A = (int)(ax.info & 0xFFu), n_obs = (int)((ax.info >> 8) & 0xFFu);
    int a2b[5] = {-1, -1, -1, -1, -1};
#pragma unroll
    for (int b = 0; b < 5; ++b) {
        const int a = (int)((ax.b2a >> (4 * b)) & 0xFu);
        if (a != 0xF) {
#pragma unroll
            for (int k = 0; k < 5; ++k)
                if (k == a) a2b[k] = b;
        }
    }
    const int refb = a2b[0];
    const int q = (p.adjust_qs & 2) ? p.pre_adj_qs : p.pre_qs, q2 = qs_squared(q), mq = p.i16_mapq, mq2 = mq * mq;
    auto cnt = [&](int s) -> uint32_t { return BIG ? cnt_g[s] : lds32(s_cnt_site + 4u * (uint32_t)s); };
    int stale = -1;
    if (ax.last >= 0) {
        const uint32_t c4 = cnt(ax.last);
        stale = tile_base_of_read(c4, tile_last_read(p, site, (uint32_t)ax.last, (int)__vsadu4(c4, 0u)));
    }
    float tsum = 0.0f, tsq = 0.0f;
    for (int s = 0; s < S; ++s) {
        const uint32_t c4 = cnt(s);
        const int n = (int)__vsadu4(c4, 0u);
        for (int i = 0; i < n; ++i) {
            const int t = tile_tail_of_read(p, site, (uint32_t)s, i);
            tsum = __fadd_rn(tsum, (float)t);
            tsq = __fadd_rn(tsq, (float)(t * t));
        }
        const int cr = (int)((c4 >> (8 * refb)) & 0xFFu);
        v[4] = __fadd_rn(v[4], (float)(q * cr));
        v[5] = __fadd_rn(v[5], (float)(q2 * cr));
        for (int a = 0; a < A; ++a) {
            if (a == n_obs) continue;
            const int b = a2b[a];
            if (b < 0 || b == 4) continue;
            const int k = (int)((c4 >> (8 * b)) & 0xFFu);
            if (a == 0) { v[8] = tile_add_const_times(v[8], mq, k); v[9] = tile_add_const_times(v[9], mq2, k); }
            else        { v[10] = tile_add_const_times(v[10], mq, k); v[11] = tile_add_const_times(v[11], mq2, k); }
        }
    }
    for (int a = 1; a < A; ++a) {
        if (a == n_obs) continue;
        const int b = a2b[a];
        if (b < 0 || b == 4) continue;
        for (int s = 0; s < S; ++s) {
            const int k = (int)((cnt(s) >> (8 * b)) & 0xFFu);
            v[6] = __fadd_rn(v[6], (float)(q * k));
            v[7] = __fadd_rn(v[7], (float)(q2 * k));
        }
    }
    v[0] = (float)ax.fw[refb];
    v[1] = (float)(ax.tot[refb] - ax.fw[refb]);
    v[12] = refb == stale ? tsum : 0.0f;
    v[13] = refb == stale ? tsq : 0.0f;
    for (int a = 1; a < A; ++a) {
        if (a == n_obs) continue;
        const int b = a2b[a];
        if (b < 0 || b == 4) continue;
        v[2] = __fadd_rn(v[2], (float)ax.fw[b]);
        v[3] = __fadd_rn(v[3], (float)(ax.tot[b] - ax.fw[b]));
        v[14] = __fadd_rn(v[14], b == stale ? tsum : 0.0f);
        v[15] = __fadd_rn(v[15], b == stale ? tsq : 0.0f);
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) out[i] = v[i];
}

// I16 of one site (vcfgl.cpp:982-1074) from the site totals.  Every accumulator of the reference is a float that adds small
// non-negative integers in (sample, read) order; while the total stays below 2^24 every partial sum is an exactly
// representable integer and the float equals the integer total.  Beyond that: tile_site_i16_seq.
template <bool BIG>
__device__ __forceinline__ void tile_site_i16(const DevParams& p, const TAux& ax, const unsigned long long site, const int S, const uint32_t s_cnt_site,
                                              const uint32_t* cnt_g, float* out)
{
    const int A = (int)(ax.info & 0xFFu), n_obs = (int)((ax.info >> 8) & 0xFFu);
    const int q = (p.adjust_qs & 2) ? p.pre_adj_qs : p.pre_qs, q2 = qs_squared(q), mq = p.i16_mapq, mq2 = mq * mq;
    // the site's last read (stale r_base)
    int stale = -1;
    if (ax.last >= 0) {
        const uint32_t c4 = BIG ? cnt_g[ax.last] : lds32(s_cnt_site + 4u * (uint32_t)ax.last);
        stale = tile_base_of_read(c4, tile_last_read(p, site, (uint32_t)ax.last, (int)__vsadu4(c4, 0u)));
    }
    int ref = 0, ref_fw = 0, nonref = 0, nonref_fw = 0;
    bool stale_ref = false, stale_nonref = false;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        const int a = (int)((ax.b2a >> (4 * b)) & 0xFu);
        if (a == 0) { ref = ax.tot[b]; ref_fw = ax.fw[b]; stale_ref = b == stale; }
        else if (a != 0xF && a < A && a != n_obs) { nonref += ax.tot[b]; nonref_fw += ax.fw[b]; stale_nonref = stale_nonref || b == stale; }
    }
    const long long qmax = max(max(q2, q), max(mq2, mq));
    if (!(qmax * (long long)max(ref, nonref) < 16777216ll && ax.tq < 16777216ull)) {
        tile_site_i16_seq<BIG>(p, ax, site, S, s_cnt_site, cnt_g, out);
        return;
    }
    const float tsum = (float)ax.ts, tsq = (float)ax.tq;
    out[0] = (float)ref_fw; out[1] = (float)(ref - ref_fw); out[2] = (float)nonref_fw; out[3] = (float)(nonref - nonref_fw);
    out[4] = (float)(q * ref); out[5] = (float)(q2 * ref); out[6] = (float)(q * nonref); out[7] = (float)(q2 * nonref);
    out[8] = (float)(mq * ref); out[9] = (float)(mq2 * ref); out[10] = (float)(mq * nonref); out[11] = (float)(mq2 * nonref);
    out[12] = stale_ref ? tsum : 0.0f; out[13] = stale_ref ? tsq : 0.0f;
    out[14] = stale_nonref ? tsum : 0.0f; out[15] = stale_nonref ? tsq : 0.0f;
}

// GL and the mantissa-encoded PL of one cell from its scores (gl_methods.cpp:338-357, vcfgl.cpp:907-939).  ALL15: every base
// pair is a genotype of the site.  With w = q/10 >= 0: GL = (-w) - max(-w) = min(w) - w, the same float as the reference's
// subtraction.
template <bool ALL15>
__device__ __forceinline__ void tile_cell_values(const float (&q)[15], const uint32_t (&off)[15], float (&g)[16], float (&u)[16])
{
    float w[16];
#pragma unroll
    for (int k = 0; k < 14; k += 2) unpack2(div10_fast2(pack2(q[k], q[k + 1])), w[k], w[k + 1]);
    w[14] = -neg_div10_fast(q[14]);
    float mn = CUDART_INF_F;
#pragma unroll
    for (int k = 0; k < 15; ++k) mn = fminf(mn, (ALL15 || off[k] != 0xFFu) ? w[k] : CUDART_INF_F);
    const f32x2 mn2 = pack2(mn, mn);
#pragma unroll
    for (int k = 0; k < 14; k += 2) {
        const f32x2 g2 = sub2(mn2, pack2(w[k], w[k + 1]));
        unpack2(g2, g[k], g[k + 1]);
        unpack2(pl_magic2(g2), u[k], u[k + 1]);
    }
    g[14] = __fsub_rn(mn, w[14]);
    u[14] = __fadd_rz(__fadd_rz(__fmul_rn(-10.0f, g[14]), 0.5f), 8388608.0f);
}

// ... scattered into the warp's stage slice in allele order
template <bool ALL15>
__device__ __forceinline__ void tile_emit_cell(const float (&q)[15], const uint4 slot, uint32_t cell_g, bool has_gl, bool has_pl)
{
    const uint32_t sw[4] = {slot.x, slot.y, slot.z, slot.w};
    uint32_t off[15];
#pragma unroll
    for (int k = 0; k < 15; ++k) off[k] = __byte_perm(sw[k >> 2], 0u, 0x4440u | (k & 3));
    float g[16], u[16];
    tile_cell_values<ALL15>(q, off, g, u);
#pragma unroll
    for (int k = 0; k < 15; ++k) {
        if (ALL15 || off[k] != 0xFFu) {
            const uint32_t dst = cell_g + off[k];
            if (has_gl) asm volatile("st.shared.f32 [%0], %1;" ::"r"(dst), "f"(g[k]) : "memory");
            if (has_pl) asm volatile("st.shared.b32 [%0+%2], %1;" ::"r"(dst), "r"(pl_from_magic_bits(u[k])), "n"(TILE_WST_G * 4) : "memory");
        }
    }
}

// ---- "pure" cells: every read shows the same base x.  The 15 scores then fall into three classes -- xx (score 0), the pairs
// that hold x once, the pairs without x -- and GL / PL are functions of the depth alone.  The table is built on the device by
// the scoring code itself (so it is bit-identical by construction) for every base and depth, and is only used when the
// classes really collapse for all four bases (`ok` stays 1).
__global__ void k_m1f_pure_table(const double* __restrict__ bsum, const double* __restrict__ het, M1Pure* __restrict__ out, int* ok)
{
    const int n = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (n > 255) return;
    M1Pure r;
    r.gl1 = r.gl0 = 0.0f;
    r.pl1 = r.pl0 = 0;
    bool good = true;
    if (n >= 1) {
        for (int x = 0; x < 4; ++x) {
            float q[15];
            m1f_scores_noclamp(n, x == 0 ? n : 0, x == 1 ? n : 0, x == 2 ? n : 0, x == 3 ? n : 0, bsum, het, q);
            uint32_t off[15];
#pragma unroll
            for (int k = 0; k < 15; ++k) off[k] = 0u;
            float g[16], u[16];
            tile_cell_values<true>(q, off, g, u);
            M1Pure c;
            c.gl1 = c.gl0 = 0.0f;
            c.pl1 = c.pl0 = 0;
            bool have1 = false, have0 = false;
#pragma unroll
            for (int k = 0; k < 5; ++k)
#pragma unroll
                for (int j = 0; j <= k; ++j) {
                    const int pair = k * (k + 1) / 2 + j, hits = (j == x) + (k == x);
                    const float gv = g[pair];
                    const int pv = pl_from_magic_bits(u[pair]);
                    if (hits == 2) good = good && __float_as_uint(gv) == 0u && pv == 0;
                    else if (hits == 1) {
                        if (!have1) { c.gl1 = gv; c.pl1 = pv; have1 = true; }
                        good = good && __float_as_uint(gv) == __float_as_uint(c.gl1) && pv == c.pl1;
                    } else {
                        if (!have0) { c.gl0 = gv; c.pl0 = pv; have0 = true; }
                        good = good && __float_as_uint(gv) == __float_as_uint(c.gl0) && pv == c.pl0;
                    }
                }
            if (x == 0) r = c;
            good = good && __float_as_uint(c.gl1) == __float_as_uint(r.gl1) && __float_as_uint(c.gl0) == __float_as_uint(r.gl0) &&
                   c.pl1 == r.pl1 && c.pl0 == r.pl0;
        }
    }
    out[n] = r;
    if (!good) atomicExch(ok, 0);
}

// builds the table into `out` ([256] M1Pure, device); returns 1 when pure cells may use it
int build_m1f_pure_table(const double* d_bsum, const double* d_het, void* out, cudaStream_t st)
{
    int* d_ok = nullptr;
    int ok = 1;
    if (cudaMalloc((void**)&d_ok, sizeof(int)) != cudaSuccess) return 0;
    cudaMemcpyAsync(d_ok, &ok, sizeof(int), cudaMemcpyHostToDevice, st);
    k_m1f_pure_table<<<2, 128, 0, st>>>(d_bsum, d_het, reinterpret_cast<M1Pure*>(out), d_ok);
    cudaMemcpyAsync(&ok, d_ok, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (cudaStreamSynchronize(st) != cudaSuccess) ok = 0;
    cudaFree(d_ok);
    return ok;
}

// GEN: any subset of the GL / PL / AD planes (else all three); BIG: a site's counts do not fit the shared-memory
// cache -> they pass through a per-CTA scratch row in global memory (L2-resident), read one chunk ahead;
// AUX: QS / I16 / INFO ADF, ADR (strand and tail-distance draws in phase A, per-site sums in an extra phase after B) and the
// further per-cell planes GP / FORMAT ADF, ADR (an extra pass per chunk in phase C)
// PURE: chunks whose cells all show a single base take the closed form (m1_pure table); compiled in only for runs where such
// chunks are the rule (low depth x error rate), because the extra branch costs the general path ~10 %
// XTRA (AUX only): GP / FORMAT ADF, ADR wanted
#ifndef TILE_MIN_CTAS_AUX
#define TILE_MIN_CTAS_AUX (TILE_MIN_CTAS - 1)
#endif
template <bool GEN, bool BIG, bool AUX, bool PURE, bool XTRA>
__global__ void __launch_bounds__(TILE_BLOCK, AUX ? TILE_MIN_CTAS_AUX : TILE_MIN_CTAS) k_tile_m1f(const __grid_constant__ DevParams p)
{
    extern __shared__ __align__(16) unsigned char tile_smem[];
    // layout: alias [256] u64 | cdf_e [256] uint4 | stage [warps][G plane, PL plane, R plane] | st [sites] | tot [sites][4] |
    //         aux [sites] (AUX only) | cnt [cap]
    constexpr int WST = 2 * TILE_WST_G + TILE_WST_R; // words per warp
    constexpr uint32_t OFF_STAGE = 2048 + 4096, OFF_ST = OFF_STAGE + TILE_WARPS * WST * 4, OFF_TOT = OFF_ST + TILE_MAX_SITES * sizeof(TSite),
                       OFF_AUX = OFF_TOT + TILE_MAX_SITES * 16, OFF_MSK = OFF_AUX + (AUX ? TILE_MAX_SITES * sizeof(TAux) : 0),
                       OFF_CNT = OFF_MSK + ((AUX && !BIG) ? (TILE_CELLS / 32) * 32 : 0);
    TSite* st = reinterpret_cast<TSite*>(tile_smem + OFF_ST);
    int* tot = reinterpret_cast<int*>(tile_smem + OFF_TOT);
    TAux* aux = reinterpret_cast<TAux*>(tile_smem + OFF_AUX);
    __shared__ int64_t s_base[4];
    __shared__ int s_next;
    __shared__ uint32_t s_ctr[2];
    __shared__ uint32_t s_zero[32];

    // thread ids and the sample count are pinned in registers (volatile moves cannot be rematerialised): ptxas
    // otherwise re-reads SR_TID / the constant bank inside the chunk loops and stalls on their latency
    int tid, S;
    asm volatile("mov.u32 %0, %%tid.x;" : "=r"(tid));
    asm volatile("mov.u32 %0, %1;" : "=r"(S) : "r"(p.S));
    const int lane = tid & 31, warp = tid >> 5;
    const int S4 = (S + 3) & ~3, PAD = S4 - S, T = p.sites_per_tile;
    const uint32_t s_smem = smem_u32(tile_smem);
    for (int i = tid; i < 256; i += TILE_BLOCK) {
        reinterpret_cast<uint2*>(tile_smem)[i] = reinterpret_cast<const uint2*>(p.pois_alias)[i];
        reinterpret_cast<uint4*>(tile_smem + 2048)[i] = reinterpret_cast<const uint4*>(p.err_cdf)[i];
    }
    for (int i = tid; i < TILE_MAX_SITES * 4; i += TILE_BLOCK) tot[i] = 0;
    if (AUX && tid < TILE_MAX_SITES) {
        TAux z;
        z.fw[0] = z.fw[1] = z.fw[2] = z.fw[3] = 0;
        z.ts = z.tq = 0ull;
        z.last = -1;
        z.tot[0] = z.tot[1] = z.tot[2] = z.tot[3] = 0;
        z.b2a = 0xFFFFFu; z.info = 0u; z._pad = 0;
        aux[tid] = z;
    }
    if (tid == 0) {
        s_next = (int)atomicAdd(p.ticket, 1u);
        s_ctr[0] = s_ctr[1] = 0u;
    }
    if (tid < 32) s_zero[tid] = 0u;
    TileRng R;
    R.s_alias = s_smem;
    R.s_cdf_e = s_smem + 2048;
    R.fixed_depth = p.depth_mode == VGL_DEPTH_FIXED ? (int)p.depth_mean : -1;
    R.has_err = p.error_rate > 0.0;
    // iv / S4 for iv < 2^16 (exact while iv * S4 < 2^32)
    const uint32_t inv_s4 = (uint32_t)(((1ull << 32) + S4 - 1) / S4);
    const bool explode = p.do_unobserved >= 3;
    const bool add_unobs = p.do_unobserved == 1 || p.do_unobserved == 2 || p.do_unobserved == 4 || p.do_unobserved == 5;
    // GEN: the plane tests are pinned in a register (the compiler would otherwise re-read the kernel parameters at every store)
    uint32_t plane_flags = (p.gl != nullptr ? 1u : 0u) | (p.pl != nullptr ? 2u : 0u) | (p.ad != nullptr ? 4u : 0u);
    asm volatile("mov.u32 %0, %0;" : "+r"(plane_flags));
    const bool has_gl = GEN ? (plane_flags & 1u) != 0u : true, has_pl = GEN ? (plane_flags & 2u) != 0u : true, has_ad = GEN ? (plane_flags & 4u) != 0u : true;
    const bool want_tail = AUX && (p.tag_mask & VGL_TAG_I16) != 0;
    // further per-cell planes of the AUX variant: 1 = GP, 2 = FORMAT ADF, 4 = FORMAT ADR (staged through the same slices after GL / PL / AD)
    uint32_t xflags = 0u;
    if (XTRA) {
        xflags = (p.gp != nullptr ? 1u : 0u) | (p.adf != nullptr ? 2u : 0u) | (p.adr != nullptr ? 4u : 0u);
        asm volatile("mov.u32 %0, %0;" : "+r"(xflags));
    }
    const bool stage_gl = XTRA ? (has_gl || (xflags & 1u)) : has_gl; // GP is made from the staged GL values
    const uint32_t s_wg = s_smem + OFF_STAGE + warp * WST * 4; // this warp's GL slice; PL at +TILE_WST_G words, AD at +2*TILE_WST_G
    const uint32_t s_wr = s_wg + 2 * TILE_WST_G * 4;
    const uint32_t s_cnt = s_smem + OFF_CNT, s_st = s_smem + OFF_ST;
    // BIG: per-CTA row in global memory = counts [S4], then (AUX) the chunk masks [S4 / 32 + 1][8]
    uint32_t* const cnt_g = BIG ? p.cnt_scratch + (size_t)blockIdx.x * tile_m1f_row_words(S4) : nullptr;
    uint32_t* const msk_g = BIG ? cnt_g + S4 : nullptr;
    const uint32_t s_msk = s_smem + OFF_MSK;
    uint32_t s_ctrA = smem_u32(&s_ctr[0]), s_ctrC = smem_u32(&s_ctr[1]);
    bool first_tile = true;

    for (;;) {
        __syncthreads(); // previous tile fully done (st / tot / cnt / chunk tickets); s_next published
        const int tile = s_next;
        if (tile >= p.n_tiles) break;
        if (first_tile) { // see tile_ticket_issue
            const uint32_t opaque_zero = lds32(smem_u32(&s_zero[lane])); // 0, but not provably the same in every lane
            s_ctrA += opaque_zero;
            s_ctrC += opaque_zero;
            first_tile = false;
        }
        const int site0 = tile * T;
        const int nsl = min(T, p.n_sites - site0);
        const int nv = nsl * S4;            // virtual cells
        const int nchunk = (nv + 31) >> 5;
        const int64_t cell0 = (int64_t)site0 * S;
        const uint8_t* __restrict__ gt_t = p.gt + cell0;
        int32_t* __restrict__ dp_t = p.dp + cell0;
        const unsigned long long site_base = (unsigned long long)(p.first_site + site0);

        // ---------------- phase A: sample, FORMAT/DP, per-site base totals.  The genotypes of a warp's next chunk
        // are loaded before the current chunk is processed.
        {
            int cur = tile_ticket_get(tile_ticket_issue(s_ctrA, lane));
            int nxt = tile_ticket_get(tile_ticket_issue(s_ctrA, lane));
            int iv = cur * 32 + lane;
            int sl = (int)__umulhi((uint32_t)iv, inv_s4), v = iv - sl * S4;
            bool real = iv < nv && v < S;
            uint32_t gt = 0xFFu;
            if (real) gt = gt_t[(uint32_t)(iv - sl * PAD)];
            while (cur < nchunk) {
                const int raw = tile_ticket_issue(s_ctrA, lane); // the chunk after next
                const int iv2 = nxt * 32 + lane;
                const int sl2 = (int)__umulhi((uint32_t)iv2, inv_s4), v2 = iv2 - sl2 * S4;
                const bool real2 = iv2 < nv && v2 < S;
                uint32_t gt2 = 0xFFu;
                if (real2) gt2 = gt_t[(uint32_t)(iv2 - sl2 * PAD)];
                const uint32_t ad = tile_sample_cell(p, R, site_base + (uint32_t)sl, (uint32_t)v, gt); // non-cells: missing genotype -> 0
                if (real) dp_t[(uint32_t)(iv - sl * PAD)] = (int)__vsadu4(ad, 0u); // sum of the four byte counts
                if (iv < nv) {
                    if (BIG) cnt_g[iv] = ad;
                    else sts32(s_cnt + (uint32_t)iv * 4u, ad);
                }
                // site totals: packed 16-bit fields through REDUX; a chunk usually lies within one site
                const int first = __shfl_sync(0xffffffffu, sl, 0);
                const uint32_t w01 = __byte_perm(ad, 0u, 0x4140), w23 = __byte_perm(ad, 0u, 0x4342);
                if (__all_sync(0xffffffffu, sl == first)) {
                    const uint32_t a01 = __reduce_add_sync(0xffffffffu, w01), a23 = __reduce_add_sync(0xffffffffu, w23);
                    if (lane < 4 && first < nsl) {
                        const uint32_t w = (lane & 2) ? a23 : a01;
                        const uint32_t val = (lane & 1) ? (w >> 16) : (w & 0xFFFFu);
                        if (val) atomicAdd(&tot[first * 4 + lane], (int)val);
                    }
                } else if (__all_sync(0xffffffffu, sl == first || sl == first + 1)) {
                    const bool in0 = sl == first;
                    const uint32_t a01 = __reduce_add_sync(0xffffffffu, in0 ? w01 : 0u), a23 = __reduce_add_sync(0xffffffffu, in0 ? w23 : 0u);
                    const uint32_t b01 = __reduce_add_sync(0xffffffffu, in0 ? 0u : w01), b23 = __reduce_add_sync(0xffffffffu, in0 ? 0u : w23);
                    if (lane < 8) {
                        const uint32_t w = (lane & 4) ? ((lane & 2) ? b23 : b01) : ((lane & 2) ? a23 : a01);
                        const uint32_t val = (lane & 1) ? (w >> 16) : (w & 0xFFFFu);
                        const int ts = first + (lane >> 2);
                        if (val && ts < nsl) atomicAdd(&tot[ts * 4 + (lane & 3)], (int)val);
                    }
                } else if (sl < nsl) { // tiny sites: a chunk spans many
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const int val = (int)((ad >> (8 * b)) & 0xFFu);
                        if (val) atomicAdd(&tot[sl * 4 + b], val);
                    }
                }
                if (AUX) { // per base: which cells of the chunk show only that base / that base among others (the QS terms 1 / fractional)
                    const int n_ = (int)__vsadu4(ad, 0u);
                    const uint32_t nz = __vcmpne4(ad, 0u), eqn = __vcmpeq4(ad, (uint32_t)n_ * 0x01010101u);
                    const uint32_t full = nz & eqn, frac = nz & ~eqn;
                    uint32_t mk[8];
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        mk[b] = __ballot_sync(0xffffffffu, (full >> (8 * b)) & 1u);
                        mk[4 + b] = __ballot_sync(0xffffffffu, (frac >> (8 * b)) & 1u);
                    }
                    if (lane < 8) {
                        uint32_t mine = mk[0];
#pragma unroll
                        for (int k = 1; k < 8; ++k) mine = lane == k ? mk[k] : mine;
                        if (BIG) msk_g[(size_t)cur * 8 + lane] = mine;
                        else sts32(s_msk + (uint32_t)cur * 32u + 4u * (uint32_t)lane, mine);
                    }
                }
                if (AUX) { // strand and tail-distance draws, summed per site
                    const int n = (int)__vsadu4(ad, 0u);
                    const int nmax = __reduce_max_sync(0xffffffffu, n);
                    const uint32_t fw4 = tile_strand_counts(p, site_base + (uint32_t)sl, (uint32_t)v, ad, nmax);
                    uint32_t tsum = 0u, tsq = 0u;
                    if (want_tail) tile_tail_sums(p, site_base + (uint32_t)sl, (uint32_t)v, n, nmax, tsum, tsq);
                    const int lastv = n > 0 ? v : -1;
                    const uint32_t f01 = __byte_perm(fw4, 0u, 0x4140), f23 = __byte_perm(fw4, 0u, 0x4342);
                    const bool one = __all_sync(0xffffffffu, sl == first), two = __all_sync(0xffffffffu, sl == first || sl == first + 1);
                    if (one || two) {
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            if (h == 1 && one) break;
                            const bool in = sl == first + h;
                            const uint32_t a01 = __reduce_add_sync(0xffffffffu, in ? f01 : 0u), a23 = __reduce_add_sync(0xffffffffu, in ? f23 : 0u);
                            const uint32_t ts = __reduce_add_sync(0xffffffffu, in ? tsum : 0u), tq = __reduce_add_sync(0xffffffffu, in ? tsq : 0u);
                            const int lm = __reduce_max_sync(0xffffffffu, in ? lastv : -1);
                            const int site_h = first + h;
                            if (site_h < nsl) {
                                if (lane < 4) {
                                    const uint32_t w = (lane & 2) ? a23 : a01;
                                    const uint32_t val = (lane & 1) ? (w >> 16) : (w & 0xFFFFu);
                                    if (val) atomicAdd(&aux[site_h].fw[lane], (int)val);
                                } else if (lane == 4) {
                                    if (ts) atomicAdd(&aux[site_h].ts, (unsigned long long)ts);
                                } else if (lane == 5) {
                                    if (tq) atomicAdd(&aux[site_h].tq, (unsigned long long)tq);
                                } else if (lane == 6) {
                                    if (lm >= 0) atomicMax(&aux[site_h].last, lm);
                                }
                            }
                        }
                    } else if (sl < nsl && n > 0) {
#pragma unroll
                        for (int b = 0; b < 4; ++b) {
                            const int val = (int)((fw4 >> (8 * b)) & 0xFFu);
                            if (val) atomicAdd(&aux[sl].fw[b], val);
                        }
                        if (tsum) atomicAdd(&aux[sl].ts, (unsigned long long)tsum);
                        if (tsq) atomicAdd(&aux[sl].tq, (unsigned long long)tsq);
                        atomicMax(&aux[sl].last, lastv);
                    }
                }
                cur = nxt; iv = iv2; sl = sl2; v = v2; real = real2; gt = gt2;
                nxt = tile_ticket_get(raw);
            }
        }
        __syncthreads();

        // ---------------- phase B (warp 0): per-site record (vcfgl.cpp:396-404, 665-782, 806-843 INFO part)
        if (warp == 0) {
            if (lane == 0) { // phase A is over for every warp: rearm its chunk tickets; next tile's ticket (tiles are independent)
                s_ctr[0] = 0u;
                s_next = (int)atomicAdd(p.ticket, 1u);
            }
            { // pull the next tile's genotypes into L2 while this tile is scored (its first loads would otherwise wait on DRAM)
                const int nt = __shfl_sync(0xffffffffu, lane == 0 ? s_next : 0, 0);
                const int64_t lo = (int64_t)nt * T * S + lane * 128;
                if (nt < p.n_tiles && lane * 128 < T * S && lo < p.n_cells) asm volatile("prefetch.global.L2 [%0];" ::"l"(p.gt + lo));
            }
            tile_phase_b(p, lane, nsl, site0, tile, S, T, tot, st, explode, add_unobs, s_base, s_ctr, AUX ? aux : nullptr);
        }
        __syncthreads();
        if (p.zero_holes) tile_zero_holes(p, tid, nsl, S, s_base);

        // ---------------- phase AUX: QS (thread per site and base; float sums in sample order, vcfgl.cpp:845-898) and
        // I16 (thread per site, vcfgl.cpp:982-1074) from the cached counts and the site totals
        if (AUX) {
            const int sl = tid >> 2, b = tid & 3;
            if (sl < nsl && (aux[sl].info >> 16)) {
                const uint32_t b2a_ = aux[sl].b2a;
                const uint32_t s_cnt_site = s_cnt + (uint32_t)(sl * S4) * 4u;
                vgl_site_out* const rec = p.sites + site0 + sl;
                const int a = (int)((b2a_ >> (4 * b)) & 0xFu);
                if ((p.tag_mask & VGL_TAG_QS) && a != 0xF) {
                    // QS[a] = sum over samples, in order, of (float)(q c_b) / (float)(q n) (vcfgl.cpp:845-898).  Cells without the
                    // base add +0 (identity), cells with nothing but the base add exactly 1 (tile_add_ones runs them in bulk);
                    // only the cells that mix the base with others take a division.  The chunk masks of phase A say which is which.
                    const int q = (p.adjust_qs & 2) ? p.pre_adj_qs : p.pre_qs;
                    float acc = 0.0f;
                    const int v_lo = sl * S4, v_hi = v_lo + S; // the site's virtual cells
                    for (int c = v_lo >> 5; c <= (v_hi - 1) >> 5; ++c) {
                        const int lo = max(v_lo - c * 32, 0), hi = min(v_hi - c * 32, 32);
                        const uint32_t range = low_bits(hi) & ~low_bits(lo);
                        uint32_t fullm = (BIG ? msk_g[(size_t)c * 8 + b] : lds32(s_msk + (uint32_t)c * 32u + 4u * (uint32_t)b)) & range;
                        uint32_t fracm = (BIG ? msk_g[(size_t)c * 8 + 4 + b] : lds32(s_msk + (uint32_t)c * 32u + 16u + 4u * (uint32_t)b)) & range;
                        while (fracm) {
                            const int pos = __ffs(fracm) - 1;
                            const uint32_t before = low_bits(pos);
                            acc = tile_add_ones(acc, __popc(fullm & before));
                            fullm &= ~before;
                            const int iv = c * 32 + pos;
                            const uint32_t c4 = BIG ? cnt_g[iv] : lds32(s_cnt + 4u * (uint32_t)iv);
                            const float sum = (float)(q * (int)__vsadu4(c4, 0u));
                            acc = __fadd_rn(acc, __fdiv_rn((float)(q * (int)((c4 >> (8 * b)) & 0xFFu)), sum));
                            fracm &= fracm - 1u;
                        }
                        acc = tile_add_ones(acc, __popc(fullm));
                    }
                    rec->qs[a] = acc;
                }
            }
            if ((p.tag_mask & VGL_TAG_I16) && tid < nsl && (aux[tid].info >> 16)) { // a thread per site (one warp)
                const TAux ax = aux[tid];
                tile_site_i16<BIG>(p, ax, site_base + (uint32_t)tid, S, s_cnt + (uint32_t)(tid * S4) * 4u, cnt_g, p.sites[site0 + tid].i16);
            }
            __syncthreads();
            if (tid < nsl) { // clear the phase-A accumulators for the next tile
                aux[tid].fw[0] = aux[tid].fw[1] = aux[tid].fw[2] = aux[tid].fw[3] = 0;
                aux[tid].ts = aux[tid].tq = 0ull;
                aux[tid].last = -1;
            }
        }

        // ---------------- phase C: score + emit, one warp per chunk of 32 virtual cells
        float* const gl_t = has_gl ? p.gl + s_base[0] : nullptr;
        int32_t* const pl_t = has_pl ? p.pl + s_base[0] : nullptr;
        int32_t* const ad_t = has_ad ? p.ad + s_base[1] : nullptr;
        float* const gp_t = (XTRA && (xflags & 1u)) ? p.gp + s_base[0] : nullptr;
        int32_t* const adf_t = (XTRA && (xflags & 2u)) ? p.adf + s_base[1] : nullptr;
        int32_t* const adr_t = (XTRA && (xflags & 4u)) ? p.adr + s_base[1] : nullptr;
        const uint4* const pure_tab = reinterpret_cast<const uint4*>(p.m1_pure);
        // chunk tickets run two ahead and the counts of the next chunk are fetched before the current one is scored
        auto load_counts = [&](int chunk) -> uint32_t {
            const int i = chunk * 32 + lane;
            if (i >= nv) return 0u;
            return BIG ? cnt_g[i] : lds32(s_cnt + (uint32_t)i * 4u);
        };
        int cur = tile_ticket_get(tile_ticket_issue(s_ctrC, lane));
        int nxt = tile_ticket_get(tile_ticket_issue(s_ctrC, lane));
        uint32_t c4 = load_counts(cur);
        for (; cur < nchunk;) {
            const int raw = tile_ticket_issue(s_ctrC, lane);
            const uint32_t c4_next = load_counts(nxt);
            const int iv = cur * 32 + lane;
            int sl = (int)__umulhi((uint32_t)iv, inv_s4);
            int v = iv - sl * S4;
            if (sl >= nsl) { sl = nsl - 1; v = S4; } // past the tile: sits at the end of the last block
            const uint4 t1 = lds128(s_st + (uint32_t)sl * 64u + 16u); // g_rel, r_rel, AG, sel4
            const uint4 t2 = lds128(s_st + (uint32_t)sl * 64u + 32u); // sel01, sel23, g_end, r_end
            const int A = (int)(t1.z & 0xFF), G = (int)__byte_perm(t1.z, 0u, 0x4441);
            const bool live = v < S && G > 0;
            const int vv = min(v, S);
            const int gpos = (int)t1.x + vv * G, rpos = (int)t1.y + vv * A;
            const int gend = v < S ? gpos + G : (int)t2.z;
            const int rend = v < S ? rpos + A : (int)t2.w;
            const int g_lo = __shfl_sync(0xffffffffu, gpos, 0), g_hi = __shfl_sync(0xffffffffu, gend, 31);
            const int r_lo = __shfl_sync(0xffffffffu, rpos, 0), r_hi = __shfl_sync(0xffffffffu, rend, 31);
            // cells that emit nothing (padding slots, skipped sites, past the tile) compute along and store into a scratch cell
            const uint32_t cell_g = live ? s_wg + (uint32_t)(gpos - g_lo) * 4u : s_wg + TILE_G_TRASH * 4u;
            const uint32_t cell_r = live ? s_wr + (uint32_t)(rpos - r_lo) * 4u : s_wr + TILE_R_TRASH * 4u;
            const uint4 slot = lds128(s_st + (uint32_t)sl * 64u);
            bulk_wait_read(); // this warp's previous copies (issued by lane 0) must have finished reading the slice
            __syncwarp();
            const int c0 = (int)__byte_perm(c4, 0u, 0x4440), c1 = (int)__byte_perm(c4, 0u, 0x4441);
            const int c2 = (int)__byte_perm(c4, 0u, 0x4442), c3 = (int)__byte_perm(c4, 0u, 0x4443);
            const int n = (int)__vsadu4(c4, 0u);
            const uint32_t seen4 = __vcmpne4(c4, 0u);
            if (PURE && __all_sync(0xffffffffu, !live || __popc(seen4) <= 8)) {
                // every cell of the chunk is pure (or empty): GL / PL by class from the depth table, written slot by slot
                const int x = ((__ffs(seen4 | 0x80000000u) - 1) >> 3) & 3;
                M1Pure tv;
                {
                    const uint4 t = __ldg(pure_tab + n);
                    tv.gl1 = __uint_as_float(t.x); tv.gl0 = __uint_as_float(t.y); tv.pl1 = (int32_t)t.z; tv.pl0 = (int32_t)t.w;
                }
                const uint32_t cm = lds32(s_st + (uint32_t)sl * 64u + 48u + 4u * (uint32_t)x);
                const int gmax = __reduce_max_sync(0xffffffffu, live ? G : 0);
                const uint32_t dstb = cell_g;
#pragma unroll
                for (int g = 0; g < 15; ++g) {
                    if (g >= gmax) break;
                    const bool one = (cm >> g) & 1u;
                    if (g < G && live) {
                        if (stage_gl) sts32(dstb + 4u * g, __float_as_uint(one ? tv.gl1 : tv.gl0));
                        if (has_pl) sts32(dstb + 4u * g + TILE_WST_G * 4, (uint32_t)(one ? tv.pl1 : tv.pl0));
                    }
                }
                if (live) { // the slot of xx
                    const uint32_t hs = dstb + ((cm >> 16) & 0xFu) * 4u;
                    if (stage_gl) sts32(hs, 0u);
                    if (has_pl) sts32(hs + TILE_WST_G * 4, 0u);
                }
            } else {
                // the all-15 flag of the lane's site is 0 for a skipped site: its lanes store into the scratch cell and need the
                // slot test (their offsets may be 0xFF)
                float q[15];
                m1f_scores_noclamp(n, c0, c1, c2, c3, p.m1_bsum, p.m1_het, q);
                if (__all_sync(0xffffffffu, (t1.z >> 16) != 0u)) tile_emit_cell<true>(q, slot, cell_g, stage_gl, has_pl);
                else tile_emit_cell<false>(q, slot, cell_g, stage_gl, has_pl);
            }
            if (has_ad) { // AD in allele order (vcfgl.cpp:806-831): byte permute, selector 4 reads 0
                sts32(cell_r, __byte_perm(c4, 0u, t2.x));
                if (A > 1) sts32(cell_r + 4, __byte_perm(c4, 0u, t2.x >> 16));
                if (A > 2) sts32(cell_r + 8, __byte_perm(c4, 0u, t2.y));
                if (A > 3) sts32(cell_r + 12, __byte_perm(c4, 0u, t2.y >> 16));
                if (A > 4) sts32(cell_r + 16, __byte_perm(c4, 0u, t1.w));
            }
            if (live && n == 0) { // gl_methods.cpp:359-366
#pragma unroll 1
                for (int g = 0; g < G; ++g) {
                    sts32(cell_g + 4 * g, VGL_F32_MISSING_BITS);
                    sts32(cell_g + 4 * (TILE_WST_G + g), (uint32_t)VGL_I32_MISSING);
                }
            }
            if (v == S && G > 0) { // first padding slot of a site: zero the block's padding
                const uint32_t pg = s_wg + (uint32_t)(gpos - g_lo) * 4u, pr = s_wr + (uint32_t)(rpos - r_lo) * 4u;
#pragma unroll 1
                for (int g = 0; g < gend - gpos; ++g) {
                    sts32(pg + 4 * g, 0u);
                    sts32(pg + 4 * (TILE_WST_G + g), 0u);
                }
#pragma unroll 1
                for (int a = 0; a < rend - rpos; ++a) sts32(pr + 4 * a, 0u);
            }
            fence_async_smem();
            __syncwarp();
            const uint32_t gb = (uint32_t)(g_hi - g_lo) * 4u, rb = (uint32_t)(r_hi - r_lo) * 4u;
            if (lane == 0) {
                if (gb) {
                    if (has_gl) bulk_store(gl_t + g_lo, s_wg, gb);
                    if (has_pl) bulk_store(pl_t + g_lo, s_wg + TILE_WST_G * 4, gb);
                }
                if (rb && has_ad) bulk_store(ad_t + r_lo, s_wr, rb);
                bulk_commit();
            }
            if (XTRA && xflags) {
                // GP (vcfgl.cpp:941-970) and FORMAT ADF / ADR (vcfgl.cpp:806-831) go through the same slices once the copies above
                // have read them: GP replaces PL, ADF then ADR replace AD; the padding words are already zero.  The forward reads
                // per base are the draws phase A summed per site.
                uint32_t fw4 = 0u;
                if (xflags & 6u) {
                    const int nmax = __reduce_max_sync(0xffffffffu, n);
                    fw4 = tile_strand_counts(p, site_base + (uint32_t)sl, (uint32_t)v, c4, nmax);
                }
                bulk_wait_read();
                __syncwarp();
                if ((xflags & 1u) && live) {
                    if (n == 0) {
#pragma unroll 1
                        for (int g = 0; g < G; ++g) sts32(cell_g + 4 * (TILE_WST_G + g), VGL_F32_MISSING_BITS);
                    } else {
                        float sum = 0.0f;
#pragma unroll 1
                        for (int g = 0; g < G; ++g) {
                            const float e10 = __double2float_rn(exp10((double)__uint_as_float(lds32(cell_g + 4 * g))));
                            sts32(cell_g + 4 * (TILE_WST_G + g), __float_as_uint(e10));
                            sum = __fadd_rn(sum, e10);
                        }
#pragma unroll 1
                        for (int g = 0; g < G; ++g)
                            sts32(cell_g + 4 * (TILE_WST_G + g), __float_as_uint(__fdiv_rn(__uint_as_float(lds32(cell_g + 4 * (TILE_WST_G + g))), sum)));
                    }
                }
                auto put_r = [&](uint32_t c) { // per-base counts in allele order, like AD
                    sts32(cell_r, __byte_perm(c, 0u, t2.x));
                    if (A > 1) sts32(cell_r + 4, __byte_perm(c, 0u, t2.x >> 16));
                    if (A > 2) sts32(cell_r + 8, __byte_perm(c, 0u, t2.y));
                    if (A > 3) sts32(cell_r + 12, __byte_perm(c, 0u, t2.y >> 16));
                    if (A > 4) sts32(cell_r + 16, __byte_perm(c, 0u, t1.w));
                };
                if (xflags & 2u) put_r(fw4);
                fence_async_smem();
                __syncwarp();
                if (lane == 0 && (xflags & 3u)) {
                    if (gb && (xflags & 1u)) bulk_store(gp_t + g_lo, s_wg + TILE_WST_G * 4, gb);
                    if (rb && (xflags & 2u)) bulk_store(adf_t + r_lo, s_wr, rb);
                    bulk_commit();
                }
                if (xflags & 4u) {
                    bulk_wait_read();
                    __syncwarp();
                    put_r(__vsub4(c4, fw4));
                    fence_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        if (rb) bulk_store(adr_t + r_lo, s_wr, rb);
                        bulk_commit();
                    }
                }
            }
            cur = nxt;
            c4 = c4_next;
            nxt = tile_ticket_get(raw);
        }
    }
    bulk_wait_all(); // global writes of this warp's last copies complete before exit
    // the last CTA to leave rearms the tile ticket for the next launch on this slot (no memset between launches)
    if (tid == 0) {
        const unsigned done = atomicAdd(p.ticket + 1, 1u);
        if (done == gridDim.x - 1) {
            p.ticket[0] = 0u;
            p.ticket[1] = 0u;
        }
    }
}

static size_t tile_dyn_smem(bool big)
{
    return 2048 + 4096 + (size_t)TILE_WARPS * (2 * TILE_WST_G + TILE_WST_R) * 4 + TILE_MAX_SITES * sizeof(TSite) + TILE_MAX_SITES * 16 +
           (big ? 0 : (size_t)TILE_CELLS * 4);
}

template <bool GEN, bool BIG, bool AUX, bool PURE, bool XTRA>
static void launch_tile_p(const DevParams& p, cudaStream_t st, int n_sms)
{
    const size_t dyn = tile_dyn_smem(BIG) + (AUX ? TILE_MAX_SITES * sizeof(TAux) + (BIG ? 0 : (TILE_CELLS / 32) * 32) : 0);
    cudaFuncSetAttribute(k_tile_m1f<GEN, BIG, AUX, PURE, XTRA>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    cudaFuncSetAttribute(k_tile_m1f<GEN, BIG, AUX, PURE, XTRA>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_tile_m1f<GEN, BIG, AUX, PURE, XTRA>, TILE_BLOCK, dyn);
    if (per_sm < 1) per_sm = 1;
    if (per_sm > TILE_SCRATCH_CTAS_PER_SM) per_sm = TILE_SCRATCH_CTAS_PER_SM;
    int grid = n_sms * per_sm;
    if (grid > p.n_tiles) grid = p.n_tiles;
    k_tile_m1f<GEN, BIG, AUX, PURE, XTRA><<<grid, TILE_BLOCK, dyn, st>>>(p);
}
template <bool GEN, bool BIG, bool AUX>
static void launch_tile_t(const DevParams& p, cudaStream_t st, int n_sms)
{
    const bool xtra = AUX && (p.gp != nullptr || p.adf != nullptr || p.adr != nullptr);
    if (AUX && xtra) { // the extra planes come with the general code (no closed form for pure chunks: GP needs the staged GL values of every cell anyway)
        launch_tile_p<GEN, BIG, AUX, false, AUX>(p, st, n_sms);
    } else if (p.m1_pure != nullptr) launch_tile_p<GEN, BIG, AUX, true, false>(p, st, n_sms);
    else launch_tile_p<GEN, BIG, AUX, false, false>(p, st, n_sms);
}

// aux: QS / I16 / INFO ADF, ADR wanted (TILE_M1F_AUX_TAGS)
void launch_tile_m1f(const DevParams& p, cudaStream_t st, int n_sms, bool aux)
{
    const bool all3 = p.gl && p.pl && p.ad, big = tile_m1f_scratch_words(p.S, 1) > 0;
    if (aux) {
        if (big) launch_tile_t<true, true, true>(p, st, n_sms);
        else launch_tile_t<true, false, true>(p, st, n_sms);
    } else if (all3 && !big) launch_tile_t<false, false, false>(p, st, n_sms);
    else if (all3) launch_tile_t<false, true, false>(p, st, n_sms);
    else if (!big) launch_tile_t<true, false, false>(p, st, n_sms);
    else launch_tile_t<true, true, false>(p, st, n_sms);
}

// ---- the count-level sampler's draws read by read, in the replay layout (vgl_native_draws): pass 0 writes the depths,
// pass 1 the reads.  The reads of a cell are listed grouped by base (A.., C.., G.., T..); in the site's last cell with
// reads the read picked by P_LAST moves to the end (it is the site's last simulated read, vcfgl.cpp:657).  The read
// listed at position k carries tail distance k of the cell's stream; strands follow their reads.
__global__ void k_tile_m1f_draws(const DevParams p, int pass, int32_t* depths, const int64_t* off, uint8_t* bases, uint8_t* strands, uint8_t* tails)
{
    __shared__ __align__(16) unsigned char sm[2048 + 4096];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        reinterpret_cast<uint2*>(sm)[i] = reinterpret_cast<const uint2*>(p.pois_alias)[i];
        reinterpret_cast<uint4*>(sm + 2048)[i] = reinterpret_cast<const uint4*>(p.err_cdf)[i];
    }
    __syncthreads();
    TileRng R;
    R.s_alias = smem_u32(sm);
    R.s_cdf_e = R.s_alias + 2048;
    R.fixed_depth = p.depth_mode == VGL_DEPTH_FIXED ? (int)p.depth_mean : -1;
    R.has_err = p.error_rate > 0.0;
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.n_cells) return;
    const int64_t sl = c / p.S;
    const uint32_t sample = (uint32_t)(c - sl * p.S);
    const unsigned long long site = (unsigned long long)(p.first_site + sl);
    const uint32_t ad = tile_sample_cell(p, R, site, sample, p.gt[c]);
    const int n = (int)__vsadu4(ad, 0u);
    if (pass == 0) { depths[c] = n; return; }
    if (n == 0) return;
    bool last = true;
    for (int s2 = (int)sample + 1; s2 < p.S && last; ++s2) last = depths[sl * p.S + s2] == 0;
    const int pick = last ? tile_last_read(p, site, sample, n) : -1;
    u32x4 blk;
    int cur_blk = -1;
    auto strand_of = [&](int r) -> uint8_t {
        if ((r >> 7) != cur_blk) {
            cur_blk = r >> 7;
            blk = philox_rk(p, (uint32_t)site, (uint32_t)(site >> 32) & 0xFFu, sample, ((uint32_t)P_STRAND << 24) | (uint32_t)cur_blk);
        }
        return ((tile_word(blk, (r & 127) >> 5) >> (r & 31)) & 1u) ? 0 : 1; // 0 = forward
    };
    const int64_t o = off[c];
    int k = 0;
    for (int r = 0; r < n; ++r) {
        if (r == pick) continue;
        bases[o + k] = (uint8_t)tile_base_of_read(ad, r);
        strands[o + k] = strand_of(r);
        tails[o + k] = (uint8_t)tile_tail_of_read(p, site, sample, k);
        ++k;
    }
    if (pick >= 0) {
        bases[o + k] = (uint8_t)tile_base_of_read(ad, pick);
        strands[o + k] = strand_of(pick);
        tails[o + k] = (uint8_t)tile_tail_of_read(p, site, sample, k);
    }
}

void launch_tile_m1f_draws(const DevParams& p, cudaStream_t st, int pass, int32_t* depths, const int64_t* off, uint8_t* bases, uint8_t* strands,
                           uint8_t* tails)
{
    const unsigned grid = (unsigned)((p.n_cells + 127) / 128);
    k_tile_m1f_draws<<<grid, 128, 0, st>>>(p, pass, depths, off, bases, strands, tails);
}

int tile_m1f_sites_per_tile(int S)
{
    const int S4 = (S + 3) & ~3;
    int T = TILE_CELLS / S4;
    return T < 1 ? 1 : (T > TILE_MAX_SITES ? TILE_MAX_SITES : T);
}
// 32-bit words of global scratch the kernel needs for S samples on a device with n_sms SMs (0: counts fit shared memory)
size_t tile_m1f_scratch_words(int S, int n_sms)
{
    const int S4 = (S + 3) & ~3;
    return S4 > TILE_CELLS ? tile_m1f_row_words(S4) * TILE_SCRATCH_CTAS_PER_SM * n_sms : 0;
}

} // namespace vgl
