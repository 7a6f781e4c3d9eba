// k_tile_m2 -- GL model 2 (the GATK-style per-read likelihood, gl_methods.cpp:4-150) in the tile framework of
// tile_m1f.cu: native RNG, same-mean Poisson or fixed depth, tags GL / PL / AD / DP (+ INFO/AD, INFO/DP).
//   FIXED  one run-constant quality score (--error-qs 0, or --error-qs 1 = per-site beta-distributed base-picking
//          error rate, vcfgl.cpp:425-437): homT / het / homF are run constants (vcfgl.cpp:1713-1740)
//   LUT    per-read quality score (--error-qs 2, --precise-gl 0): each read's error probability is beta-distributed,
//          its (binned / adjusted) quality score picks the three constants from qScore_to_log10_gl (gl_methods.cpp:99-104)
//
// Model 2 adds one of three constants to every genotype for every read and max-normalises the vector after EVERY
// read in float (gl_methods.cpp:27-58), so the result depends on the ORDER of a cell's reads: the kernel works on
// the read sequence, not on counts.  The sequence is still drawn at count level where that is exact:
//   depth            alias table (as the model-1 tile kernel)
//   haplotype picks  one random bit per read
//   mis-calls        number of mis-called reads E ~ Binomial(n, e), their positions uniform without replacement, wrong
//                    base uniform over the other three -- the joint law of n iid reads with P(error) = e
//   LUT: quality     per read one alias-table draw from the law of the (binned / adjusted) quality score of a
//        scores      Beta(a, b) error probability, P(q) = I(p_hi) - I(p_lo), tabulated on the host (tables.cpp).  The
//                    reference draws a read's quality independently of whether the read was mis-called (vcfgl.cpp:485, 495)
// Every draw is a pure function of (seed, site, sample[, read]); phase C re-derives the sequence of phase A instead
// of storing it.  Cells deeper than 64 reads use one Philox block per read (the per-read sampler of kernels.cu).
//
// Phases per tile as in tile_m1f.cu: A sample + FORMAT/DP + site totals, B per-site record, C score + emit
// (scatter in allele order into the warp's shared-memory slice, one bulk async copy per plane).
#include "tables.h"
#include "tile_common.cuh"

namespace vgl {

#define M2_TAB_BYTES (M2_TAB_DOUBLES * 8) // per quality score: pair table [4][17] doubles, then class table [2][8]
#define M2_TAB_MAXQ 8                     // scores whose tables fit the shared-memory copy
#define M2_TAB_CLS 544                    // byte offset of the class table
#define M2_SCR_BYTES 2048                 // per-warp scratch: 16 words per lane (the quality classes of up to 64 reads, LUT mode)
#ifndef M2_MIN_CTAS_LUT
#define M2_MIN_CTAS_LUT 4                // MODE 2 (per-read quality classes): more registers beat a fifth resident CTA (0.706 -> 0.648 ms on cfg3(ii))
#endif
#ifndef M2_MIN_CTAS
#define M2_MIN_CTAS 5
#endif

// BIG variant: words of a CTA's global row = counts [S4] | chunk records [S4 / 32 + 1] x 4
__host__ __device__ inline size_t m2_big_row_words(int S4) { return (size_t)S4 + (size_t)4 * (S4 / 32 + 1); }

struct __align__(16) M2SiteE {
    double e;  // base-picking error probability of the site
    float l2;  // log2(1 - e) when the float CDF walk is usable, else 0
    float er;  // e / (1 - e)
};

// rare paths kept out of line (the kernel's hot loops should stay within the instruction cache)
__device__ __noinline__ int m2_binom_inversion(int n, double e, uint32_t u) { return binom_inversion(n, e, u01_32(u)); }
__device__ __noinline__ double m2_site_beta(const DevParams& p, unsigned long long site)
{
    Stream bs;
    Key key;
    key.k0 = p.k0; key.k1 = p.k1;
    bs.init(key, (int64_t)site, 0xFFFFFFFFu, 0, P_SITE);
    return beta_draw(bs, p.beta_a, p.beta_b);
}

struct M2Rng {
    uint32_t s_alias; // shared address: Poisson alias table
    uint32_t s_cdf_e; // shared address: [256] uint4 P(E <= j | n) * 2^32 (run-constant error rate)
    uint32_t s_qcls;  // shared address: LUT mode, [256] (threshold24 << 8 | alias) of the minor classes' conditional law, then [256] class info words
    int fixed_depth;
    bool has_err;
};

// bit i of x moves to bit 2i (x < 2^16)
__device__ __forceinline__ uint32_t spread16(uint32_t x)
{
    x = (x | (x << 8)) & 0x00FF00FFu;
    x = (x | (x << 4)) & 0x0F0F0F0Fu;
    x = (x | (x << 2)) & 0x33333333u;
    x = (x | (x << 1)) & 0x55555555u;
    return x;
}

// read i of a cell deeper than 64 reads: one Philox block per read, as CellSource::read (cell_source.cuh)
__device__ __noinline__ int m2_deep_base(const DevParams& p, unsigned long long site, uint32_t sample, int i, int g0, int g1, double e)
{
    const u32x4 w = philox_rk(p, (uint32_t)site, ((uint32_t)(site >> 32) & 0xFFu) | ((uint32_t)i << 8), sample, (uint32_t)P_READ << 24);
    const int truth = (w.y >> 31) ? g1 : g0;
    int base = truth;
    if (u01_32(w.x) < e) base = (truth + 1 + (int)mulhi32(w.z, 3u)) & 3;
    return base;
}

// depth of a cell from block 0 of its P_COUNTS counter
__device__ __forceinline__ int m2_depth(const DevParams& p, const M2Rng& R, const u32x4& b0, uint32_t gt, uint32_t sample)
{
    int n;
    if (R.fixed_depth >= 0) {
        n = R.fixed_depth;
    } else {
        const uint32_t col = b0.x >> 24;
        uint2 en;
        if (p.alias_row) en = __ldg(reinterpret_cast<const uint2*>(p.pois_alias) + (size_t)__ldg(p.alias_row + min(sample, (uint32_t)p.S - 1u)) * 256u + col); // the sample's own mean (padding lanes: any row, their depth is dropped)
        else en = lds64(R.s_alias + col * 8u);
        const unsigned long long frac = ((unsigned long long)__funnelshift_l(b0.y, b0.x, 8) << 32) | (b0.y << 8);
        const unsigned long long thr = ((unsigned long long)en.y << 32) | (en.x & 0xFFFFFF00u);
        n = frac < thr ? (int)col : (int)(en.x & 0xFFu);
    }
    if (gt & 0x88u) n = 0; // missing genotype: depth drawn but discarded (vcfgl.cpp:371-379)
    return n;
}

// One FIXED-mode cell.  Returns the packed 8-bit base counts; with SEQ also the read sequence as 2-bit codes
// (read i in bits 2(i&15) of w[i>>4]) when n <= 64.  Draws: block 0 = {x,y: depth; z: number of errors; w: haplotype
// bits 0..31}, block 1 = {x: haplotype bits 32..63; y,z,w: errors 1..3}; further errors and re-draws of occupied
// positions from block 10 on.
template <bool SEQ, bool SITE_E>
__device__ __forceinline__ uint32_t m2_cell_fixed(const DevParams& p, const M2Rng& R, unsigned long long site, uint32_t sample, uint32_t gt,
                                                  const M2SiteE& se, int& n_out, uint32_t (&w)[4])
{
    const int g0 = gt & 0x3, g1 = (gt >> 4) & 0x3;
    const uint32_t c0 = (uint32_t)site, c1 = (uint32_t)(site >> 32) & 0xFFu;
    const u32x4 b0 = philox_rk(p, c0, c1, sample, (uint32_t)P_COUNTS << 24);
    const u32x4 b1 = philox_rk(p, c0, c1, sample, ((uint32_t)P_COUNTS << 24) | 1u); // independent of b0: the two chains overlap
    const int n = m2_depth(p, R, b0, gt, sample);
    n_out = n;
    if (SEQ) w[0] = w[1] = w[2] = w[3] = 0u;
    if (n == 0) return 0u;
    if (n > 64) { // deep cell: per-read draws
        uint32_t ad = 0u;
        for (int i = 0; i < n; ++i) ad += 1u << (8 * m2_deep_base(p, site, sample, i, g0, g1, se.e));
        return ad;
    }
    const unsigned long long h = ((unsigned long long)b1.x << 32) | b0.w;
    const unsigned long long hm = h & (n >= 64 ? ~0ull : ((1ull << n) - 1ull));
    const bool het = g0 != g1;
    const int k0 = het ? __popcll(hm) : n;
    uint32_t ad = ((uint32_t)k0 << (8 * g0)) + ((uint32_t)(n - k0) << (8 * g1));
    if (SEQ) {
        const uint32_t base = 0x55555555u * (uint32_t)g1, dx = (uint32_t)(g0 ^ g1);
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (16 * k < n) w[k] = base ^ (spread16((uint32_t)(h >> (16 * k)) & 0xFFFFu) * dx);
    }
    // number of mis-called reads
    int E = 0;
    if (SITE_E) {
        if (se.e > 0.0) {
            const float p0 = exp2f((float)n * se.l2);
            const float uf = ((float)(b0.z >> 8) + 0.5f) * 5.9604645e-08f; // 24-bit uniform in (0,1]: the top word rounds to 1.0f
            if (se.l2 != 0.0f && p0 > 1e-30f) {
                float pr = p0, cdf = p0;
                while (uf > cdf && E < n) {
                    pr *= (float)(n - E) / (float)(E + 1) * se.er;
                    cdf += pr;
                    ++E;
                }
                // The float CDF can end below uf: it often ends at 0.99999994f or lower, and the top word's uf is 1.0f.  The walk
                // has then run to E = n; such a cell takes the exact inversion in double from the same word.  Sending every
                // uf > 0.998f there, as sample_counts does, made k_tile_m2 12% slower on cfg3(i) (0.62 -> 0.70 ms per batch, B200
                // at 1000 W): one lane in 500 takes it, so one warp-wide pass in 16 waits for a double-precision inversion.
                if (uf > cdf) E = m2_binom_inversion(n, se.e, b0.z);
            } else {
                E = m2_binom_inversion(n, se.e, b0.z);
            }
        }
    } else if (R.has_err) {
        const uint4 c = lds128(R.s_cdf_e + (uint32_t)n * 16u);
        E = (b0.z >= c.x) + (b0.z >= c.y) + (b0.z >= c.z);
        if (b0.z >= c.w) E = m2_binom_inversion(n, se.e, b0.z);
    }
    if (E > 0) {
        unsigned long long hit = 0ull;
        Stream st;
        Key key;
        key.k0 = p.k0; key.k1 = p.k1;
        st.init(key, (int64_t)site, sample, 0, P_COUNTS);
        st.block = 10;
        for (int j = 0; j < E; ++j) {
            uint32_t r = j == 0 ? b1.y : (j == 1 ? b1.z : (j == 2 ? b1.w : st.next()));
            uint32_t pos, woff;
            for (;;) {
                const uint32_t q = mulhi32(r, 3u * (uint32_t)n);
                pos = (q * 0xAAABu) >> 17; // q / 3, q < 192
                woff = q - 3u * pos;
                if (!((hit >> pos) & 1ull)) break;
                r = st.next();
            }
            hit |= 1ull << pos;
            const int old = het ? (((h >> pos) & 1ull) ? g0 : g1) : g0;
            const int neu = (old + 1 + (int)woff) & 3;
            ad += (1u << (8 * neu)) - (1u << (8 * old));
            if (SEQ) {
                const uint32_t sh = 2u * (pos & 15u), flip = (uint32_t)(old ^ neu) << sh;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if ((int)(pos >> 4) == k) w[k] ^= flip;
            }
        }
    }
    return ad;
}

// LUT mode, cells deeper than 64 reads: the quality score of read i from word i&3 of block 0x10000 + (i>>2) of the cell's
// P_QS counter -> alias draw from the full class law.
// Returns the class info word (q | out-of-range << 9 | dense index << 16).
__device__ __forceinline__ uint32_t m2_lut_qs(const DevParams& p, const M2Rng& R, unsigned long long site, uint32_t sample, int i, u32x4& qblk)
{
    if ((i & 3) == 0) qblk = philox_rk(p, (uint32_t)site, (uint32_t)(site >> 32) & 0xFFu, sample, ((uint32_t)P_QS << 24) | (uint32_t)(0x10000 + (i >> 2)));
    const uint32_t r = (i & 3) == 0 ? qblk.x : ((i & 3) == 1 ? qblk.y : ((i & 3) == 2 ? qblk.z : qblk.w));
    const uint32_t col = r >> 24;
    const uint32_t en = __ldg(p.qcls + col); // the full class law (deep cells only: global memory)
    const uint32_t cls = (r & 0xFFFFFFu) < (en >> 8) ? col : (en & 0xFFu);
    const uint32_t info = lds32(R.s_qcls + 1024u + cls * 4u);
    if (info & 0x200u) atomicExch(p.status, (int)VGL_ERANGE); // apply_qs_bins() -> ERROR, vcfgl.cpp:63
    return info;
}

// one read of base b (ACGT int) with constants c2 / c1 / c0 (both / one / no allele of the genotype equals the
// read) added to all 15 base pairs, then the max over the site's genotypes is subtracted (gl_methods.cpp:27-58).
// Base pairs that are not genotypes of the site were initialised to -inf and stay there.
__device__ __forceinline__ void m2_update(float (&gl)[15], int b, double c2, double c1, double c0)
{
    const bool p0 = b == 0, p1 = b == 1, p2 = b == 2, p3 = b == 3;
    double a[15];
    a[0] = p0 ? c2 : c0;
    a[2] = p1 ? c2 : c0;
    a[5] = p2 ? c2 : c0;
    a[9] = p3 ? c2 : c0;
    a[14] = c0;
    a[1] = (p0 || p1) ? c1 : c0;
    a[3] = (p0 || p2) ? c1 : c0;
    a[4] = (p1 || p2) ? c1 : c0;
    a[6] = (p0 || p3) ? c1 : c0;
    a[7] = (p1 || p3) ? c1 : c0;
    a[8] = (p2 || p3) ? c1 : c0;
    a[10] = p0 ? c1 : c0;
    a[11] = p1 ? c1 : c0;
    a[12] = p2 ? c1 : c0;
    a[13] = p3 ? c1 : c0;
    float mx = -CUDART_INF_F;
#pragma unroll
    for (int k = 0; k < 15; ++k) {
        gl[k] = __double2float_rn(__dadd_rn((double)gl[k], a[k])); // float += double
        mx = fmaxf(mx, gl[k]);
    }
#pragma unroll
    for (int k = 0; k < 15; ++k) gl[k] = __fsub_rn(gl[k], mx);
}

// ---- table-driven forms (constants finite and non-zero, or -inf; the host checks).  The float -> double conversion
// of a GL value is done by integer arithmetic: every value is <= 0, so with the sign bit set
// hi = (bits >> 3) + 0xA8000000, lo = bits << 29 is the exact double; +0 / -0 map to -2^-383 / -2^-127, which vanish
// in the sum with any table constant, and -inf maps to -2^128, which the double -> float conversion turns back into -inf.
__device__ __forceinline__ double m2_f2d(float f)
{
    const uint32_t b = __float_as_uint(f);
    return __hiloint2double((int)((b >> 3) + 0xA8000000u), (int)(b << 29));
}
__device__ __forceinline__ double lds_f64(uint32_t a)
{
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
    return v;
}
// one read on all 15 base pairs; t = shared address of the read base's row of the pair table
__device__ __forceinline__ void m2_update_pairs(float (&gl)[15], uint32_t t)
{
    float mx = -CUDART_INF_F;
#pragma unroll
    for (int k = 0; k < 15; ++k) {
        gl[k] = __double2float_rn(__dadd_rn(m2_f2d(gl[k]), lds_f64(t + 8u * k)));
        mx = fmaxf(mx, gl[k]);
    }
#pragma unroll
    for (int k = 0; k < 15; ++k) gl[k] = __fsub_rn(gl[k], mx);
}
// one read on the six classes of a two-base cell; t = shared address of the class row ([read is x])
__device__ __forceinline__ void m2_update_classes(float (&gc)[6], uint32_t t)
{
    float mx = -CUDART_INF_F;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        gc[k] = __double2float_rn(__dadd_rn(m2_f2d(gc[k]), lds_f64(t + 8u * k)));
        mx = fmaxf(mx, gc[k]);
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) gc[k] = __fsub_rn(gc[k], mx);
}
// bit i = byte i of x is non-zero
__device__ __forceinline__ uint32_t nonzero_bytes(uint32_t x)
{
    return (((__vcmpne4(x, 0u)) & 0x01010101u) * 0x01020408u) >> 24;
}

// the reads of one cell, in order
template <int MODE>
struct M2Reads {
    uint32_t w0, w1, w2, w3, cur; // packed 2-bit base codes (cells of at most 64 reads)
    bool deep;
    unsigned long long site;
    uint32_t sample;
    int g0, g1;
    double e;
    u32x4 qblk;
    // returns the base of read i (reads must be asked in order)
    __device__ __forceinline__ int base(const DevParams& p, int i)
    {
        if (deep) return m2_deep_base(p, site, sample, i, g0, g1, e);
        if ((i & 15) == 0) cur = (i >> 4) == 0 ? w0 : ((i >> 4) == 1 ? w1 : ((i >> 4) == 2 ? w2 : w3));
        const int b = (int)(cur & 3u);
        cur >>= 2;
        return b;
    }
};

// ---- per-read quality-score classes of a LUT-mode cell of at most 64 reads, drawn at count level: the number of reads M whose
// class is not the dominant one (M ~ Binomial(n, p_minor): threshold table, exact inversion beyond it), their positions
// (uniform without replacement) and their classes (alias table of the conditional law) -- the joint law of n iid draws
// from the class law.  Words of the cell's P_QS stream: word 0 = M, then per minor read one word for the position
// (+ one per re-draw of an occupied position) and one for the class.  Cells deeper than 64 reads draw every read's
// class on its own (m2_lut_qs).
__device__ __forceinline__ int m2_qs_minor_count(const DevParams& p, int n, uint32_t u)
{
    const uint4 c = __ldg(reinterpret_cast<const uint4*>(p.qm_cdf) + n);
    int M = (u >= c.x) + (u >= c.y) + (u >= c.z);
    if (u >= c.w) M = m2_binom_inversion(n, p.q_minor, u);
    return M;
}
// calls put(position, class) for each of the cell's minor reads; returns their number
template <typename PUT>
__device__ __forceinline__ int m2_qs_minor_reads(const DevParams& p, const M2Rng& R, unsigned long long site, uint32_t sample, int n, PUT put)
{
    Stream st;
    Key key;
    key.k0 = p.k0; key.k1 = p.k1;
    st.init(key, (int64_t)site, sample, 0, P_QS);
    const int M = m2_qs_minor_count(p, n, st.next());
    unsigned long long hit = 0ull;
    for (int j = 0; j < M; ++j) {
        uint32_t pos;
        for (;;) {
            pos = mulhi32(st.next(), (uint32_t)n);
            if (!((hit >> pos) & 1ull)) break;
        }
        hit |= 1ull << pos;
        const uint32_t r = st.next(), col = r >> 24;
        const uint32_t en = lds32(R.s_qcls + col * 4u); // conditional alias table
        put(pos, (r & 0xFFFFFFu) < (en >> 8) ? col : (en & 0xFFu));
    }
    return M;
}

// final GL / PL of a cell, scattered into the warp's stage slice in allele order (vcfgl.cpp:907-939)
__device__ __forceinline__ void m2_emit_cell(const float (&gl)[15], const uint4 slot, uint32_t cell_g, bool has_gl, bool has_pl)
{
    const uint32_t sw[4] = {slot.x, slot.y, slot.z, slot.w};
#pragma unroll
    for (int k = 0; k < 15; ++k) {
        const uint32_t off = __byte_perm(sw[k >> 2], 0u, 0x4440u | (k & 3));
        if (off != 0xFFu) {
            const uint32_t dst = cell_g + off;
            if (has_gl) asm volatile("st.shared.f32 [%0], %1;" ::"r"(dst), "f"(gl[k]) : "memory");
            if (has_pl) {
                const float u = __fadd_rz(__fadd_rz(__fmul_rn(-10.0f, gl[k]), 0.5f), 8388608.0f);
                asm volatile("st.shared.b32 [%0+%2], %1;" ::"r"(dst), "r"(pl_from_magic_bits(u)), "n"(TILE_WST_G * 4) : "memory");
            }
        }
    }
}

// base pairs (bit k = pair k) that hold base b twice / exactly once
__device__ __forceinline__ uint32_t m2_hom_bit(int b) { return 1u << ((b * (b + 3)) >> 1); }
__device__ __forceinline__ uint32_t m2_het_mask(int b)
{
    // pairs (j, k), j < k <= 4, with j == b or k == b
    return b == 0 ? 0x044Au : (b == 1 ? 0x0892u : (b == 2 ? 0x1118u : 0x21C0u));
}

struct __align__(16) M2Chunk { // per chunk of 32 virtual cells, written in phase A
    uint32_t base2, base15; // first list position of the chunk's two-base / general mixed cells (the latter counted from the end)
    uint32_t mask2, mask15; // lanes of those cells
};

// MODE 0: FIXED with the run-constant error rate, 1: FIXED with a per-site error rate, 2: LUT (per-read qs)
// TAB: the constants of every quality score in use fit the shared-memory tables (always in FIXED mode) -> table-driven
// updates, the six-class form for cells whose reads show at most two bases, and (PURE) the closed form of cells whose
// reads all agree.
//
// Phase C is split in two.  Model 2 renormalises after every read, so a cell costs one dependent update chain per read --
// but most cells are "pure" (every read shows the same base with the same quality score), and their vector depends on
// the depth alone (m2_pure_table).  Phase A lists the other ("mixed") cells of the tile; phase M walks that list densely
// (every lane a mixed cell), runs the per-read chains and parks the 15 results per cell in a per-CTA scratch row in
// global memory (L2-resident); phase C then only assembles: table values for pure cells, parked values for mixed ones.
template <int MODE, bool BIG, bool TAB, bool GLPL>
__global__ void __launch_bounds__(TILE_BLOCK, MODE == 2 ? M2_MIN_CTAS_LUT : M2_MIN_CTAS) k_tile_m2(const __grid_constant__ DevParams p)
{
    extern __shared__ __align__(16) unsigned char tile_smem[];
    // layout: alias [256] u64 | cdf_e [256] uint4 | stage | st [sites] | tot [sites][4] | site_e [sites] |
    //         constant tables [nq] | class map [16][8] | per-warp scratch [warps][2 KB] | qs tables [512] (LUT) |
    //         chunk records | cnt [cap]
    constexpr int WST = 2 * TILE_WST_G + TILE_WST_R;
    constexpr int NQ_SMEM = MODE == 2 ? M2_TAB_MAXQ : 1;
    constexpr uint32_t OFF_STAGE = 2048 + 4096, OFF_ST = OFF_STAGE + TILE_WARPS * WST * 4, OFF_TOT = OFF_ST + TILE_MAX_SITES * sizeof(TSite),
                       OFF_SE = OFF_TOT + TILE_MAX_SITES * 16, OFF_TAB = OFF_SE + TILE_MAX_SITES * sizeof(M2SiteE),
                       OFF_CMAP = OFF_TAB + NQ_SMEM * M2_TAB_BYTES, OFF_SCR = OFF_CMAP + 512, OFF_QCLS = OFF_SCR + (MODE == 2 ? TILE_WARPS * M2_SCR_BYTES : 0),
                       OFF_CHK = OFF_QCLS + (MODE == 2 ? 2048 : 0), OFF_CNT = OFF_CHK + (BIG ? 0 : (TILE_CELLS / 32) * sizeof(M2Chunk));
    TSite* st = reinterpret_cast<TSite*>(tile_smem + OFF_ST);
    int* tot = reinterpret_cast<int*>(tile_smem + OFF_TOT);
    M2SiteE* site_e = reinterpret_cast<M2SiteE*>(tile_smem + OFF_SE);
    __shared__ int64_t s_base[4];
    __shared__ int s_next;
    __shared__ uint32_t s_ctr[4];
    __shared__ uint32_t s_mix[2];
    __shared__ uint32_t s_hist[72]; // two-base mixed cells per depth (0..64), then the running offsets of the counting sort
    __shared__ uint32_t s_zero[32];

    int tid, S;
    asm volatile("mov.u32 %0, %%tid.x;" : "=r"(tid));
    asm volatile("mov.u32 %0, %1;" : "=r"(S) : "r"(p.S));
    const int lane = tid & 31, warp = tid >> 5;
    const int S4 = (S + 3) & ~3, PAD = S4 - S, T = p.sites_per_tile;
    const uint32_t s_smem = smem_u32(tile_smem);
    for (int i = tid; i < 256; i += TILE_BLOCK) {
        reinterpret_cast<uint2*>(tile_smem)[i] = reinterpret_cast<const uint2*>(p.pois_alias)[i];
        reinterpret_cast<uint4*>(tile_smem + 2048)[i] = reinterpret_cast<const uint4*>(p.err_cdf)[i];
        if (MODE == 2) { // words 0..255: the conditional alias table of the minor classes, 256..511: class info words
            reinterpret_cast<uint32_t*>(tile_smem + OFF_QCLS)[i] = p.qcls[512 + i];
            reinterpret_cast<uint32_t*>(tile_smem + OFF_QCLS)[256 + i] = p.qcls[256 + i];
        }
    }
    for (int i = tid; i < TILE_MAX_SITES * 4; i += TILE_BLOCK) tot[i] = 0;
    if (TAB) {
        for (int i = tid; i < p.m2_nq * M2_TAB_DOUBLES; i += TILE_BLOCK) reinterpret_cast<double*>(tile_smem + OFF_TAB)[i] = p.m2_tab[i];
        for (int i = tid; i < 128; i += TILE_BLOCK) reinterpret_cast<uint32_t*>(tile_smem + OFF_CMAP)[i] = p.m2_cmap[i];
    }
    if (tid == 0) {
        s_next = (int)atomicAdd(p.ticket, 1u);
        s_ctr[0] = s_ctr[1] = s_ctr[2] = s_ctr[3] = 0u;
        s_mix[0] = s_mix[1] = 0u;
    }
    if (tid < 72) s_hist[tid] = 0u;
    if (tid < 32) s_zero[tid] = 0u;
    const uint32_t s_tab = s_smem + OFF_TAB, s_cmap = s_smem + OFF_CMAP;
    const uint32_t s_scrw = s_smem + OFF_SCR + warp * M2_SCR_BYTES + lane * 4; // this lane's column of the warp's scratch: word w at + 128 w
    M2Rng R;
    R.s_alias = s_smem;
    R.s_cdf_e = s_smem + 2048;
    R.s_qcls = s_smem + OFF_QCLS;
    R.fixed_depth = p.depth_mode == VGL_DEPTH_FIXED ? (int)p.depth_mean : -1;
    R.has_err = p.error_rate > 0.0;
    const uint32_t inv_s4 = (uint32_t)(((1ull << 32) + S4 - 1) / S4);
    const bool explode = p.do_unobserved >= 3;
    const bool add_unobs = p.do_unobserved == 1 || p.do_unobserved == 2 || p.do_unobserved == 4 || p.do_unobserved == 5;
    // GLPL: both the GL and the PL plane exist (compile time); else the plane tests are pinned in registers (the compiler would
    // otherwise re-read the kernel parameters for every one of the 15 stores of a cell)
    uint32_t plane_flags = (p.gl != nullptr ? 1u : 0u) | (p.pl != nullptr ? 2u : 0u) | (p.ad != nullptr ? 4u : 0u);
    asm volatile("mov.u32 %0, %0;" : "+r"(plane_flags));
    const bool has_gl = GLPL || (plane_flags & 1u), has_pl = GLPL || (plane_flags & 2u), has_ad = (plane_flags & 4u) != 0u;
    const bool pure_ok = TAB && p.m2_pure != nullptr;
    const uint32_t s_wg = s_smem + OFF_STAGE + warp * WST * 4;
    const uint32_t s_wr = s_wg + 2 * TILE_WST_G * 4;
    const uint32_t s_cnt = s_smem + OFF_CNT, s_st = s_smem + OFF_ST, s_chk = s_smem + OFF_CHK;
    // BIG: per-CTA rows in global memory: counts [S4] | chunk records [S4 / 32 + 1]
    uint32_t* const cnt_g = BIG ? p.cnt_scratch + (size_t)blockIdx.x * m2_big_row_words(S4) : nullptr;
    M2Chunk* const chk_g = BIG ? reinterpret_cast<M2Chunk*>(cnt_g + S4) : nullptr;
    // every variant: the CTA's row of parked results (16 floats per mixed cell) followed by the list of mixed cells (L2-resident)
    const int list_cap = BIG ? S4 : TILE_CELLS;
    float* const park = p.m2_park + (size_t)blockIdx.x * (size_t)list_cap * 18;
    uint32_t* const list_g = reinterpret_cast<uint32_t*>(park + (size_t)list_cap * 16);
    uint32_t* const sorted_g = list_g + list_cap; // the two-base cells ordered by depth: list position << 16 | virtual cell
    uint32_t s_ctrA = smem_u32(&s_ctr[0]), s_ctrC = smem_u32(&s_ctr[1]), s_ctrM = smem_u32(&s_ctr[2]), s_ctrN = smem_u32(&s_ctr[3]);
    bool first_tile = true;
    M2SiteE run_e;
    run_e.e = p.error_rate;
    run_e.l2 = 0.0f;
    run_e.er = 0.0f;
    const uint32_t dom_cls = (uint32_t)p.q_dom;          // LUT mode: the dominant class and its table offset

    auto list_put = [&](uint32_t pos, uint32_t iv) { __stcg(list_g + pos, iv); };
    auto list_get = [&](uint32_t pos) -> uint32_t { return __ldcg(list_g + pos); };

    for (;;) {
        __syncthreads();
        const int tile = s_next;
        if (tile >= p.n_tiles) break;
        if (first_tile) {
            const uint32_t opaque_zero = lds32(smem_u32(&s_zero[lane]));
            s_ctrA += opaque_zero;
            s_ctrC += opaque_zero;
            s_ctrM += opaque_zero;
            s_ctrN += opaque_zero;
            first_tile = false;
        }
        const int site0 = tile * T;
        const int nsl = min(T, p.n_sites - site0);
        const int nv = nsl * S4;
        const int nchunk = (nv + 31) >> 5;
        const int64_t cell0 = (int64_t)site0 * S;
        const uint8_t* __restrict__ gt_t = p.gt + cell0;
        int32_t* __restrict__ dp_t = p.dp + cell0;
        const unsigned long long site_base = (unsigned long long)(p.first_site + site0);

        if (MODE == 1) { // per-site beta-distributed base-picking error rate (vcfgl.cpp:425-437), same draw as cell_source.cuh
            if (tid < nsl) {
                const double e = m2_site_beta(p, site_base + (unsigned)tid);
                M2SiteE se;
                se.e = e;
                se.l2 = (e > 0.0 && e <= 0.5) ? log2f((float)(1.0 - e)) : 0.0f;
                se.er = (float)(e / (1.0 - e));
                site_e[tid] = se;
            }
            __syncthreads();
        }

        // ---------------- phase A: counts, FORMAT/DP, per-site base totals, the list of mixed cells
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
                uint32_t ad = 0u;
                int n = 0;
                if (real) {
                    uint32_t wseq[4];
                    ad = m2_cell_fixed<false, MODE == 1>(p, R, site_base + (uint32_t)sl, (uint32_t)v, gt, MODE == 1 ? site_e[sl] : run_e, n, wseq);
                    dp_t[(uint32_t)(iv - sl * PAD)] = n;
                }
                if (iv < nv) {
                    if (BIG) cnt_g[iv] = ad;
                    else sts32(s_cnt + (uint32_t)iv * 4u, ad);
                }
                // cell kind: pure (closed form), two-base mixed (six classes), general mixed (15 base pairs)
                {
                    const int nb = __popc(nonzero_bytes(ad));
                    bool pure = pure_ok && nb == 1 && n <= 64;
                    if (MODE == 2 && pure) { // every read of the dominant quality class?
                        const u32x4 q0 = philox_rk(p, (uint32_t)(site_base + (uint32_t)sl), (uint32_t)((site_base + (uint32_t)sl) >> 32) & 0xFFu, (uint32_t)v,
                                                   (uint32_t)P_QS << 24);
                        pure = m2_qs_minor_count(p, n, q0.x) == 0;
                    }
                    const bool mixed = n > 0 && !pure;
                    const bool two = mixed && TAB && nb <= 2 && n <= 64;
                    const uint32_t m2 = __ballot_sync(0xffffffffu, two), m15 = __ballot_sync(0xffffffffu, mixed && !two);
                    uint32_t b2 = 0u, b15 = 0u;
                    if (lane == 0) {
                        if (m2) b2 = atomicAdd(&s_mix[0], (uint32_t)__popc(m2));
                        if (m15) b15 = atomicAdd(&s_mix[1], (uint32_t)__popc(m15));
                        M2Chunk c;
                        c.base2 = b2; c.base15 = b15; c.mask2 = m2; c.mask15 = m15;
                        if (BIG) chk_g[cur] = c;
                        else *reinterpret_cast<M2Chunk*>(tile_smem + OFF_CHK + (size_t)cur * sizeof(M2Chunk)) = c;
                    }
                    b2 = __shfl_sync(0xffffffffu, b2, 0);
                    b15 = __shfl_sync(0xffffffffu, b15, 0);
                    const uint32_t lt = low_bits(lane);
                    if (two) {
                        list_put(b2 + (uint32_t)__popc(m2 & lt), (uint32_t)iv);
                        atomicAdd(&s_hist[n], 1u);
                    }
                    else if (mixed) list_put((uint32_t)list_cap - 1u - (b15 + (uint32_t)__popc(m15 & lt)), (uint32_t)iv);
                }
                // site totals (counts of one chunk stay below 2^16 per base: 32 cells x 255 reads)
                const int first = __shfl_sync(0xffffffffu, sl, 0);
                const uint32_t w01 = __byte_perm(ad, 0u, 0x4140), w23 = __byte_perm(ad, 0u, 0x4342);
                if (__all_sync(0xffffffffu, sl == first)) {
                    const uint32_t a01 = __reduce_add_sync(0xffffffffu, w01), a23 = __reduce_add_sync(0xffffffffu, w23);
                    if (lane < 4 && first < nsl) {
                        const uint32_t ww = (lane & 2) ? a23 : a01;
                        const uint32_t val = (lane & 1) ? (ww >> 16) : (ww & 0xFFFFu);
                        if (val) atomicAdd(&tot[first * 4 + lane], (int)val);
                    }
                } else if (sl < nsl) {
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const int val = (int)((ad >> (8 * b)) & 0xFFu);
                        if (val) atomicAdd(&tot[sl * 4 + b], val);
                    }
                }
                cur = nxt; iv = iv2; sl = sl2; v = v2; real = real2; gt = gt2;
                nxt = tile_ticket_get(raw);
            }
        }
        __syncthreads();

        // ---------------- phase B (warp 0): per-site record
        if (warp == 0) {
            if (lane == 0) {
                s_ctr[0] = 0u;
                s_next = (int)atomicAdd(p.ticket, 1u);
            }
            { // pull the next tile's genotypes into L2 while this tile is scored
                const int nt = __shfl_sync(0xffffffffu, lane == 0 ? s_next : 0, 0);
                const int64_t lo = (int64_t)nt * T * S + lane * 128;
                if (nt < p.n_tiles && lane * 128 < T * S && lo < p.n_cells) asm volatile("prefetch.global.L2 [%0];" ::"l"(p.gt + lo));
            }
            tile_phase_b(p, lane, nsl, site0, tile, S, T, tot, st, explode, add_unobs, s_base, s_ctr);
        } else if (warp == 1) { // counting sort of the two-base cells by depth: histogram -> exclusive offsets
            const uint32_t h0 = s_hist[lane], h1 = s_hist[32 + lane], h2 = lane == 0 ? s_hist[64] : 0u;
            uint32_t i0 = h0, i1 = h1;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const uint32_t t0 = __shfl_up_sync(0xffffffffu, i0, off), t1 = __shfl_up_sync(0xffffffffu, i1, off);
                if (lane >= off) { i0 += t0; i1 += t1; }
            }
            const uint32_t tot0 = __shfl_sync(0xffffffffu, i0, 31), tot1 = __shfl_sync(0xffffffffu, i1, 31);
            s_hist[lane] = i0 - h0;
            s_hist[32 + lane] = tot0 + i1 - h1;
            if (lane == 0) s_hist[64] = tot0 + tot1 + 0u * h2;
        }
        __syncthreads();
        if (p.zero_holes) tile_zero_holes(p, tid, nsl, S, s_base);

        // ---------------- phase M: the mixed cells, one per lane, in list order
        const int n_two = (int)s_mix[0], n_gen = (int)s_mix[1];
        auto cell_setup = [&](uint32_t iv, M2Reads<MODE>& rd, uint32_t& c4, uint32_t& pv, int& n) {
            const int sl = (int)__umulhi(iv, inv_s4), v = (int)iv - sl * S4;
            c4 = BIG ? cnt_g[iv] : lds32(s_cnt + iv * 4u);
            n = (int)__vsadu4(c4, 0u);
            const uint4 slot = lds128(s_st + (uint32_t)sl * 64u);
            pv = (nonzero_bytes(~slot.x) | (nonzero_bytes(~slot.y) << 4) | (nonzero_bytes(~slot.z) << 8) | (nonzero_bytes(~slot.w) << 12)) & 0x7FFFu;
            const uint32_t gt = gt_t[(uint32_t)((int)iv - sl * PAD)];
            rd.g0 = gt & 0x3;
            rd.g1 = (gt >> 4) & 0x3;
            rd.site = site_base + (uint32_t)sl;
            rd.sample = (uint32_t)v;
            rd.e = MODE == 1 ? site_e[sl].e : run_e.e;
            rd.deep = n > 64;
            rd.w0 = rd.w1 = rd.w2 = rd.w3 = rd.cur = 0u;
            if (!rd.deep) {
                int nn;
                uint32_t wseq[4];
                m2_cell_fixed<true, MODE == 1>(p, R, rd.site, (uint32_t)v, gt, MODE == 1 ? site_e[sl] : run_e, nn, wseq);
                rd.w0 = wseq[0]; rd.w1 = wseq[1]; rd.w2 = wseq[2]; rd.w3 = wseq[3];
            }
        };
        // LUT mode: the quality class of every read of the lane's cell (<= 64 reads) as bytes in the lane's scratch column
        auto qs_classes = [&](const M2Reads<MODE>& rd, int n, int nmax) {
            if (MODE != 2) return;
            const uint32_t fill = dom_cls * 0x01010101u;
            for (int w = 0; w * 4 < nmax && w < 16; ++w) sts32(s_scrw + 128u * (uint32_t)w, fill);
            if (n > 0 && n <= 64)
                m2_qs_minor_reads(p, R, rd.site, rd.sample, n, [&](uint32_t pos, uint32_t cls) {
                    asm volatile("st.shared.u8 [%0], %1;" ::"r"(s_scrw + 128u * (pos >> 2) + (pos & 3u)), "r"(cls) : "memory");
                });
        };
        auto read_qoff = [&](M2Reads<MODE>& rd, int i, int& qs) -> uint32_t { // table offset (and score) of read i's quality class
            qs = 0;
            if (MODE != 2) return 0u;
            uint32_t info;
            if (rd.deep) {
                info = m2_lut_qs(p, R, rd.site, rd.sample, i, rd.qblk);
            } else {
                uint32_t cls;
                asm volatile("ld.shared.u8 %0, [%1];" : "=r"(cls) : "r"(s_scrw + 128u * ((uint32_t)i >> 2) + ((uint32_t)i & 3u)));
                info = lds32(R.s_qcls + 1024u + cls * 4u);
                if (info & 0x200u) atomicExch(p.status, (int)VGL_ERANGE); // apply_qs_bins() -> ERROR, vcfgl.cpp:63
            }
            qs = (int)(info & 0xFFu);
            return ((info >> 16) & 0xFFu) * (uint32_t)M2_TAB_BYTES;
        };
        if (TAB) { // order the two-base cells by depth, so that the 32 cells a warp takes run read loops of (nearly) equal length
            for (int j = tid; j < n_two; j += TILE_BLOCK) {
                const uint32_t iv = list_get((uint32_t)j);
                const uint32_t c4 = BIG ? cnt_g[iv] : lds32(s_cnt + iv * 4u);
                const uint32_t pos = atomicAdd(&s_hist[__vsadu4(c4, 0u)], 1u);
                __stcg(sorted_g + pos, ((uint32_t)j << 16) | iv);
            }
            __syncthreads();
        }
        if (TAB) { // two-base cells: six classes {xx, xy, yy, x., y., ..}
            int g = tile_ticket_get(tile_ticket_issue(s_ctrM, lane));
            while (g * 32 < n_two) {
                const int raw = tile_ticket_issue(s_ctrM, lane);
                const bool act = g * 32 + lane < n_two;
                const uint32_t ent = act ? __ldcg(sorted_g + g * 32 + lane) : 0u;
                const int j = (int)(ent >> 16);
                M2Reads<MODE> rd;
                uint32_t c4 = 0u, pv = 0u;
                int n = 0;
                if (act) cell_setup(ent & 0xFFFFu, rd, c4, pv, n);
                else { rd.deep = false; rd.w0 = rd.w1 = rd.w2 = rd.w3 = rd.cur = 0u; rd.site = 0; rd.sample = 0; rd.g0 = rd.g1 = 0; rd.e = 0.0; }
                const int nmax = __reduce_max_sync(0xffffffffu, n);
                qs_classes(rd, n, nmax);
                const uint32_t seen = nonzero_bytes(c4);
                const int x = __ffs(seen | 16u) - 1, rest = seen & (seen - 1u);
                const int y = rest ? __ffs(rest) - 1 : ((x + 1) & 3);
                const uint32_t cm_ent = s_cmap + (uint32_t)(((x & 3) * 4 + y) * 32);
                const uint4 cm = lds128(cm_ent);
                const uint2 ids = lds64(cm_ent + 16u);
                float gc[6];
                gc[0] = (pv & cm.x & 0xFFFFu) ? -0.0f : -CUDART_INF_F;
                gc[1] = (pv & (cm.x >> 16)) ? -0.0f : -CUDART_INF_F;
                gc[2] = (pv & cm.y & 0xFFFFu) ? -0.0f : -CUDART_INF_F;
                gc[3] = (pv & (cm.y >> 16)) ? -0.0f : -CUDART_INF_F;
                gc[4] = (pv & cm.z & 0xFFFFu) ? -0.0f : -CUDART_INF_F;
                gc[5] = (pv & (cm.z >> 16)) ? -0.0f : -CUDART_INF_F;
                for (int i = 0; i < nmax; ++i) {
                    if (i < n) {
                        const int b = rd.base(p, i);
                        int qs;
                        const uint32_t qoff = read_qoff(rd, i, qs);
                        m2_update_classes(gc, s_tab + qoff + M2_TAB_CLS + (b == x ? 64u : 0u));
                    }
                }
                if (act) { // the 15 base pairs from the six classes, parked for phase C
                    const unsigned long long id64 = ((unsigned long long)ids.y << 32) | ids.x;
                    float gl[16];
#pragma unroll
                    for (int k = 0; k < 15; ++k) {
                        const uint32_t c = (uint32_t)((id64 >> (3 * k)) & 7ull);
                        gl[k] = c == 0 ? gc[0] : (c == 1 ? gc[1] : (c == 2 ? gc[2] : (c == 3 ? gc[3] : (c == 4 ? gc[4] : gc[5]))));
                    }
                    gl[15] = 0.0f;
                    float4* dst = reinterpret_cast<float4*>(park + (size_t)j * 16);
                    dst[0] = make_float4(gl[0], gl[1], gl[2], gl[3]);
                    dst[1] = make_float4(gl[4], gl[5], gl[6], gl[7]);
                    dst[2] = make_float4(gl[8], gl[9], gl[10], gl[11]);
                    dst[3] = make_float4(gl[12], gl[13], gl[14], gl[15]);
                }
                g = tile_ticket_get(raw);
            }
        }
        { // general cells: all 15 base pairs
            int g = tile_ticket_get(tile_ticket_issue(s_ctrN, lane));
            while (g * 32 < n_gen) {
                const int raw = tile_ticket_issue(s_ctrN, lane);
                const int j = g * 32 + lane;
                const bool act = j < n_gen;
                const uint32_t pos = (uint32_t)list_cap - 1u - (uint32_t)j;
                M2Reads<MODE> rd;
                uint32_t c4 = 0u, pv = 0u;
                int n = 0;
                if (act) cell_setup(list_get(pos), rd, c4, pv, n);
                else { rd.deep = false; rd.w0 = rd.w1 = rd.w2 = rd.w3 = rd.cur = 0u; rd.site = 0; rd.sample = 0; rd.g0 = rd.g1 = 0; rd.e = 0.0; }
                const int nmax = __reduce_max_sync(0xffffffffu, n);
                qs_classes(rd, n, min(nmax, 64));
                float gl[16];
#pragma unroll
                for (int k = 0; k < 15; ++k) gl[k] = ((pv >> k) & 1u) ? -0.0f : -CUDART_INF_F; // bcf_utils.h:310
                gl[15] = 0.0f;
                for (int i = 0; i < nmax; ++i) {
                    if (i < n) {
                        const int b = rd.base(p, i);
                        int qs;
                        const uint32_t qoff = read_qoff(rd, i, qs);
                        float (&g15)[15] = *reinterpret_cast<float (*)[15]>(gl);
                        if (TAB) {
                            m2_update_pairs(g15, s_tab + qoff + (uint32_t)b * 136u);
                        } else if (MODE == 2) {
                            m2_update(g15, b, __ldg(p.lut_log10 + qs), __ldg(p.lut_log10 + 257 + qs), __ldg(p.lut_log10 + 514 + qs));
                        } else {
                            m2_update(g15, b, p.homT, p.het, p.homF);
                        }
                    }
                }
                if (act) {
                    float4* dst = reinterpret_cast<float4*>(park + (size_t)pos * 16);
                    dst[0] = make_float4(gl[0], gl[1], gl[2], gl[3]);
                    dst[1] = make_float4(gl[4], gl[5], gl[6], gl[7]);
                    dst[2] = make_float4(gl[8], gl[9], gl[10], gl[11]);
                    dst[3] = make_float4(gl[12], gl[13], gl[14], gl[15]);
                }
                g = tile_ticket_get(raw);
            }
        }
        __syncthreads(); // parked values are visible to the CTA (global memory, same CTA: the barrier orders them)
        if (tid == 0) { s_ctr[2] = s_ctr[3] = 0u; s_mix[0] = s_mix[1] = 0u; }
        if (tid < 72) s_hist[tid] = 0u;

        // ---------------- phase C: assemble + emit, one warp per chunk of 32 virtual cells
        float* const gl_t = has_gl ? p.gl + s_base[0] : nullptr;
        int32_t* const pl_t = has_pl ? p.pl + s_base[0] : nullptr;
        int32_t* const ad_t = has_ad ? p.ad + s_base[1] : nullptr;
        int cur = tile_ticket_get(tile_ticket_issue(s_ctrC, lane));
        for (; cur < nchunk;) {
            const int raw = tile_ticket_issue(s_ctrC, lane);
            const int iv = cur * 32 + lane;
            const uint32_t c4 = iv < nv ? (BIG ? cnt_g[iv] : lds32(s_cnt + (uint32_t)iv * 4u)) : 0u;
            M2Chunk ck;
            if (BIG) ck = chk_g[cur];
            else {
                const uint4 t = lds128(s_chk + (uint32_t)cur * 16u);
                ck.base2 = t.x; ck.base15 = t.y; ck.mask2 = t.z; ck.mask15 = t.w;
            }
            // parked values of a mixed cell: issue the loads first
            const uint32_t lt = low_bits(lane);
            const bool is2 = (ck.mask2 >> lane) & 1u, is15 = (ck.mask15 >> lane) & 1u;
            float4 pk0, pk1, pk2, pk3;
            pk0 = pk1 = pk2 = pk3 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (is2 || is15) {
                const uint32_t pos = is2 ? ck.base2 + (uint32_t)__popc(ck.mask2 & lt) : (uint32_t)list_cap - 1u - (ck.base15 + (uint32_t)__popc(ck.mask15 & lt));
                const float4* src = reinterpret_cast<const float4*>(park + (size_t)pos * 16);
                pk0 = __ldcg(src); pk1 = __ldcg(src + 1); pk2 = __ldcg(src + 2); pk3 = __ldcg(src + 3);
            }
            int sl = (int)__umulhi((uint32_t)iv, inv_s4);
            int v = iv - sl * S4;
            if (sl >= nsl) { sl = nsl - 1; v = S4; }
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
            const uint32_t cell_g = live ? s_wg + (uint32_t)(gpos - g_lo) * 4u : s_wg + TILE_G_TRASH * 4u;
            const uint32_t cell_r = live ? s_wr + (uint32_t)(rpos - r_lo) * 4u : s_wr + TILE_R_TRASH * 4u;
            const uint4 slot = lds128(s_st + (uint32_t)sl * 64u);
            const int n = (int)__vsadu4(c4, 0u);
            float gl[15];
            if (is2 || is15) {
                gl[0] = pk0.x; gl[1] = pk0.y; gl[2] = pk0.z; gl[3] = pk0.w;
                gl[4] = pk1.x; gl[5] = pk1.y; gl[6] = pk1.z; gl[7] = pk1.w;
                gl[8] = pk2.x; gl[9] = pk2.y; gl[10] = pk2.z; gl[11] = pk2.w;
                gl[12] = pk3.x; gl[13] = pk3.y; gl[14] = pk3.z;
            } else { // pure cell (or no reads: overwritten below): +0 for xx, the table's two values for x? and ??
                const int x = __ffs(nonzero_bytes(c4) | 16u) - 1;
                float2 tv = make_float2(0.f, 0.f);
                if (pure_ok) tv = __ldg(reinterpret_cast<const float2*>(p.m2_pure) + (MODE == 2 ? p.q_dom_idx * 65 : 0) + min(n, 64));
                const uint32_t hom = m2_hom_bit(x & 3), het = m2_het_mask(x & 3);
#pragma unroll
                for (int k = 0; k < 15; ++k) gl[k] = ((hom >> k) & 1u) ? 0.0f : (((het >> k) & 1u) ? tv.x : tv.y);
            }
            bulk_wait_read();
            __syncwarp();
            m2_emit_cell(gl, slot, cell_g, has_gl, has_pl);
            if (has_ad) {
                sts32(cell_r, __byte_perm(c4, 0u, t2.x));
                if (A > 1) sts32(cell_r + 4, __byte_perm(c4, 0u, t2.x >> 16));
                if (A > 2) sts32(cell_r + 8, __byte_perm(c4, 0u, t2.y));
                if (A > 3) sts32(cell_r + 12, __byte_perm(c4, 0u, t2.y >> 16));
                if (A > 4) sts32(cell_r + 16, __byte_perm(c4, 0u, t1.w));
            }
            if (live && n == 0) { // gl_methods.cpp:60-66
#pragma unroll 1
                for (int g = 0; g < G; ++g) {
                    sts32(cell_g + 4 * g, VGL_F32_MISSING_BITS);
                    sts32(cell_g + 4 * (TILE_WST_G + g), (uint32_t)VGL_I32_MISSING);
                }
            }
            if (v == S && G > 0) {
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
            if (lane == 0) {
                const uint32_t gb = (uint32_t)(g_hi - g_lo) * 4u, rb = (uint32_t)(r_hi - r_lo) * 4u;
                if (gb) {
                    if (has_gl) bulk_store(gl_t + g_lo, s_wg, gb);
                    if (has_pl) bulk_store(pl_t + g_lo, s_wg + TILE_WST_G * 4, gb);
                }
                if (rb && has_ad) bulk_store(ad_t + r_lo, s_wr, rb);
                bulk_commit();
            }
            cur = tile_ticket_get(raw);
        }
    }
    bulk_wait_all();
    if (tid == 0) {
        const unsigned done = atomicAdd(p.ticket + 1, 1u);
        if (done == gridDim.x - 1) {
            p.ticket[0] = 0u;
            p.ticket[1] = 0u;
        }
    }
}

template <int MODE>
static size_t tile_m2_dyn_smem(bool big)
{
    return 2048 + 4096 + (size_t)TILE_WARPS * (2 * TILE_WST_G + TILE_WST_R) * 4 + TILE_MAX_SITES * sizeof(TSite) + TILE_MAX_SITES * 16 +
           TILE_MAX_SITES * sizeof(M2SiteE) + (MODE == 2 ? M2_TAB_MAXQ : 1) * M2_TAB_BYTES + 512 + (MODE == 2 ? TILE_WARPS * M2_SCR_BYTES : 0) +
           (MODE == 2 ? 2048 : 0) + (big ? 0 : (size_t)(TILE_CELLS / 32) * sizeof(M2Chunk) + (size_t)TILE_CELLS * 4);
}

template <int MODE, bool BIG, bool TAB, bool GLPL>
static int tile_m2_ctas_per_sm()
{
    const size_t dyn = tile_m2_dyn_smem<MODE>(BIG);
    cudaFuncSetAttribute(k_tile_m2<MODE, BIG, TAB, GLPL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    cudaFuncSetAttribute(k_tile_m2<MODE, BIG, TAB, GLPL>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_tile_m2<MODE, BIG, TAB, GLPL>, TILE_BLOCK, dyn);
    if (per_sm < 1) per_sm = 1;
    if (per_sm > TILE_SCRATCH_CTAS_PER_SM) per_sm = TILE_SCRATCH_CTAS_PER_SM;
    return per_sm;
}

template <int MODE, bool BIG, bool TAB, bool GLPL>
static void launch_tile_m2_g(const DevParams& p, cudaStream_t st, int n_sms)
{
    const size_t dyn = tile_m2_dyn_smem<MODE>(BIG);
    int grid = n_sms * tile_m2_ctas_per_sm<MODE, BIG, TAB, GLPL>();
    if (grid > p.n_tiles) grid = p.n_tiles;
    k_tile_m2<MODE, BIG, TAB, GLPL><<<grid, TILE_BLOCK, dyn, st>>>(p);
}
template <int MODE, bool BIG, bool TAB>
static void launch_tile_m2_t(const DevParams& p, cudaStream_t st, int n_sms)
{
    if (p.gl && p.pl) launch_tile_m2_g<MODE, BIG, TAB, true>(p, st, n_sms);
    else launch_tile_m2_g<MODE, BIG, TAB, false>(p, st, n_sms);
}

// mode: 0 FIXED / run-constant error rate, 1 FIXED / per-site error rate, 2 LUT (per-read quality scores)
void launch_tile_m2(const DevParams& p, cudaStream_t st, int n_sms, int mode)
{
    const bool big = tile_m1f_scratch_words(p.S, 1) > 0, tab = p.m2_tab != nullptr && p.m2_nq <= M2_TAB_MAXQ;
    if (mode == 0) { if (big) launch_tile_m2_t<0, true, true>(p, st, n_sms); else launch_tile_m2_t<0, false, true>(p, st, n_sms); }
    else if (mode == 1) { if (big) launch_tile_m2_t<1, true, true>(p, st, n_sms); else launch_tile_m2_t<1, false, true>(p, st, n_sms); }
    else if (tab) { if (big) launch_tile_m2_t<2, true, true>(p, st, n_sms); else launch_tile_m2_t<2, false, true>(p, st, n_sms); }
    else { if (big) launch_tile_m2_t<2, true, false>(p, st, n_sms); else launch_tile_m2_t<2, false, false>(p, st, n_sms); }
}

// global scratch of the model-2 tile kernel for S samples on n_sms SMs: 32-bit words of the per-CTA rows (counts, list, chunk
// records; 0 unless a site exceeds the shared-memory tile) and floats of the parked results (16 per cell of a tile)
size_t tile_m2_row_words(int S, int n_sms)
{
    const int S4 = (S + 3) & ~3;
    return S4 > TILE_CELLS ? m2_big_row_words(S4) * TILE_SCRATCH_CTAS_PER_SM * (size_t)n_sms : 0;
}
size_t tile_m2_park_floats(int S, int n_sms)
{
    const int S4 = (S + 3) & ~3;
    return (size_t)(S4 > TILE_CELLS ? S4 : TILE_CELLS) * 18 * TILE_SCRATCH_CTAS_PER_SM * (size_t)n_sms; // + two list words per cell
}

// ---- the sampler's per-read draws in the replay layout (vgl_native_draws): pass 0 writes the depths, pass 1 the reads
__global__ void k_tile_m2_draws(const DevParams p, int mode, int pass, int32_t* depths, const int64_t* off, uint8_t* bases, uint8_t* qs,
                                double* eprob)
{
    __shared__ __align__(16) unsigned char sm[2048 + 4096 + 2048];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        reinterpret_cast<uint2*>(sm)[i] = reinterpret_cast<const uint2*>(p.pois_alias)[i];
        reinterpret_cast<uint4*>(sm + 2048)[i] = reinterpret_cast<const uint4*>(p.err_cdf)[i];
        if (mode == 2) {
            reinterpret_cast<uint32_t*>(sm + 6144)[i] = p.qcls[512 + i];
            reinterpret_cast<uint32_t*>(sm + 6144)[256 + i] = p.qcls[256 + i];
        }
    }
    __syncthreads();
    M2Rng R;
    R.s_alias = smem_u32(sm);
    R.s_cdf_e = R.s_alias + 2048;
    R.s_qcls = R.s_alias + 6144;
    R.fixed_depth = p.depth_mode == VGL_DEPTH_FIXED ? (int)p.depth_mean : -1;
    R.has_err = p.error_rate > 0.0;
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.n_cells) return;
    const int64_t sl = c / p.S;
    const uint32_t sample = (uint32_t)(c - sl * p.S);
    const unsigned long long site = (unsigned long long)(p.first_site + sl);
    const uint32_t gt = p.gt[c];
    const int g0 = gt & 0x3, g1 = (gt >> 4) & 0x3;
    M2SiteE se;
    se.e = p.error_rate;
    se.l2 = se.er = 0.0f;
    if (mode == 1) {
        const double e = m2_site_beta(p, site);
        se.e = e;
        se.l2 = (e > 0.0 && e <= 0.5) ? log2f((float)(1.0 - e)) : 0.0f;
        se.er = (float)(e / (1.0 - e));
    }
    int n;
    uint32_t w[4];
    if (mode == 1) m2_cell_fixed<true, true>(p, R, site, sample, gt, se, n, w);
    else m2_cell_fixed<true, false>(p, R, site, sample, gt, se, n, w);
    if (pass == 0) { depths[c] = n; return; }
    for (int i = 0; i < n; ++i) {
        int b;
        if (n > 64) b = m2_deep_base(p, site, sample, i, g0, g1, se.e);
        else b = (int)((w[i >> 4] >> (2 * (i & 15))) & 3u);
        bases[off[c] + i] = (uint8_t)b;
        if (mode == 1) eprob[off[c] + i] = se.e; // the site's error rate
    }
    if (mode == 2) {
        if (n > 64) {
            u32x4 qblk;
            for (int i = 0; i < n; ++i) qs[off[c] + i] = (uint8_t)(m2_lut_qs(p, R, site, sample, i, qblk) & 0xFFu);
        } else {
            const uint8_t qd = (uint8_t)(lds32(R.s_qcls + 1024u + (uint32_t)p.q_dom * 4u) & 0xFFu);
            for (int i = 0; i < n; ++i) qs[off[c] + i] = qd;
            uint8_t* const q0 = qs + off[c];
            const uint32_t s_info = R.s_qcls + 1024u;
            int32_t* const status = p.status;
            m2_qs_minor_reads(p, R, site, sample, n, [&](uint32_t pos, uint32_t cls) {
                const uint32_t info = lds32(s_info + cls * 4u);
                if (info & 0x200u) atomicExch(status, (int)VGL_ERANGE);
                q0[pos] = (uint8_t)(info & 0xFFu);
            });
        }
    }
}

void launch_tile_m2_draws(const DevParams& p, cudaStream_t st, int mode, int pass, int32_t* depths, const int64_t* off, uint8_t* bases, uint8_t* qs,
                          double* eprob)
{
    const unsigned grid = (unsigned)((p.n_cells + 127) / 128);
    k_tile_m2_draws<<<grid, 128, 0, st>>>(p, mode, pass, depths, off, bases, qs, eprob);
}

} // namespace vgl
