// Hand-written sm_100a kernels of the vcfgl simulate-and-score hot path.
//
//   k_sim   one thread per (site, sample) cell: depth, reads, per-base counts
//           (reference: vcfgl.cpp:364-389, 441-640; rng.h:284-351)
//   k_site  one warp per site: INFO/DP, INFO/AD*, allele order, unobserved allele,
//           skip codes, QS, I16 (vcfgl.cpp:396-404, 647-782, 845-898, 982-1074)
//   k_scan  one CTA: exclusive scan of the per-site FORMAT block sizes
//   k_emit  one thread per cell: genotype likelihoods (gl_methods.cpp +
//           htslib/errmod.c:143-208), PL, GP, AD/ADF/ADR in allele order
//           (vcfgl.cpp:806-843, 907-970), staged per CTA in shared memory and
//           written with 128-bit stores
//
// HBM-bound integer/fp work: no tensor cores.  All arithmetic whose rounding
// is visible in the reference's output uses explicit _rn intrinsics so that
// nvcc cannot contract it into FMAs (the reference is plain x86-64 SSE2).
#include "cell_source.cuh"
#include "m1f.cuh"

namespace vgl {

// ==========================================================================
// k_sim
// ==========================================================================
__global__ void __launch_bounds__(VGL_BLOCK) k_sim(const __grid_constant__ DevParams p)
{
    const int64_t c = (int64_t)blockIdx.x * VGL_BLOCK + threadIdx.x;
    if (c >= p.n_cells) return;
    const uint8_t gt = p.gt[c];
    CellSource cs;
    cs.init(p, c, gt);
    int n = 0;
    // a missing genotype discards the drawn depth (vcfgl.cpp:371-379)
    if ((gt & 0xF) != VGL_GT_MISSING && (gt >> 4) != VGL_GT_MISSING) n = cs.depth(p);
    if (n > 65535) n = 65535;
    uint64_t ad = 0, fwd = 0;
    int q0 = 0, q1 = 0, q2 = 0, q3 = 0, s0 = 0, s1 = 0, s2 = 0, s3 = 0;
    uint32_t tsum = 0, tsq = 0;
    int last = -1;
    const bool qsum_adj = (p.adjust_qs & 2) != 0;
    for (int i = 0; i < n; ++i) {
        const Read r = cs.read(p, i);
        const int sh = 16 * r.base;
        ad += 1ull << sh;
        if (p.sample_strand && r.strand == 0) fwd += 1ull << sh;
        if (p.need_cellq) { // vcfgl.cpp:557-564
            const int q = qsum_adj ? r.adjqs : r.qs;
            const int q2v = qs_squared(q);
            q0 += r.base == 0 ? q : 0; s0 += r.base == 0 ? q2v : 0;
            q1 += r.base == 1 ? q : 0; s1 += r.base == 1 ? q2v : 0;
            q2 += r.base == 2 ? q : 0; s2 += r.base == 2 ? q2v : 0;
            q3 += r.base == 3 ? q : 0; s3 += r.base == 3 ? q2v : 0;
        }
        if (p.need_tail) {
            tsum += (uint32_t)r.tail;
            tsq += (uint32_t)(r.tail * r.tail);
            last = r.base;
        }
    }
    p.dp[c] = n;
    uint4 rec;
    rec.x = (uint32_t)ad; rec.y = (uint32_t)(ad >> 32);
    rec.z = (uint32_t)fwd; rec.w = (uint32_t)(fwd >> 32);
    reinterpret_cast<uint4*>(p.cell)[c] = rec;
    if (p.need_cellq) {
        int4* q = reinterpret_cast<int4*>(p.cellq + c);
        q[0] = make_int4(q0, q1, q2, q3);
        q[1] = make_int4(s0, s1, s2, s3);
    }
    if (p.need_tail) {
        uint4 t;
        t.x = tsum; t.y = tsq; t.z = (uint32_t)last; t.w = 0;
        reinterpret_cast<uint4*>(p.celltail)[c] = t;
    }
}

// ==========================================================================
// k_draws: write every read of the native simulator out (pileup / self-replay support,
// reference: -printPileup vcfgl.cpp:616-634 exposes the same per-read data)
// ==========================================================================
__global__ void __launch_bounds__(VGL_BLOCK) k_draws(const __grid_constant__ DevParams p, const int64_t* __restrict__ off,
                                                     uint8_t* bases, uint8_t* strands, uint8_t* qs, uint8_t* adjqs,
                                                     uint8_t* tails, double* eprob)
{
    const int64_t c = (int64_t)blockIdx.x * VGL_BLOCK + threadIdx.x;
    if (c >= p.n_cells) return;
    const int n = p.dp[c];
    if (n == 0) return;
    CellSource cs;
    cs.init(p, c, p.gt[c]);
    const int64_t o = off[c];
    for (int i = 0; i < n; ++i) {
        const Read r = cs.read(p, i);
        bases[o + i] = (uint8_t)r.base;
        strands[o + i] = (uint8_t)r.strand;
        tails[o + i] = (uint8_t)r.tail;
        if (p.error_qs == 2) {
            qs[o + i] = (uint8_t)(r.qs < 0 ? 0 : r.qs);
            adjqs[o + i] = (uint8_t)(r.adjqs < 0 ? 0 : r.adjqs);
            eprob[o + i] = r.eprob;
        } else if (p.error_qs == 1) {
            eprob[o + i] = cs.e_pick; // the site's error rate
        }
    }
}

void launch_draws(const DevParams& p, cudaStream_t st, const int64_t* off, uint8_t* bases, uint8_t* strands, uint8_t* qs,
                  uint8_t* adjqs, uint8_t* tails, double* eprob)
{
    const unsigned grid = (unsigned)((p.n_cells + VGL_BLOCK - 1) / VGL_BLOCK);
    k_draws<<<grid, VGL_BLOCK, 0, st>>>(p, off, bases, strands, qs, adjqs, tails, eprob);
}

// ==========================================================================
// k_site
// ==========================================================================
__device__ __forceinline__ int warp_sum(int v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// v += c, k times, as the reference's float accumulator would (vcfgl.cpp:1009-1022)
__device__ __forceinline__ float add_const_times(float v, int c, int k)
{
    const float cf = (float)c;
    if (v + (float)k * cf < 16777216.0f && v == truncf(v)) return v + (float)(k * c); // all partial sums exact
    for (int i = 0; i < k; ++i) v = __fadd_rn(v, cf);
    return v;
}

struct CellQs {
    int qsum[4], qsumsq[4];
};

__device__ __forceinline__ CellQs load_cellq(const DevParams& p, int64_t c)
{
    CellQs o;
    if (p.need_cellq) {
        const int4* q = reinterpret_cast<const int4*>(p.cellq + c);
        const int4 a = q[0], b = q[1];
        o.qsum[0] = a.x; o.qsum[1] = a.y; o.qsum[2] = a.z; o.qsum[3] = a.w;
        o.qsumsq[0] = b.x; o.qsumsq[1] = b.y; o.qsumsq[2] = b.z; o.qsumsq[3] = b.w;
    } else { // one qs for every read (vcfgl.cpp:566-576)
        const int q = (p.adjust_qs & 2) ? p.pre_adj_qs : p.pre_qs;
        const int q2 = qs_squared(q);
        const CellRec r = p.cell[c];
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            o.qsum[b] = q * (int)r.ad[b];
            o.qsumsq[b] = q2 * (int)r.ad[b];
        }
    }
    return o;
}

__global__ void __launch_bounds__(VGL_BLOCK) k_site(const __grid_constant__ DevParams p)
{
    const int lane = threadIdx.x & 31;
    const int sl = (int)(((int64_t)blockIdx.x * VGL_BLOCK + threadIdx.x) >> 5);
    if (sl >= p.n_sites) return;
    const int S = p.S;
    const int64_t c0 = (int64_t)sl * S;

    int dp = 0, ad[4] = {0, 0, 0, 0}, fw[4] = {0, 0, 0, 0};
    for (int s = lane; s < S; s += 32) {
        dp += p.dp[c0 + s];
        const CellRec r = p.cell[c0 + s];
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            ad[b] += r.ad[b];
            fw[b] += r.fwd[b];
        }
    }
    dp = warp_sum(dp);
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        ad[b] = warp_sum(ad[b]);
        fw[b] = warp_sum(fw[b]);
    }
    if (lane != 0) return;

    vgl_site_out o;
    o.skip_code = 0;
    o.n_alleles = o.n_alleles_observed = o.n_genotypes = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) o.alleles2acgt[i] = o.acgt2alleles[i] = -1;
    o.info_dp = dp;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        o.info_ad[i] = o.info_adf[i] = o.info_adr[i] = 0;
        o.qs[i] = 0.0f;
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) o.i16[i] = 0.0f;
    o._pad = 0;
    o.g_off = o.r_off = 0;

    if (dp == 0) {
        // vcfgl.cpp:396-404 + simulate_site_with_no_reads (vcfgl.cpp:228-315)
        if (p.rm_empty) {
            o.skip_code = -4;
        } else if (!p.do_gvcf) {
            if (p.do_unobserved <= 2) { o.n_alleles = 1; o.n_genotypes = 1; o.n_alleles_observed = 0; }
            else if (p.do_unobserved == 3) { o.n_alleles = 4; o.n_genotypes = 10; o.n_alleles_observed = 4; }
            else { o.n_alleles = 5; o.n_genotypes = 15; o.n_alleles_observed = 4; }
        }
    } else {
        int n_obs = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) n_obs += ad[b] > 0;
        if (p.rm_invar_sim && n_obs == 1) { // vcfgl.cpp:675-681
            o.skip_code = -3;
        } else {
            // stable descending order of A,C,G,T by INFO/AD (vcfgl.cpp:700-718)
            const bool explode = p.do_unobserved >= 3;
            int n_alleles = 0;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                int rank = 0;
#pragma unroll
                for (int x = 0; x < 4; ++x) rank += (ad[x] > ad[b]) || (ad[x] == ad[b] && x < b);
                if (ad[b] > 0 || explode) { // unobserved bases are dropped unless exploded (vcfgl.cpp:722-735)
                    o.acgt2alleles[b] = (int8_t)rank;
                    o.alleles2acgt[rank] = (int8_t)b;
                    ++n_alleles;
                }
            }
            o.n_alleles_observed = n_alleles;
            const bool add_unobs = p.do_unobserved == 1 || p.do_unobserved == 2 || p.do_unobserved == 4 || p.do_unobserved == 5;
            if (add_unobs) { // vcfgl.cpp:756-762
                o.alleles2acgt[n_alleles] = 4;
                o.acgt2alleles[4] = (int8_t)n_alleles;
                ++n_alleles;
            }
            o.n_alleles = n_alleles;
            o.n_genotypes = n_alleles * (n_alleles + 1) / 2;
            const int A = n_alleles;
            // INFO/AD, ADF, ADR (vcfgl.cpp:833-841)
            for (int a = 0; a < A; ++a) {
                const int b = o.alleles2acgt[a];
                if (b < 0 || b == 4) continue;
                if (p.tag_mask & VGL_TAG_INFO_AD) o.info_ad[a] = ad[b];
                if (p.tag_mask & VGL_TAG_INFO_ADF) o.info_adf[a] = fw[b];
                if (p.tag_mask & VGL_TAG_INFO_ADR) o.info_adr[a] = ad[b] - fw[b];
            }
            // QS: per-sample normalised quality sums, float, sample order (vcfgl.cpp:845-898)
            if (p.tag_mask & VGL_TAG_QS) {
                for (int s = 0; s < S; ++s) {
                    const CellQs q = load_cellq(p, c0 + s);
                    float sum = 0.0f;
#pragma unroll
                    for (int b = 0; b < 4; ++b) sum = __fadd_rn(sum, (float)q.qsum[b]);
                    if (sum != 0.0f) {
#pragma unroll
                        for (int b = 0; b < 4; ++b) {
                            const int a = o.acgt2alleles[b];
                            if (a < 0) continue;
                            o.qs[a] = __fadd_rn(o.qs[a], __fdiv_rn((float)q.qsum[b], sum));
                        }
                    }
                }
            }
            // I16 (vcfgl.cpp:982-1074)
            if (p.tag_mask & VGL_TAG_I16) {
                float* v = o.i16;
                const int refb = o.alleles2acgt[0];
                // tail distances: every read's value lands on the base of the site's LAST read
                // (stale r_base, vcfgl.cpp:657-658); float accumulation in read order
                float tsum = 0.0f, tsq = 0.0f;
                int stale = -1;
                {
                    uint64_t isum = 0, isq = 0;
                    for (int s = 0; s < S; ++s) {
                        const CellTail t = p.celltail[c0 + s];
                        isum += t.sum;
                        isq += t.sumsq;
                        if (t.last_base >= 0) stale = t.last_base;
                    }
                    if (isq < 16777216ull) { // every partial sum is an exactly representable integer
                        tsum = (float)isum;
                        tsq = (float)isq;
                    } else {
                        for (int s = 0; s < S; ++s) {
                            const int64_t c = c0 + s;
                            const int n = p.dp[c];
                            if (n == 0) continue;
                            CellSource cs;
                            cs.init(p, c, p.gt[c]);
                            for (int i = 0; i < n; ++i) {
                                const int t = cs.read(p, i).tail;
                                tsum = __fadd_rn(tsum, (float)t);
                                tsq = __fadd_rn(tsq, (float)(t * t));
                            }
                        }
                    }
                }
                v[0] = (float)fw[refb];
                v[1] = (float)(ad[refb] - fw[refb]);
                const int mq = p.i16_mapq, mq2 = mq * mq;
                for (int s = 0; s < S; ++s) {
                    const CellQs q = load_cellq(p, c0 + s);
                    v[4] = __fadd_rn(v[4], (float)q.qsum[refb]);
                    v[5] = __fadd_rn(v[5], (float)q.qsumsq[refb]);
                    const CellRec r = p.cell[c0 + s];
                    for (int a = 0; a < A; ++a) {
                        if (a == o.n_alleles_observed) continue; // the unobserved allele has no mapq
                        const int b = o.alleles2acgt[a];
                        if (b < 0 || b == 4) continue;
                        const int k = r.ad[b];
                        if (a == 0) { v[8] = add_const_times(v[8], mq, k); v[9] = add_const_times(v[9], mq2, k); }
                        else        { v[10] = add_const_times(v[10], mq, k); v[11] = add_const_times(v[11], mq2, k); }
                    }
                }
                v[12] = refb == stale ? tsum : 0.0f;
                v[13] = refb == stale ? tsq : 0.0f;
                for (int a = 1; a < A; ++a) {
                    if (a == o.n_alleles_observed) continue;
                    const int b = o.alleles2acgt[a];
                    if (b < 0 || b == 4) continue;
                    v[2] = __fadd_rn(v[2], (float)fw[b]);
                    v[3] = __fadd_rn(v[3], (float)(ad[b] - fw[b]));
                    for (int s = 0; s < S; ++s) {
                        const CellQs q = load_cellq(p, c0 + s);
                        v[6] = __fadd_rn(v[6], (float)q.qsum[b]);
                        v[7] = __fadd_rn(v[7], (float)q.qsumsq[b]);
                    }
                    v[14] = __fadd_rn(v[14], b == stale ? tsum : 0.0f);
                    v[15] = __fadd_rn(v[15], b == stale ? tsq : 0.0f);
                }
            }
        }
    }
    // block sizes (in 4-byte elements, padded to 16 B) go through g_off/r_off into the scan
    if (o.skip_code == 0) {
        o.g_off = (((int64_t)S * o.n_genotypes) + 3) & ~3ll;
        o.r_off = (((int64_t)S * o.n_alleles) + 3) & ~3ll;
    }
    p.sites[sl] = o;
    if (p.pairmap) {
        int b2a[5];
#pragma unroll
        for (int i = 0; i < 5; ++i) b2a[i] = o.acgt2alleles[i];
        p.pairmap[sl] = make_pairmap(b2a);
    }
}

// ==========================================================================
// k_scan: exclusive scan of the per-site block sizes (single CTA, 1024 threads)
// ==========================================================================
__global__ void __launch_bounds__(1024) k_scan(const __grid_constant__ DevParams p)
{
    __shared__ int64_t wsum_g[32], wsum_r[32];
    __shared__ int64_t carry_g, carry_r;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) carry_g = carry_r = 0;
    __syncthreads();
    for (int base = 0; base < p.n_sites; base += 1024) {
        const int i = base + tid;
        int64_t g = 0, r = 0;
        if (i < p.n_sites) {
            g = p.sites[i].g_off;
            r = p.sites[i].r_off;
        }
        int64_t ig = g, ir = r; // inclusive warp scan
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t tg = __shfl_up_sync(0xffffffffu, ig, o);
            const int64_t tr = __shfl_up_sync(0xffffffffu, ir, o);
            if (lane >= o) { ig += tg; ir += tr; }
        }
        if (lane == 31) { wsum_g[wid] = ig; wsum_r[wid] = ir; }
        __syncthreads();
        if (wid == 0) {
            int64_t wg = wsum_g[lane], wr = wsum_r[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int64_t tg = __shfl_up_sync(0xffffffffu, wg, o);
                const int64_t tr = __shfl_up_sync(0xffffffffu, wr, o);
                if (lane >= o) { wg += tg; wr += tr; }
            }
            wsum_g[lane] = wg;
            wsum_r[lane] = wr;
        }
        __syncthreads();
        const int64_t pre_g = carry_g + (wid ? wsum_g[wid - 1] : 0);
        const int64_t pre_r = carry_r + (wid ? wsum_r[wid - 1] : 0);
        if (i < p.n_sites) {
            p.sites[i].g_off = pre_g + ig - g;
            p.sites[i].r_off = pre_r + ir - r;
        }
        __syncthreads();
        if (tid == 0) {
            carry_g += wsum_g[31];
            carry_r += wsum_r[31];
        }
        __syncthreads();
    }
    if (tid == 0) {
        p.totals[0] = carry_g;
        p.totals[1] = carry_r;
    }
}

// ==========================================================================
// k_emit
// ==========================================================================
struct SiteView {
    int A, G, n_obs_alleles, skip;
    int a2b[5]; // alleles2acgt
    int b2a[5]; // acgt2alleles
    int64_t g_off, r_off;
};

__device__ __forceinline__ int gt_index(int a, int b) { return a > b ? a * (a + 1) / 2 + b : b * (b + 1) / 2 + a; }

// CTA-wide: copy a staged span [lo, hi) of 4-byte elements (element index space of `plane`) from
// shared memory to global memory; stage[i] holds element (base + i), base % 4 == 0.
__device__ __forceinline__ void store_span(uint32_t* __restrict__ plane, const uint32_t* stage, int64_t base, int64_t lo, int64_t hi)
{
    const int n_chunks = (int)((hi - base + 3) >> 2);
    for (int ch = threadIdx.x; ch < n_chunks; ch += VGL_BLOCK) {
        const int64_t e = base + 4ll * ch;
        const uint4 v = *reinterpret_cast<const uint4*>(stage + 4 * ch);
        if (e >= lo && e + 4 <= hi) {
            *reinterpret_cast<uint4*>(plane + e) = v; // 128-bit store, 16 B aligned
        } else {
            if (e + 0 >= lo && e + 0 < hi) plane[e + 0] = v.x;
            if (e + 1 >= lo && e + 1 < hi) plane[e + 1] = v.y;
            if (e + 2 >= lo && e + 2 < hi) plane[e + 2] = v.z;
            if (e + 3 >= lo && e + 3 < hi) plane[e + 3] = v.w;
        }
    }
}

// errmod likelihood (phred-scaled) of the unordered base pair (j, k), j,k in 0..4, from per-base
// read counts c[] and running sums bs[] (htslib/errmod.c:181-205, m = 5; index 4 never has reads)
__device__ __forceinline__ float errmod_pair(int j, int k, int n, const int (&c)[5], const double (&bs)[5], const double* __restrict__ het)
{
    float acc = 0.0f;
#pragma unroll
    for (int i = 0; i < 4; ++i) // float accumulator fed doubles (errmod.c:182,187,197)
        if (i != j && i != k && c[i] > 0) acc = __double2float_rn(__dadd_rn((double)acc, bs[i]));
    float q;
    if (j == k) {
        q = acc; // others == 0 implies acc == 0 (errmod.c:189-191)
    } else {
        const int cjk = c[j] + c[k];
        const double h = het[cjk << 8 | c[k]];
        q = (n - cjk) ? __double2float_rn(__dadd_rn(h, (double)acc)) : __double2float_rn(h);
    }
    return q < 0.0f ? 0.0f : q;
}

template <int MODE>
__global__ void __launch_bounds__(VGL_BLOCK) k_emit(const __grid_constant__ DevParams p)
{
    __shared__ __align__(16) uint32_t stage_gl[VGL_STAGE_ELEMS];
    __shared__ __align__(16) uint32_t stage_x[VGL_STAGE_ELEMS];
    __shared__ int64_t span[4]; // g_lo, g_hi, r_lo, r_hi

    const int tid = threadIdx.x;
    const int64_t c = (int64_t)blockIdx.x * VGL_BLOCK + tid;
    const bool live = c < p.n_cells;
    const int S = p.S;

    SiteView sv;
    sv.A = sv.G = sv.n_obs_alleles = 0;
    sv.skip = 1;
    sv.g_off = p.totals[0];
    sv.r_off = p.totals[1];
    int sample = 0, n = 0;
    if (live) {
        const int64_t sl = c / S;
        sample = (int)(c - sl * S);
        const vgl_site_out* so = p.sites + sl;
        sv.skip = so->skip_code != 0 || so->n_alleles == 0;
        sv.A = sv.skip ? 0 : so->n_alleles;
        sv.G = sv.skip ? 0 : so->n_genotypes;
        sv.n_obs_alleles = so->n_alleles_observed;
        sv.g_off = so->g_off;
        sv.r_off = so->r_off;
#pragma unroll
        for (int i = 0; i < 5; ++i) {
            sv.a2b[i] = so->alleles2acgt[i];
            sv.b2a[i] = so->acgt2alleles[i];
        }
        n = p.dp[c];
    }
    const int A = sv.A, G = sv.G;
    const int64_t gpos = sv.g_off + (int64_t)sample * G; // first GL element of this cell
    const int64_t rpos = sv.r_off + (int64_t)sample * A;
    if (tid == 0) { span[0] = gpos; span[2] = rpos; }
    if (tid == VGL_BLOCK - 1) {
        // include the site's tail padding when this is the last sample of its site
        int64_t ge = gpos + G, re = rpos + A;
        if (live && sample == S - 1) { ge = (ge + 3) & ~3ll; re = (re + 3) & ~3ll; }
        span[1] = ge; span[3] = re;
    }
    __syncthreads();
    const int64_t g_lo = span[0], g_hi = span[1], r_lo = span[2], r_hi = span[3];
    const int64_t g_base = g_lo & ~3ll, r_base = r_lo & ~3ll;
    float* my_gl = reinterpret_cast<float*>(stage_gl) + (gpos - g_base);
    uint32_t* my_x = stage_x + (gpos - g_base);
    // zero the padding after the last sample of a site so that the copy-out is deterministic
    const bool pad_owner = live && !sv.skip && sample == S - 1;
    const int g_pad = pad_owner ? (int)((((int64_t)S * G + 3) & ~3ll) - (int64_t)S * G) : 0;
    const int r_pad = pad_owner ? (int)((((int64_t)S * A + 3) & ~3ll) - (int64_t)S * A) : 0;

    // ------------------------------------------------------------------ GL
    if (live && !sv.skip) {
        if (n == 0) { // gl_methods.cpp:60-66
            for (int g = 0; g < G; ++g) my_gl[g] = f32_missing();
        } else {
            CellSource cs;
            if (MODE != GL_M1_FIXED || n > 255) cs.init(p, c, p.gt[c]);
            if (MODE == GL_M1_FIXED) {
                // ---- model 1, fixed qs: counts only (gl_methods.cpp:304-369)
                int cnt[5];
                int nn = n;
                {
                    const CellRec r = p.cell[c];
                    cnt[0] = r.ad[0]; cnt[1] = r.ad[1]; cnt[2] = r.ad[2]; cnt[3] = r.ad[3]; cnt[4] = 0;
                }
                if (n > 255) { // errmod.c:156-159: only 255 randomly kept reads are scored
                    cnt[0] = cnt[1] = cnt[2] = cnt[3] = 0;
                    nn = 255;
                    if (p.replay) {
                        // binary search this cell in the sorted deep-cell list
                        int64_t lo = 0, hi = p.rp_n_deep - 1, at = -1;
                        while (lo <= hi) {
                            const int64_t mid = (lo + hi) >> 1;
                            const int64_t v = p.rp_deep_cells[mid];
                            if (v == c) { at = mid; break; }
                            if (v < c) lo = mid + 1; else hi = mid - 1;
                        }
                        if (at >= 0)
                            for (int i = 0; i < 255; ++i) {
                                const int b = p.rp_deep_codes[at * 255 + i] & 0xf;
                                cnt[0] += b == 0; cnt[1] += b == 1; cnt[2] += b == 2; cnt[3] += b == 3;
                            }
                    } else {
                        Subsampler sub;
                        sub.init(cs, n);
                        for (int i = 0; i < n; ++i) {
                            const int b = cs.read(p, i).base;
                            if (sub.keep()) { cnt[0] += b == 0; cnt[1] += b == 1; cnt[2] += b == 2; cnt[3] += b == 3; }
                        }
                    }
                }
                float q[15];
                m1f_scores(nn, cnt[0], cnt[1], cnt[2], cnt[3], p.m1_bsum, p.m1_het, q);
                const uint64_t pairmap = p.pairmap[c / S];
                float mx = -CUDART_INF_F;
#pragma unroll
                for (int k = 0; k < 15; ++k) {
                    q[k] = neg_div10(q[k], p.fast_div != 0); // gl_methods.cpp:343
                    if (((pairmap >> (4 * k)) & 0xF) != 0xF) mx = fmaxf(mx, q[k]);
                }
#pragma unroll
                for (int k = 0; k < 15; ++k) { // gl_methods.cpp:355-357
                    const int slot = (int)((pairmap >> (4 * k)) & 0xF);
                    if (slot != 0xF) my_gl[slot] = __fsub_rn(q[k], mx);
                }
            } else if (MODE == GL_M1_PERREAD) {
                // ---- model 1, per-read qs (gl_methods.cpp:233-302 + errmod.c:143-208)
                uint16_t codes[255];
                int nn = 0;
                const bool gl_adj = (p.adjust_qs & 1) != 0;
                if (n > 255 && p.replay) {
                    int64_t lo = 0, hi = p.rp_n_deep - 1, at = -1;
                    while (lo <= hi) {
                        const int64_t mid = (lo + hi) >> 1;
                        const int64_t v = p.rp_deep_cells[mid];
                        if (v == c) { at = mid; break; }
                        if (v < c) lo = mid + 1; else hi = mid - 1;
                    }
                    if (at >= 0) for (int i = 0; i < 255; ++i) codes[i] = p.rp_deep_codes[at * 255 + i];
                    nn = at >= 0 ? 255 : 0;
                } else {
                    Subsampler sub;
                    if (n > 255) sub.init(cs, n);
                    for (int i = 0; i < n; ++i) {
                        const Read r = cs.read(p, i);
                        if (n > 255 && !sub.keep()) continue;
                        int q = gl_adj ? r.adjqs : r.qs;
                        if (q < 0) { atomicExch(p.status, (int)VGL_ERANGE); q = 0; } // the reference stops on ASSERT(qs >= 0) (zero beta draw / negative --adjust-by)
                        codes[nn++] = (uint16_t)(q << 5 | r.base);
                    }
                }
                for (int i = 1; i < nn; ++i) { // ascending insertion sort (errmod.c:160)
                    const uint16_t v = codes[i];
                    int j = i - 1;
                    while (j >= 0 && codes[j] > v) { codes[j + 1] = codes[j]; --j; }
                    codes[j + 1] = v;
                }
                int cnt[5] = {0, 0, 0, 0, 0};
                double bs[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
                for (int i = nn - 1; i >= 0; --i) { // errmod.c:165-178; strand bit never set -> w == c
                    const int code = codes[i];
                    int qual = code >> 5;
                    qual = qual < 4 ? 4 : (qual > 63 ? 63 : qual);
                    const int b = code & 0xf;
#pragma unroll
                    for (int x = 0; x < 4; ++x)
                        if (x == b) {
                            const double t = __dmul_rn(__ldg(p.em_fk + cnt[x]), __ldg(p.em_beta + ((size_t)qual << 16 | (size_t)nn << 8 | cnt[x])));
                            bs[x] = __dadd_rn(bs[x], t);
                            ++cnt[x];
                        }
                }
                float mx = -CUDART_INF_F;
#pragma unroll
                for (int k = 0; k < 5; ++k) {
#pragma unroll
                    for (int j = 0; j <= k; ++j) {
                        const int aj = sv.b2a[j], ak = sv.b2a[k];
                        if (aj < 0 || ak < 0) continue;
                        // -4.343 * lhet is recomputed from the pre-multiplied table: identical product
                        const float q = errmod_pair(j, k, nn, cnt, bs, p.m1_het);
                        const float v = __fdiv_rn(-q, 10.0f);
                        my_gl[gt_index(aj, ak)] = v;
                        mx = fmaxf(mx, v);
                    }
                }
                for (int g = 0; g < G; ++g) my_gl[g] = __fsub_rn(my_gl[g], mx);
            } else {
                // ---- model 2 (gl_methods.cpp:4-231): every read adds homT / het / homF to every
                // genotype and the vector is max-normalised after EVERY read, in float
                float gl[15];
#pragma unroll
                for (int g = 0; g < 15; ++g) gl[g] = -0.0f; // bcf_utils.h:310
                const bool gl_adj = (p.adjust_qs & 1) != 0;
                for (int i = 0; i < n; ++i) {
                    const Read r = cs.read(p, i);
                    double c2, c1, c0; // two / one / no allele of the genotype equals the read
                    if (MODE == GL_M2_FIXED) {
                        c2 = p.homT; c1 = p.het; c0 = p.homF;
                    } else if (MODE == GL_M2_LUT) {
                        int q = gl_adj ? r.adjqs : r.qs;
                        if (q < 0) { atomicExch(p.status, (int)VGL_ERANGE); q = 0; } // vcfgl.cpp:558 ASSERT(adjqScore_i != -1)
                        c2 = __ldg(p.lut_log10 + q); c1 = __ldg(p.lut_log10 + 257 + q); c0 = __ldg(p.lut_log10 + 514 + q);
                    } else {
                        const double e = r.eprob;
                        if (e == 0.0) { c2 = 0.0; c1 = -0.30103; c0 = -CUDART_INF; }
                        else {
                            c2 = log10(1.0 - e);
                            c1 = log10(__dadd_rn((1.0 - e) / 2.0, e / 6.0));
                            c0 = log10(e / 3.0);
                        }
                    }
                    const int ao = sv.b2a[r.base];
                    float mx = -CUDART_INF_F;
#pragma unroll
                    for (int a2 = 0; a2 < 5; ++a2) {
#pragma unroll
                        for (int a1 = 0; a1 <= a2; ++a1) {
                            const int g = a2 * (a2 + 1) / 2 + a1;
                            if (a2 < A) {
                                const int hits = (a1 == ao) + (a2 == ao);
                                const double add = hits == 2 ? c2 : (hits == 1 ? c1 : c0);
                                gl[g] = __double2float_rn(__dadd_rn((double)gl[g], add));
                                mx = gl[g] > mx ? gl[g] : mx;
                            }
                        }
                    }
#pragma unroll
                    for (int g = 0; g < 15; ++g)
                        if (g < G) gl[g] = __fsub_rn(gl[g], mx);
                }
#pragma unroll
                for (int g = 0; g < 15; ++g)
                    if (g < G) my_gl[g] = gl[g];
            }
        }
        for (int g = 0; g < g_pad; ++g) my_gl[G + g] = 0.0f;
    }
    __syncthreads();
    if (p.gl) store_span(reinterpret_cast<uint32_t*>(p.gl), stage_gl, g_base, g_lo, g_hi);

    // ------------------------------------------------------------------ GP (vcfgl.cpp:941-970)
    if (p.gp) {
        if (live && !sv.skip) {
            float* gp = reinterpret_cast<float*>(my_x);
            if (n == 0) {
                for (int g = 0; g < G; ++g) gp[g] = f32_missing();
            } else {
                float sum = 0.0f;
                for (int g = 0; g < G; ++g) {
                    const float v = __double2float_rn(exp10((double)my_gl[g]));
                    gp[g] = v;
                    sum = __fadd_rn(sum, v);
                }
                for (int g = 0; g < G; ++g) gp[g] = __fdiv_rn(gp[g], sum);
            }
            for (int g = 0; g < g_pad; ++g) gp[G + g] = 0.0f;
        }
        __syncthreads();
        store_span(reinterpret_cast<uint32_t*>(p.gp), stage_x, g_base, g_lo, g_hi);
        __syncthreads();
    }
    // ------------------------------------------------------------------ PL (vcfgl.cpp:907-939)
    if (p.pl) {
        if (live && !sv.skip) {
            int32_t* pl = reinterpret_cast<int32_t*>(my_x);
            for (int g = 0; g < G; ++g) {
                const float v = my_gl[g];
                int32_t x;
                if (__float_as_uint(v) == VGL_F32_MISSING_BITS) x = VGL_I32_MISSING;
                else if (v == -CUDART_INF_F) x = 255;
                else {
                    // lroundf((float)(-10.0 * (double)gl)): the double product is exact, so one float multiply rounds identically
                    x = (int32_t)lroundf(__fmul_rn(-10.0f, v));
                    x = x > 255 ? 255 : x;
                }
                pl[g] = x;
            }
            for (int g = 0; g < g_pad; ++g) pl[G + g] = 0;
        }
        __syncthreads();
        store_span(reinterpret_cast<uint32_t*>(p.pl), stage_x, g_base, g_lo, g_hi);
        __syncthreads();
    }
    // ------------------------------------------------------------------ AD / ADF / ADR (vcfgl.cpp:806-831)
    if (p.ad || p.adf || p.adr) {
        CellRec r;
        if (live && !sv.skip) r = p.cell[c];
        int32_t* my_r = reinterpret_cast<int32_t*>(stage_x) + (rpos - r_base);
#pragma unroll 1
        for (int which = 0; which < 3; ++which) {
            int32_t* plane = which == 0 ? p.ad : (which == 1 ? p.adf : p.adr);
            if (!plane) continue;
            if (live && !sv.skip) {
                for (int a = 0; a < A; ++a) {
                    const int b = sv.a2b[a];
                    int v = 0;
                    if (b >= 0 && b < 4) v = which == 0 ? r.ad[b] : (which == 1 ? r.fwd[b] : r.ad[b] - r.fwd[b]);
                    my_r[a] = v;
                }
                for (int a = 0; a < r_pad; ++a) my_r[A + a] = 0;
            }
            __syncthreads();
            store_span(reinterpret_cast<uint32_t*>(plane), stage_x, r_base, r_lo, r_hi);
            __syncthreads();
        }
    }
}

// ==========================================================================
// launchers
// ==========================================================================
void launch_sim(const DevParams& p, cudaStream_t st)
{
    const unsigned grid = (unsigned)((p.n_cells + VGL_BLOCK - 1) / VGL_BLOCK);
    k_sim<<<grid, VGL_BLOCK, 0, st>>>(p);
}

void launch_site(const DevParams& p, cudaStream_t st)
{
    const unsigned grid = (unsigned)(((int64_t)p.n_sites * 32 + VGL_BLOCK - 1) / VGL_BLOCK);
    k_site<<<grid, VGL_BLOCK, 0, st>>>(p);
}

void launch_scan(const DevParams& p, cudaStream_t st) { k_scan<<<1, 1024, 0, st>>>(p); }

void launch_emit(const DevParams& p, cudaStream_t st)
{
    const unsigned grid = (unsigned)((p.n_cells + VGL_BLOCK - 1) / VGL_BLOCK);
    switch (p.gl_mode) {
    case GL_M1_FIXED: k_emit<GL_M1_FIXED><<<grid, VGL_BLOCK, 0, st>>>(p); break;
    case GL_M1_PERREAD: k_emit<GL_M1_PERREAD><<<grid, VGL_BLOCK, 0, st>>>(p); break;
    case GL_M2_FIXED: k_emit<GL_M2_FIXED><<<grid, VGL_BLOCK, 0, st>>>(p); break;
    case GL_M2_LUT: k_emit<GL_M2_LUT><<<grid, VGL_BLOCK, 0, st>>>(p); break;
    default: k_emit<GL_M2_PRECISE><<<grid, VGL_BLOCK, 0, st>>>(p); break;
    }
}

} // namespace vgl
