// VGL_HOST_BGZF -- the BCF record stream of a batch (bcf.cu) compressed on the device into BGZF blocks, the container the
// reference writes by default (-O b: htslib/bgzf.c, thread pool set up at vcfgl.cpp:1791-1803).  What crosses PCIe is the
// compressed stream; the host appends it to the file after its own header block(s) and ends the file with the BGZF EOF block.
//
// A BGZF block is a gzip member with a "BC" extra field holding the block size (htslib/bgzf.c:  18-byte header, raw deflate
// data, CRC32 and length of the uncompressed bytes).  Every block here holds BGZF_IN = 32768 bytes of the record stream (the
// last one less) and is compressed by one CTA on its own, so every match distance lies inside deflate's 32 KiB window:
//
//   k_bgzf_first    thread per block: the first record that reaches into it (binary search over the record offsets)
//   k_bgzf_ranges   warp per block: the block cut into ranges of whole cells and the gaps between them.  The record stream is not
//                   searched byte by byte: k_bcf_emit leaves a descriptor of every record's FORMAT planes, so the compressor knows
//                   where each sample's vector of a tag ("cell": the 15 GL floats, the 15 PL values ...) starts.
//   k_bgzf_deflate  persistent CTAs, one per SM, a block per round.  Cells are hashed whole; a cell whose bytes occurred earlier
//                   in the block as a cell becomes ONE length/distance pair pointing at the first such occurrence (cells never
//                   overlap, so the parse needs no sequential pass; the simulated tags repeat heavily: every sample with the same
//                   read counts has the same vectors).  The 32-bit words of the unmatched cells go through a second, finer table
//                   (a new vector mostly differs from older ones in a few values) and become matches of length 4 where that is
//                   shorter than four literals; the rest are literals.  Codes: one dynamic Huffman code per context (RFC 1951
//                   3.2.7), built on the host from the symbol counts of the context's first record stream (tables.cpp
//                   bgzf_build_code; this kernel in its statistics mode); every block starts with the same precomputed header
//                   bits.  Bit lengths per segment -> CTA-wide prefix sum -> every task ORs its bits into the block image in shared
//                   memory; a block that does not fit the image (three quarters of its input) is stored (3.2.4).  CRC32: the
//                   CTA's last four warps, 64-byte chunks combined by multiplication with x^(8 n) mod P (the identity zlib's
//                   crc32_combine uses), beside the 28 warps that run the phases above.
//   k_bgzf_scan     exclusive prefix of the compressed block sizes
//   k_bgzf_pack     blocks moved back to back into the stream the host receives
//
// Parity: inflating the blocks gives back the VGL_HOST_BCF stream byte for byte (tests/test_gpu_bgzf.py: zlib on the host).
#include "vgl_internal.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>

namespace vgl {

namespace {

constexpr int BGZF_IN = 32768;                  // uncompressed bytes per block
constexpr int BGZF_THREADS = 1024;
constexpr int MAX_SEG = 8192;                   // segments (cells, literal runs) of a block
constexpr int MIN_CELL = 8;                      // vectors shorter than this are not matched: a length / distance pair costs as much as their
                                                 // few literals under the context's code, and a block of 5-byte cells has 6500 segments
constexpr int RUN = 64;                         // bytes of a literal run segment
constexpr int OUT_WORDS = 24576 / 4;               // the block image; a block that does not fit (three quarters of its input) is stored
constexpr int HASH_SLOTS = 8192;
constexpr int MAX_RANGES = 32 * 16;
constexpr int WORD_BITS = 12, WORD_SLOTS = 1 << WORD_BITS; // word table of the unmatched cells (half of the cell table's memory)
constexpr int DT = BGZF_THREADS - 128;       // threads of the compressor's phases; the CTA's last four warps do the CRC
constexpr int SEG_PER_THREAD = (MAX_SEG + DT - 1) / DT;
constexpr int CRC_CHUNK = 64;                  // bytes a thread takes in the CRC pass

struct Seg { // 8 bytes
    uint16_t pos, len;   // position in the block, bytes
    uint32_t info;       // SEG_MATCH | distance; SEG_LIT | bits of quarters 0, 1, 2 (8 bits each); SEG_CELL: a match candidate
};
constexpr uint32_t SEG_MATCH = 1u << 31, SEG_LIT = 1u << 30, SEG_CELL = 1u << 29;
constexpr uint32_t CAP_BITS = (uint32_t)OUT_WORDS * 32u - 96u; // what the block image holds

__device__ __forceinline__ uint32_t rev_bits(uint32_t code, int n) { return __brev(code) >> (32 - n); }

// distance code, number and value of its extra bits (1 <= dist <= 32768)
__device__ __forceinline__ void dist_code(int dist, int& dc, int& deb, uint32_t& dev)
{
    if (dist <= 4) { dc = dist - 1; deb = 0; dev = 0u; }
    else {
        const int u = dist - 1, hb = 31 - __clz(u);
        deb = hb - 1;
        dc = 2 * hb + ((u >> deb) & 1);
        dev = (uint32_t)u & ((1u << deb) - 1u);
    }
}
// index of the length symbol (257 + ...) of a match length
__device__ __forceinline__ int len_symbol(int len)
{
    const int t = len - 3;
    if (t < 8) return t;
    if (len == 258) return 28;
    const int hb = 31 - __clz(t);
    return 4 * (hb - 1) + ((t >> (hb - 2)) & 3);
}
// length / distance pair (3 <= len <= 258) from the context's code tables: up to 20 + 15 + 13 bits
__device__ __forceinline__ void match_code(const uint32_t* len_tab, const uint32_t* dist_tab, int len, int dist, unsigned long long& bits, int& n)
{
    const uint32_t le = len_tab[len - 3];
    int dc, deb;
    uint32_t dev;
    dist_code(dist, dc, deb, dev);
    const uint32_t de = dist_tab[dc];
    int nb = (int)(le >> 24);
    unsigned long long b = le & 0xFFFFFFu;
    b |= (unsigned long long)(de & 0xFFFFu) << nb;
    nb += (int)(de >> 16);
    b |= (unsigned long long)dev << nb;
    bits = b;
    n = nb + deb;
}
__device__ __forceinline__ int match_bits(const uint32_t* len_tab, const uint32_t* dist_tab, int len, int dist)
{
    int dc, deb;
    uint32_t dev;
    dist_code(dist, dc, deb, dev);
    return (int)(len_tab[len - 3] >> 24) + (int)(dist_tab[dc] >> 16) + deb;
}

// ORs `n` (<= 32) bits into the block image at bit offset `at`
__device__ __forceinline__ void put_bits(uint32_t* out, unsigned at, uint32_t bits, int n)
{
    const unsigned w = at >> 5, sh = at & 31u;
    atomicOr(&out[w], bits << sh);
    if (sh + (unsigned)n > 32u) atomicOr(&out[w + 1], bits >> (32u - sh));
}

// ... up to 57 bits
__device__ __forceinline__ void put_bits64(uint32_t* out, unsigned at, unsigned long long bits, int n)
{
    const unsigned w = at >> 5, sh = at & 31u;
    atomicOr(&out[w], (uint32_t)bits << sh);
    const unsigned long long rest = bits >> (32u - sh); // sh = 0: the upper word
    if (sh + (unsigned)n > 32u) atomicOr(&out[w + 1], (uint32_t)rest);
    if (sh + (unsigned)n > 64u) atomicOr(&out[w + 2], (uint32_t)(rest >> 32));
}

// a * b mod P over GF(2) in the reflected representation of CRC-32 (P = 0xEDB88320): shifts a CRC across the bytes that follow
__host__ __device__ inline uint32_t crc_mul(uint32_t a, uint32_t b)
{
    uint32_t m = 1u << 31, p = 0u;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1u)) == 0u) break;
        }
        m >>= 1;
        b = (b & 1u) ? (b >> 1) ^ 0xEDB88320u : b >> 1;
    }
    return p;
}

// the same product, branch-free (device: every lane takes the same 32 steps)
__device__ __forceinline__ uint32_t crc_mul_dev(uint32_t a, uint32_t b)
{
    uint32_t p = 0u;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        p ^= b & (uint32_t)((int32_t)a >> 31); // bit 31 of a: the x^0 term in the reflected representation
        a <<= 1;
        b = (b >> 1) ^ (0xEDB88320u & (0u - (b & 1u)));
    }
    return p;
}

// first record whose bytes reach into block b (the last record that starts at or before the block's first byte)
__global__ void __launch_bounds__(256) k_bgzf_first(const BgzfArgs a)
{
    const long long total = a.totals[3];
    const long long nblk = total > a.in_cap ? 0 : (total + BGZF_IN - 1) / BGZF_IN;
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < nblk; b += (long long)gridDim.x * blockDim.x) {
        const long long b0 = b * BGZF_IN;
        int lo = 0, hi = a.n_sites; // rec_off[lo] <= b0 < rec_off[hi]; rec_off is non-decreasing
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (a.rec_off[mid] <= b0) lo = mid; else hi = mid;
        }
        a.blk_first[b] = lo;
    }
}

// 32-bit word at byte offset `pos` of shared memory (any alignment)
__device__ __forceinline__ uint32_t word_at(const uint8_t* base, uint32_t pos)
{
    const uint32_t* w = reinterpret_cast<const uint32_t*>(base) + (pos >> 2);
    const uint32_t sh = (pos & 3u) * 8u;
    return sh ? __funnelshift_r(w[0], w[1], sh) : w[0];
}

// The part of every record that lies in block `blk` ([b0, b0 + L) of the stream), split at the FORMAT planes: ranges of whole
// cells and the gaps between them (one warp, a lane per record).  rng[i] = {pos, len, cell bytes (0: gap), first segment}.
// state: 0 = ranges written, 1 = the block goes out as literals, 2 = more than cap_rng ranges (nothing written)
__device__ void bgzf_block_ranges(const BgzfArgs& a, int blk, long long b0, int L, int lane, uint32_t* rng, int cap_rng, int& n_rng, int& n_seg, int& state)
{
    const int lo = a.blk_first[blk];
    const int r = lo + lane;
    int my_n = 0;
    uint32_t my[16][3]; // pos, len, cell
    long long rs = 0, re = 0;
    if (r < a.n_sites) { rs = a.rec_off[r]; re = a.rec_off[r + 1]; }
    const bool has = r < a.n_sites && re > rs && rs < b0 + L && re > b0;
    if (has) {
        const BcfRecPlanes pl = a.planes[r];
        long long cur = max(rs, b0); // next byte of the record not yet put into a range
        const long long end = min(re, b0 + L);
        for (int k = 0; k < (int)pl.n && k < 7; ++k) {
            const long long ps = rs + pl.off[k], pe = ps + (long long)pl.cell[k] * a.S;
            if (pl.cell[k] < MIN_CELL || pl.cell[k] > RUN || pe <= cur || ps >= end) continue; // short vectors go out as literals (see MIN_CELL); segments at most RUN
            // full cells of this plane inside [cur, end)
            long long c_lo = ps >= cur ? 0 : (cur - ps + pl.cell[k] - 1) / pl.cell[k];
            long long c_hi = pe <= end ? a.S : (end - ps) / pl.cell[k];
            if (c_hi <= c_lo) continue;
            const long long cs = ps + c_lo * pl.cell[k], ce = ps + c_hi * pl.cell[k];
            if (cs > cur) { my[my_n][0] = (uint32_t)(cur - b0); my[my_n][1] = (uint32_t)(cs - cur); my[my_n][2] = 0u; ++my_n; }
            my[my_n][0] = (uint32_t)(cs - b0); my[my_n][1] = (uint32_t)(ce - cs); my[my_n][2] = pl.cell[k]; ++my_n;
            cur = ce;
        }
        if (cur < end) { my[my_n][0] = (uint32_t)(cur - b0); my[my_n][1] = (uint32_t)(end - cur); my[my_n][2] = 0u; ++my_n; }
    }
    // more than 32 records in one block (a handful of samples): the block goes out as literals, nothing to gain there
    const long long last_end = __shfl_sync(0xffffffffu, has ? re : 0, 31);
    const bool overflow = lo + 32 < a.n_sites && last_end < b0 + L && __shfl_sync(0xffffffffu, (int)has, 31);
    int segs_mine = 0, bytes_mine = 0;
    for (int k = 0; k < my_n; ++k) {
        segs_mine += my[k][2] ? (int)(my[k][1] / my[k][2]) : (int)((my[k][1] + RUN - 1) / RUN);
        bytes_mine += (int)my[k][1];
    }
    const bool covered = __reduce_add_sync(0xffffffffu, bytes_mine) == L; // else: records beyond the 32 lanes (skipped sites in between)
    int inc_r = my_n, inc_s = segs_mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t1 = __shfl_up_sync(0xffffffffu, inc_r, o), t2 = __shfl_up_sync(0xffffffffu, inc_s, o);
        if (lane >= o) { inc_r += t1; inc_s += t2; }
    }
    const int tot_r = __shfl_sync(0xffffffffu, inc_r, 31), tot_s = __shfl_sync(0xffffffffu, inc_s, 31);
    n_rng = tot_r;
    n_seg = tot_s;
    if (overflow || !covered || tot_s > MAX_SEG || tot_r > MAX_RANGES) {
        state = 1;
    } else if (tot_r > cap_rng) {
        state = 2;
    } else {
        state = 0;
        int r0 = inc_r - my_n, s0 = inc_s - segs_mine;
        for (int k = 0; k < my_n; ++k) {
            rng[(r0 + k) * 4 + 0] = my[k][0]; rng[(r0 + k) * 4 + 1] = my[k][1]; rng[(r0 + k) * 4 + 2] = my[k][2]; rng[(r0 + k) * 4 + 3] = (uint32_t)s0;
            s0 += my[k][2] ? (int)(my[k][1] / my[k][2]) : (int)((my[k][1] + RUN - 1) / RUN);
        }
    }
}

// a warp per block: the block's ranges into its slot of rng_g ({ranges, segments, state, -}, then the ranges).  The grid is
// sized on the host's estimate of the batch's blocks; the loop covers the real count (a short batch that carries most of the
// pass-through blob makes more blocks than its share of sites predicts).
__global__ void __launch_bounds__(256) k_bgzf_ranges(const BgzfArgs a)
{
    const long long total = a.totals[3];
    const long long nblk = total > a.in_cap ? 0 : (total + BGZF_IN - 1) / BGZF_IN;
    const int lane = threadIdx.x & 31;
    for (long long blk = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); blk < nblk; blk += (long long)gridDim.x * 8) {
        const long long b0 = blk * BGZF_IN;
        const int L = (int)min((long long)BGZF_IN, total - b0);
        uint32_t* const g = a.rng_g + (size_t)blk * BGZF_RNG_WORDS;
        int n_r = 0, n_s = 0, state = 0;
        bgzf_block_ranges(a, (int)blk, b0, L, lane, g + 4, BGZF_RNG_LIST, n_r, n_s, state);
        if (lane == 0) { g[0] = (uint32_t)n_r; g[1] = (uint32_t)n_s; g[2] = (uint32_t)state; g[3] = 0u; }
    }
}

#ifdef BGZF_PROF // development: cycles between the kernel's barriers, summed over blocks (make bgzfprof; tools/prof_bgzf.py)
__device__ unsigned long long g_bgzf_prof[16];
#define PROFW(i) do { if (threadIdx.x == 32) { const long long t_ = clock64(); atomicAdd(&g_bgzf_prof[i], (unsigned long long)(t_ - prof_t)); prof_t = t_; } } while (0)
#define PROF(i) do { if (threadIdx.x == 0) { const long long t_ = clock64(); atomicAdd(&g_bgzf_prof[i], (unsigned long long)(t_ - prof_t)); prof_t = t_; } } while (0)
#else
#define PROF(i) do { } while (0)
#define PROFW(i) do { } while (0)
#endif
#define DSYNC() asm volatile("bar.sync 2, %0;" ::"n"(DT) : "memory")

// one block of the stream (a whole CTA); the CRC and code tables are the kernel's, loaded once per CTA
__device__ __forceinline__ void deflate_block(const BgzfArgs& a, const int blk, unsigned char* const sm, const uint32_t* const crc_tab,
                                              const uint32_t* const lit_tab, const uint32_t* const len_tab, const uint32_t* const dist_tab,
                                              const uint32_t eob_s, const uint32_t hdr_bits_s)
{
#ifdef BGZF_PROF
    long long prof_t = clock64();
#endif
    uint8_t* const in = sm;                                                       // [BGZF_IN]
    uint32_t* const out = reinterpret_cast<uint32_t*>(sm + BGZF_IN);              // [OUT_WORDS]
    Seg* const segs = reinterpret_cast<Seg*>(sm + BGZF_IN + OUT_WORDS * 4);        // [MAX_SEG]
    uint32_t* const seg_bit = reinterpret_cast<uint32_t*>(segs + MAX_SEG);        // [MAX_SEG] bit offset of every segment
    uint32_t* const htab = seg_bit + MAX_SEG;                                     // [HASH_SLOTS] tag << 16 | position
    uint32_t* const rng = htab + HASH_SLOTS;                                      // [MAX_RANGES][4]: pos, len, cell bytes (0: gap), first segment
    uint16_t* const lit_list = reinterpret_cast<uint16_t*>(rng + MAX_RANGES * 4);  // [MAX_SEG] the segments that are not matches (any order)
    __shared__ uint32_t warp_tot[32];
    __shared__ int n_rng_s, n_seg_s, lit_only_s, n_lit_s;
    __shared__ uint32_t crc_s, total_bits_s;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long total = a.totals[3];
    const long long b0 = (long long)blk * BGZF_IN;
    const int L = (int)min((long long)BGZF_IN, total - b0);

    // ---- warps 1..: the block's bytes, the CRC and literal-code tables, cleared tables; meanwhile warp 0: the ranges
    if (warp > 0) {
        const int t = tid - 32, nt = BGZF_THREADS - 32;
        // the block's bytes are requested first and stored last: everything in between runs under the latency of the loads
        const uint4* const src = reinterpret_cast<const uint4*>(a.in + b0);
        const int n16 = (L + 15) / 16; // <= 2048 = 2.07 per thread
        uint4 v0 = make_uint4(0u, 0u, 0u, 0u), v1 = v0, v2 = v0;
        if (t < n16) v0 = __ldcs(src + t);
        if (t + nt < n16) v1 = __ldcs(src + t + nt);
        if (t + 2 * nt < n16) v2 = __ldcs(src + t + 2 * nt);
        if (t == 0) { crc_s = 0u; n_lit_s = 0; }
        for (int i = t; i < OUT_WORDS / 4; i += nt) reinterpret_cast<uint4*>(out)[i] = make_uint4(0u, 0u, 0u, 0u);
        for (int i = t; i < HASH_SLOTS / 4; i += nt) reinterpret_cast<uint4*>(htab)[i] = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
        if (t < n16) reinterpret_cast<uint4*>(in)[t] = v0;
        if (t + nt < n16) reinterpret_cast<uint4*>(in)[t + nt] = v1;
        if (t + 2 * nt < n16) reinterpret_cast<uint4*>(in)[t + 2 * nt] = v2;
        PROFW(8); // load, clear, tables issued
        // Barrier 1 = warps 1 .. 31 only (the image is cleared before the header goes in).
        asm volatile("bar.sync 1, %0;" ::"r"(nt) : "memory");
        PROFW(9); // barrier of warps 1..31 (the loads have landed)
        if (!a.hist && t < (int)((hdr_bits_s + 31u) >> 5)) out[t] = a.code->hdr[t]; // the block header (the image is cleared)
    }

    // ---- ranges: made by k_bgzf_ranges ahead of this kernel (on one warp they would take as long as everything else here)
    if (warp == 0) {
        const uint32_t* const g = a.rng_g + (size_t)blk * BGZF_RNG_WORDS;
        const uint4 h = __ldg(reinterpret_cast<const uint4*>(g)); // ranges, segments, state
        int n_r = (int)h.x, n_s = (int)h.y, state = (int)h.z;
        if (state == 2) bgzf_block_ranges(a, blk, b0, L, lane, rng, MAX_RANGES, n_r, n_s, state); // more than the list holds
        else if (state == 0)
            for (int i = lane; i < n_r; i += 32) reinterpret_cast<uint4*>(rng)[i] = __ldg(reinterpret_cast<const uint4*>(g) + 1 + i);
        if (lane == 0) { n_rng_s = n_r; n_seg_s = n_s; lit_only_s = state != 0; }
    }
    __syncthreads();
    PROF(0); // load + tables || ranges
    // ---- the last four warps: CRC32 of the block -- 64-byte chunks from the end (slicing by four), each shifted across the bytes
    // behind it -- while the other 28 run the compressor's phases (their barriers are barrier 2 from here on).  The look-ups of
    // the slicing tables collide 3.5-way on the banks whoever does them; beside the latency-bound phases they cost nothing.
    if (warp >= DT / 32) {
        if (!a.hist) {
            for (int c = tid - DT; c < BGZF_IN / CRC_CHUNK; c += BGZF_THREADS - DT) {
                const int hi = L - c * CRC_CHUNK, lo2 = max(hi - CRC_CHUNK, 0);
                if (hi <= 0) break;
                uint32_t r = 0xFFFFFFFFu;
                auto step = [&](uint32_t w) {
                    r ^= w;
                    r = crc_tab[768 + (r & 0xFFu)] ^ crc_tab[512 + ((r >> 8) & 0xFFu)] ^ crc_tab[256 + ((r >> 16) & 0xFFu)] ^ crc_tab[r >> 24];
                };
                if (hi - lo2 == CRC_CHUNK && (lo2 & 15) == 0) { // a whole aligned chunk: 128-bit loads (word loads at this stride collide on four banks)
#pragma unroll
                    for (int q = 0; q < CRC_CHUNK / 16; ++q) {
                        const uint4 v = *reinterpret_cast<const uint4*>(in + lo2 + 16 * q);
                        step(v.x); step(v.y); step(v.z); step(v.w);
                    }
                } else {
                    int k = lo2;
                    for (; k < hi && ((hi - k) & 3); ++k) r = crc_tab[(r ^ in[k]) & 0xFFu] ^ (r >> 8); // head bytes: the rest is whole words
                    for (; k < hi; k += 4) step(word_at(in, (uint32_t)k));
                }
                const uint32_t part = crc_mul_dev(__ldg(a.crc_pow + c), ~r);
                if (part) atomicXor(&crc_s, part);
            }
            __threadfence_block();
            asm volatile("bar.arrive 4, %0;" ::"n"(BGZF_THREADS) : "memory"); // the CRC is in crc_s (the trailer's writers wait on barrier 4)
        }
        return; // to the kernel loop's barrier
    }
    if (lit_only_s) { // one gap over the whole block
        if (tid == 0) {
            rng[0] = 0u; rng[1] = (uint32_t)L; rng[2] = 0u; rng[3] = 0u;
            n_rng_s = 1;
            n_seg_s = (L + RUN - 1) / RUN;
        }
        DSYNC();
    }
    const int n_rng = n_rng_s, n_seg = n_seg_s;

    // ---- segment table
    for (int j = warp; j < n_rng; j += DT / 32) {
        const uint32_t pos = rng[j * 4], len = rng[j * 4 + 1], cell = rng[j * 4 + 2], first = rng[j * 4 + 3];
        const int n = cell ? (int)(len / cell) : (int)((len + RUN - 1) / RUN);
        for (int c = lane; c < n; c += 32) {
            Seg s;
            if (cell) { s.pos = (uint16_t)(pos + (uint32_t)c * cell); s.len = (uint16_t)cell; s.info = SEG_CELL; }
            else { s.pos = (uint16_t)(pos + (uint32_t)c * RUN); s.len = (uint16_t)min((uint32_t)RUN, len - (uint32_t)c * RUN); s.info = 0u; }
            segs[first + c] = s;
        }
    }
    DSYNC();
    PROF(1); // segment table

    // ---- cells: hash of the bytes, first occurrence per hash (atomicMin on tag << 16 | position; open addressing)
    auto cell_hash = [&](const Seg& s) -> uint32_t { // sum of the 32-bit words (the tail word masked) times odd constants: no chain
        uint32_t h = 2166136261u ^ s.len, c = 0x9E3779B1u;
        const int nw = s.len >> 2;
        // the cell's words share one alignment: every aligned word is loaded once and funnel-shifted with its neighbour
        const uint32_t* const aw = reinterpret_cast<const uint32_t*>(in) + (s.pos >> 2);
        const uint32_t sh = (s.pos & 3u) * 8u;
        uint32_t prev = aw[0];
        for (int k = 0; k < nw; ++k) {
            const uint32_t next = aw[k + 1];
            h += __funnelshift_r(prev, next, sh) * c;
            prev = next;
            c += 0x7F4A7C16u; // stays odd
        }
        if (s.len & 3) h += (__funnelshift_r(prev, aw[nw + 1], sh) & ((1u << (8 * (s.len & 3))) - 1u)) * c;
        h ^= h >> 15;
        h *= 0x2C1B3C6Du;
        h ^= h >> 13;
        return h;
    };
    for (int j = tid; j < n_seg; j += DT) {
        const Seg s = segs[j];
        if (!(s.info & SEG_CELL)) continue;
        const uint32_t h = cell_hash(s), tag = h >> 16, mine = (tag << 16) | s.pos;
        seg_bit[j] = h; // kept for the look-up pass
        uint32_t slot = h & (HASH_SLOTS - 1);
        for (int probe = 0; probe < 16; ++probe) {
            const uint32_t old = atomicCAS(&htab[slot], 0xFFFFFFFFu, mine);
            if (old == 0xFFFFFFFFu) break;
            if ((old >> 16) == tag) { atomicMin(&htab[slot], mine); break; }
            slot = (slot + 1) & (HASH_SLOTS - 1);
        }
    }
    DSYNC();
    PROF(2); // hash insert
    // ---- match = the first cell of the block with the same bytes; the other segments go on the list of literal segments
    for (int j0 = warp * 32; j0 < n_seg; j0 += DT) {
        const int j = j0 + lane;
        bool is_lit = false;
        if (j < n_seg) {
            const Seg s = segs[j];
            is_lit = true;
            if (s.info & SEG_CELL) {
                const uint32_t h = seg_bit[j], tag = h >> 16;
                uint32_t slot = h & (HASH_SLOTS - 1), dist = 0u;
                for (int probe = 0; probe < 16; ++probe) {
                    const uint32_t e = htab[slot];
                    if (e == 0xFFFFFFFFu) break;
                    if ((e >> 16) == tag) {
                        const uint32_t q = e & 0xFFFFu;
                        if (q < s.pos && q + s.len <= s.pos) { // an earlier cell (cells do not overlap)
                            uint32_t diff = 0u; // all words compared, no early exit: the loads are independent
                            const int nw = s.len >> 2;
                            const uint32_t* const wa = reinterpret_cast<const uint32_t*>(in) + (q >> 2);
                            const uint32_t* const wb = reinterpret_cast<const uint32_t*>(in) + (s.pos >> 2);
                            const uint32_t sha = (q & 3u) * 8u, shb = (s.pos & 3u) * 8u;
                            uint32_t pa = wa[0], pb = wb[0];
                            for (int k = 0; k < nw; ++k) {
                                const uint32_t na = wa[k + 1], nb = wb[k + 1];
                                diff |= __funnelshift_r(pa, na, sha) ^ __funnelshift_r(pb, nb, shb);
                                pa = na;
                                pb = nb;
                            }
                            for (int k = 4 * nw; k < s.len; ++k) diff |= (uint32_t)(in[q + k] ^ in[s.pos + k]);
                            if (diff == 0u) dist = s.pos - q;
                        }
                        break;
                    }
                    slot = (slot + 1) & (HASH_SLOTS - 1);
                }
                if (dist) {
                    segs[j].info = SEG_MATCH | dist;
                    seg_bit[j] = (uint32_t)match_bits(len_tab, dist_tab, s.len, (int)dist);
                    is_lit = false;
                } // else: an unmatched cell stays a candidate for word matches (SEG_CELL)
            }
        }
        const uint32_t m = __ballot_sync(0xffffffffu, is_lit);
        int base = 0;
        if (lane == 0 && m) base = atomicAdd(&n_lit_s, __popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (is_lit) lit_list[base + __popc(m & ((1u << lane) - 1u))] = (uint16_t)j;
    }
    // ---- words: the 32-bit words of the unmatched cells against each other.  A new cell mostly differs from earlier ones in a
    // few of its values; every word that occurred before in an unmatched cell (any matched cell is a copy of one) can go out
    // as a match of length 4.  The cell table's memory now holds the word table (first position per value, the value is read
    // back from the block) and, per word of the block, the distance chosen (0: literals).
    DSYNC();
    PROF(3); // match
    uint32_t* const wtab = htab;                                           // [WORD_SLOTS]
    uint16_t* const wdist = reinterpret_cast<uint16_t*>(htab + WORD_SLOTS); // [BGZF_IN / 4]
    for (int i = tid; i < HASH_SLOTS / 4; i += DT)
        reinterpret_cast<uint4*>(htab)[i] = i < WORD_SLOTS / 4 ? make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu) : make_uint4(0u, 0u, 0u, 0u);
    DSYNC();
    // quarter q of a literal segment: bytes [k0, k1), the first nwb of them whole words of an unmatched cell
    auto quarter = [&](const Seg& sg, int q, int& k0, int& k1, int& nwb) {
        if (sg.info & SEG_CELL) {
            const int nw = sg.len >> 2, qw = (nw + 3) >> 2, w0 = min(q * qw, nw), w1 = min(w0 + qw, nw);
            k0 = 4 * w0;
            k1 = q == 3 ? (int)sg.len : 4 * w1;
            nwb = 4 * (w1 - w0);
        } else {
            const int ql = (sg.len + 3) >> 2;
            k0 = min(q * ql, (int)sg.len);
            k1 = min(k0 + ql, (int)sg.len);
            nwb = 0;
        }
    };
    const int n_lit = n_lit_s;
    for (int task = tid; task < n_lit * 16; task += DT) { // insert: a word of an unmatched cell per thread
        const Seg ls = segs[lit_list[task >> 4]];
        const int k = 4 * (task & 15);
        if (!(ls.info & SEG_CELL) || k + 4 > (int)ls.len) continue;
        const uint32_t wp = ls.pos + (uint32_t)k, v = word_at(in, wp);
        uint32_t slot = (v * 2654435761u) >> (32 - WORD_BITS);
        for (int probe = 0; probe < 8; ++probe) { // (thinning out equal values with __match_any_sync first costs more than the atomics it saves)
            uint32_t cur = wtab[slot];
            if (cur == 0xFFFFFFFFu) {
                cur = atomicCAS(&wtab[slot], 0xFFFFFFFFu, wp);
                if (cur == 0xFFFFFFFFu) break;
            }
            if (word_at(in, cur) == v) {
                if (wp < cur) atomicMin(&wtab[slot], wp); // (an entry only ever moves to an earlier position of the same value)
                break;
            }
            slot = (slot + 1) & (WORD_SLOTS - 1);
        }
    }
    DSYNC();
    PROF(4); // word insert
    // ---- bit length of every segment under the context's code (the word matches are decided here: a match where it is
    // shorter than its four literals), exclusive prefix; should the image not hold them (a code built from other statistics),
    // once more under the fixed code, which always fits.  The statistics pass counts the symbols instead and stops.
    uint32_t* const hist = out; // statistics pass only (the image is clear and stays unused)
    if (a.hist) // the matches' symbols (their bit lengths are already in place)
        for (int j = tid; j < n_seg; j += DT) {
            const Seg s = segs[j];
            if (!(s.info & SEG_MATCH)) continue;
            int dc, deb;
            uint32_t dev;
            dist_code((int)(s.info & 0xFFFFu), dc, deb, dev);
            atomicAdd(&hist[257 + len_symbol(s.len)], 1u);
            atomicAdd(&hist[288 + dc], 1u);
        }
    for (int tb = 0; tb < n_lit * 4; tb += DT) { // a quarter of a literal segment per thread; lanes 4 i .. 4 i + 3 share a segment
        const int t = tb + tid;
        uint32_t part = 0u;
        int jj = 0;
        const int q = t & 3;
        if (t < n_lit * 4) {
            jj = lit_list[t >> 2];
            const Seg ls = segs[jj];
            int k0, k1, nwb;
            quarter(ls, q, k0, k1, nwb);
            int k = k0;
            for (; k < k0 + nwb; k += 4) {
                const uint32_t wp = ls.pos + (uint32_t)k, v = word_at(in, wp);
                const uint32_t e0 = lit_tab[v & 0xFFu], e1 = lit_tab[(v >> 8) & 0xFFu], e2 = lit_tab[(v >> 16) & 0xFFu], e3 = lit_tab[v >> 24];
                uint32_t nb = (e0 >> 16) + (e1 >> 16) + (e2 >> 16) + (e3 >> 16), dsel = 0u;
                uint32_t slot = (v * 2654435761u) >> (32 - WORD_BITS);
                for (int probe = 0; probe < 8; ++probe) {
                    const uint32_t cur = wtab[slot];
                    if (cur == 0xFFFFFFFFu) break;
                    if (word_at(in, cur) == v) {
                        if (cur < wp) {
                            const uint32_t mb = (uint32_t)match_bits(len_tab, dist_tab, 4, (int)(wp - cur));
                            if (mb < nb) { nb = mb; dsel = wp - cur; }
                        }
                        break;
                    }
                    slot = (slot + 1) & (WORD_SLOTS - 1);
                }
                wdist[wp >> 2] = (uint16_t)dsel;
                part += nb;
                if (a.hist) {
                    if (dsel) {
                        int dc, deb;
                        uint32_t dev;
                        dist_code((int)dsel, dc, deb, dev);
                        atomicAdd(&hist[257 + 1], 1u); // length 4
                        atomicAdd(&hist[288 + dc], 1u);
                    } else {
                        atomicAdd(&hist[v & 0xFFu], 1u); atomicAdd(&hist[(v >> 8) & 0xFFu], 1u);
                        atomicAdd(&hist[(v >> 16) & 0xFFu], 1u); atomicAdd(&hist[v >> 24], 1u);
                    }
                }
            }
            for (; k < k1; ++k) {
                const uint32_t b = in[ls.pos + k];
                part += lit_tab[b] >> 16;
                if (a.hist) atomicAdd(&hist[b], 1u);
            }
        }
        // bits of the quarters before this one, and of the whole segment
        const uint32_t p1 = __shfl_up_sync(0xffffffffu, part, 1), p2 = __shfl_up_sync(0xffffffffu, part, 2), p3 = __shfl_up_sync(0xffffffffu, part, 3);
        if (t < n_lit * 4 && q == 3) {
            seg_bit[jj] = part + p1 + p2 + p3;
            segs[jj].info = (segs[jj].info & SEG_CELL) | SEG_LIT | p3 | (p2 << 8) | (p1 << 16); // quarters 0, 1, 2
        }
    }
    if (a.hist) { // statistics pass: the counts of this block to the context's, nothing is written
        DSYNC();
        if (tid < BGZF_HIST && hist[tid]) atomicAdd(&a.hist[tid], hist[tid]);
        if (tid == 0) atomicAdd(&a.hist[256], 1u);
        return;
    }
    DSYNC();
    PROF(5); // bit lengths
    {
        uint32_t v[SEG_PER_THREAD], sum = 0u;
#pragma unroll
        for (int k = 0; k < SEG_PER_THREAD; ++k) {
            const int j = tid * SEG_PER_THREAD + k;
            v[k] = j < n_seg ? seg_bit[j] : 0u;
            sum += v[k];
        }
        uint32_t inc = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) warp_tot[warp] = inc;
        DSYNC();
        if (warp == 0) {
            uint32_t t = lane < DT / 32 ? warp_tot[lane] : 0u;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t u = __shfl_up_sync(0xffffffffu, t, o);
                if (lane >= o) t += u;
            }
            warp_tot[lane] = t;
        }
        DSYNC();
        uint32_t base = hdr_bits_s + (warp ? warp_tot[warp - 1] : 0u) + inc - sum;
#pragma unroll
        for (int k = 0; k < SEG_PER_THREAD; ++k) {
            const int j = tid * SEG_PER_THREAD + k;
            if (j < n_seg) seg_bit[j] = base;
            base += v[k];
        }
        if (tid == DT - 1) total_bits_s = base;
    }
    DSYNC();
    PROF(6); // prefix
    uint8_t* const dst = a.stage + (size_t)blk * BGZF_STRIDE + 2; // + 2: the deflate data (at + 18) starts on a word
    if (total_bits_s + (eob_s >> 16) > CAP_BITS) {
        // the image does not hold the block (it would barely shrink, or the context's code was built from other statistics):
        // a stored block (RFC 1951 3.2.4) -- BFINAL = 1, BTYPE = 00, LEN, ~LEN, the bytes
        const uint32_t bsize = 18u + 5u + (uint32_t)L + 8u;
        if (tid < 18) {
            const uint8_t hdr[18] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, (uint8_t)((bsize - 1u) & 0xFFu), (uint8_t)((bsize - 1u) >> 8)};
            dst[tid] = hdr[tid];
        }
        if (tid < 5) {
            const uint8_t sb[5] = {1, (uint8_t)(L & 0xFF), (uint8_t)(L >> 8), (uint8_t)(~L & 0xFF), (uint8_t)((~L >> 8) & 0xFF)};
            dst[18 + tid] = sb[tid];
        }
        for (int i = tid; i < L; i += DT) dst[23 + i] = in[i];
        asm volatile("bar.sync 4, %0;" ::"n"(BGZF_THREADS) : "memory"); // the CRC warps are done
        if (tid < 8) {
            const uint32_t v = tid < 4 ? crc_s : (uint32_t)L;
            dst[23 + L + tid] = (uint8_t)(v >> (8 * (tid & 3)));
        }
        if (tid == 0) a.blk_size[blk] = bsize;
        return;
    }
    // ---- bits: the segments, then the end-of-block code.
    // A literal segment is split into quarters (their bit offsets follow from the counts kept with the segment).
    if (tid == 0) put_bits(out, total_bits_s, eob_s & 0xFFFFu, (int)(eob_s >> 16));
    for (int j = tid; j < n_seg; j += DT) {
        const Seg s = segs[j];
        if (!(s.info & SEG_MATCH)) continue;
        unsigned long long bb;
        int n;
        match_code(len_tab, dist_tab, s.len, (int)(s.info & 0xFFFFu), bb, n);
        put_bits64(out, seg_bit[j], bb, n);
    }
    for (int t = tid; t < n_lit * 4; t += DT) {
        const int jj = lit_list[t >> 2], q = t & 3;
        const Seg ls = segs[jj];
        int k0, k1, nwb;
        quarter(ls, q, k0, k1, nwb);
        if (k0 >= k1) continue;
        const unsigned c = ls.info; // bits of quarters 0, 1, 2
        const unsigned cum = (q > 0 ? c & 255u : 0u) + (q > 1 ? (c >> 8) & 255u : 0u) + (q > 2 ? (c >> 16) & 255u : 0u);
        unsigned at = seg_bit[jj] + cum;
        unsigned w = at >> 5;
        int fill = (int)(at & 31u);
        unsigned long long acc = 0ull;
        auto pair = [&](uint32_t ea, uint32_t eb) { // two codes (<= 30 bits) behind the pending bits
            const uint32_t n0 = ea >> 16;
            acc |= (unsigned long long)((ea & 0xFFFFu) | ((eb & 0xFFFFu) << n0)) << fill;
            fill += (int)(n0 + (eb >> 16));
            if (fill >= 32) {
                atomicOr(&out[w], (uint32_t)acc);
                ++w;
                acc >>= 32;
                fill -= 32;
            }
        };
        int k = k0;
        for (; k < k0 + nwb; k += 4) { // whole words of an unmatched cell: a match of four bytes or four literals
            const uint32_t wp = ls.pos + (uint32_t)k, d = wdist[wp >> 2];
            if (d) {
                if (fill > 0) atomicOr(&out[w], (uint32_t)acc);
                unsigned long long bb;
                int n;
                match_code(len_tab, dist_tab, 4, (int)d, bb, n);
                at = w * 32u + (unsigned)fill;
                put_bits64(out, at, bb, n);
                at += (unsigned)n;
                w = at >> 5;
                fill = (int)(at & 31u);
                acc = 0ull;
            } else {
                const uint32_t v = word_at(in, wp);
                pair(lit_tab[v & 0xFFu], lit_tab[(v >> 8) & 0xFFu]);
                pair(lit_tab[(v >> 16) & 0xFFu], lit_tab[v >> 24]);
            }
        }
        for (; k < k1; k += 2) {
            const uint32_t ea = lit_tab[in[ls.pos + k]], eb = k + 1 < k1 ? lit_tab[in[ls.pos + k + 1]] : 0u; // past the end: no bits
            pair(ea, eb);
        }
        if (fill > 0) atomicOr(&out[w], (uint32_t)acc);
    }
    DSYNC();
    PROF(7); // emission
    // ---- the BGZF block: header, deflate data, CRC32, ISIZE -> its slot of the staging buffer
    const uint32_t nbytes = (total_bits_s + (eob_s >> 16) + 7u) >> 3; // + the end-of-block code, rounded up to a byte
    const uint32_t bsize = 18u + nbytes + 8u;
    if (tid < 18) {
        const uint8_t hdr[18] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, (uint8_t)((bsize - 1u) & 0xFFu), (uint8_t)((bsize - 1u) >> 8)};
        dst[tid] = hdr[tid];
    }
    {
        uint32_t* const dw = reinterpret_cast<uint32_t*>(dst + 18);
        const uint8_t* const ob = reinterpret_cast<const uint8_t*>(out);
        for (uint32_t i = tid; i < (nbytes >> 2); i += DT) __stcs(dw + i, out[i]);
        if (tid < (nbytes & 3u)) dst[18 + (nbytes & ~3u) + tid] = ob[(nbytes & ~3u) + tid];
    }
    asm volatile("bar.sync 4, %0;" ::"n"(BGZF_THREADS) : "memory"); // the CRC warps are done
    if (tid < 8) {
        const uint32_t v = tid < 4 ? crc_s : (uint32_t)L;
        dst[18 + nbytes + tid] = (uint8_t)(v >> (8 * (tid & 3)));
    }
    if (tid == 0) a.blk_size[blk] = bsize;
    PROF(11); // copy out (thread 0's share)
}

// Persistent CTAs (one per SM: the shared-memory budget), blocks b, b + grid, ...: no CTA launch between blocks, the tables are
// loaded once, and the next block's bytes are pulled into L2 while this one is compressed.
__global__ void __launch_bounds__(BGZF_THREADS, 1) k_bgzf_deflate(const BgzfArgs a)
{
    extern __shared__ __align__(16) unsigned char sm[];
    __shared__ uint32_t crc_tab[1024]; // slicing-by-four tables of CRC-32
    __shared__ uint32_t lit_tab[256], len_tab[256], dist_tab[32]; // the context's prefix code (BgzfCode)
    const int tid = threadIdx.x;
    const long long total = a.totals[3];
    if (total > a.in_cap) return;
    long long nblk = (total + BGZF_IN - 1) / BGZF_IN;
    if (a.hist && nblk > 8192) nblk = 8192; // the statistics pass looks at the head of the stream
    crc_tab[tid] = __ldg(a.crc_pow + 1024 + tid);
    if (tid < 256) {
        lit_tab[tid] = __ldg(a.code->lit + tid);
        len_tab[tid] = __ldg(a.code->len + tid);
        if (tid < 32) dist_tab[tid] = __ldg(a.code->dist + tid);
    }
    const uint32_t eob = __ldg(&a.code->eob), hdr_bits = __ldg(&a.code->hdr_bits);
    __syncthreads();
    for (long long blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const long long nb0 = (blk + gridDim.x) * BGZF_IN;
        if (blk + gridDim.x < nblk && tid < 256 && nb0 + 128ll * tid < total) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.in + nb0 + 128ll * tid));
        deflate_block(a, (int)blk, sm, crc_tab, lit_tab, len_tab, dist_tab, eob, hdr_bits);
        __syncthreads(); // the block's shared memory is free again
    }
}

// exclusive prefix of the block sizes; the totals for the host: [4] compressed bytes, [5] blocks
__global__ void __launch_bounds__(1024) k_bgzf_scan(const BgzfArgs a)
{
    __shared__ long long warp_sum[32];
    __shared__ long long carry_s;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const long long total = a.totals[3];
    const int nblk = total > a.in_cap ? 0 : (int)((total + BGZF_IN - 1) / BGZF_IN);
    if (tid == 0) carry_s = 0;
    __syncthreads();
    for (int base = 0; base < nblk; base += 1024) {
        const int i = base + tid;
        const long long v = i < nblk ? (long long)a.blk_size[i] : 0;
        long long x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) warp_sum[w] = x;
        __syncthreads();
        if (w == 0) {
            long long t = warp_sum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long y = __shfl_up_sync(0xffffffffu, t, o);
                if (lane >= o) t += y;
            }
            warp_sum[lane] = t;
        }
        __syncthreads();
        const long long incl = carry_s + (w ? warp_sum[w - 1] : 0) + x;
        if (i < nblk) a.blk_off[i] = incl - v;
        __syncthreads();
        if (tid == 1023) carry_s = incl;
        __syncthreads();
    }
    if (tid == 0) {
        a.totals[4] = carry_s;
        a.totals[5] = nblk;
    }
}

__global__ void __launch_bounds__(256) k_bgzf_pack(const BgzfArgs a)
{
    const long long total = a.totals[3];
    const int nblk = total > a.in_cap ? 0 : (int)((total + BGZF_IN - 1) / BGZF_IN);
    for (int b = blockIdx.x; b < nblk; b += gridDim.x) {
        const uint8_t* src = a.stage + (size_t)b * BGZF_STRIDE + 2;
        uint8_t* dst = a.out + a.blk_off[b];
        const uint32_t n = a.blk_size[b];
        // aligned words of the destination, edges by bytes
        const uint32_t head = (uint32_t)((4u - ((uintptr_t)dst & 3u)) & 3u);
        for (uint32_t i = threadIdx.x; i < min(head, n); i += 256) dst[i] = src[i];
        if (n > head) {
            const uint32_t words = (n - head) >> 2;
            for (uint32_t w = threadIdx.x; w < words; w += 256) {
                const uint8_t* s = src + head + 4u * w;
                *reinterpret_cast<uint32_t*>(dst + head + 4u * w) = (uint32_t)s[0] | ((uint32_t)s[1] << 8) | ((uint32_t)s[2] << 16) | ((uint32_t)s[3] << 24);
            }
            for (uint32_t i = head + 4u * words + threadIdx.x; i < n; i += 256) dst[i] = src[i];
        }
    }
}

} // namespace

#ifdef BGZF_PROF
extern "C" void vgl_bgzf_prof_dump()
{
    unsigned long long h[16];
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(h, g_bgzf_prof, sizeof h);
    static const char* names[12] = {"load+crc||ranges", "segment table", "hash insert", "match", "word insert", "bit lengths + words", "prefix", "emission",
                                    "  w1: issue loads", "  w1: bar 1", "  w1: crc", "copy out"};
    unsigned long long tot = 0;
    for (int i = 0; i < 8; ++i) tot += h[i];
    tot += h[11];
    fprintf(stderr, "bgzf cycles (thread 0, all blocks) %.4g\n", (double)tot);
    for (int i = 0; i < 12; ++i) fprintf(stderr, "bgzf phase %-18s %6.2f %%\n", names[i], 100.0 * (double)h[i] / (double)(tot ? tot : 1));
    memset(h, 0, sizeof h);
    cudaMemcpyToSymbol(g_bgzf_prof, h, sizeof h);
}
#endif

size_t bgzf_dyn_smem() { return (size_t)BGZF_IN + (size_t)OUT_WORDS * 4 + (size_t)MAX_SEG * (sizeof(Seg) + 4 + 2) + (size_t)HASH_SLOTS * 4 + (size_t)MAX_RANGES * 16; }

// blocks a record stream of `bytes` bytes makes
int64_t bgzf_blocks_for(int64_t bytes) { return (bytes + BGZF_IN - 1) / BGZF_IN; }

// [0..1023] x^(8 * CRC_CHUNK * k) mod P (reflected CRC-32 representation); [1024..2047] the slicing-by-four tables of CRC-32:
// T_lvl[i] = the CRC register after byte i and lvl zero bytes
void bgzf_crc_pow_table(uint32_t* t)
{
    uint32_t x8 = 1u << 31; // x^0
    for (int k = 0; k < 8; ++k) x8 = crc_mul(x8, 1u << 30); // times x
    uint32_t xc = 1u << 31;
    for (int k = 0; k < CRC_CHUNK; ++k) xc = crc_mul(xc, x8);
    t[0] = 1u << 31;
    for (int k = 1; k < 1024; ++k) t[k] = crc_mul(t[k - 1], xc);
    uint32_t* const tab = t + 1024;
    for (uint32_t i = 0; i < 256; ++i) {
        uint32_t c = i;
        for (int k = 0; k < 8; ++k) c = (c & 1u) ? (c >> 1) ^ 0xEDB88320u : c >> 1;
        tab[i] = c;
    }
    for (int lvl = 1; lvl < 4; ++lvl)
        for (uint32_t i = 0; i < 256; ++i) tab[256 * lvl + i] = tab[tab[256 * (lvl - 1) + i] & 0xFFu] ^ (tab[256 * (lvl - 1) + i] >> 8);
}

void launch_bgzf(const BgzfArgs& a, int64_t max_blocks, cudaStream_t st, int n_sms)
{
    cudaFuncSetAttribute(k_bgzf_deflate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bgzf_dyn_smem()); // per device
    k_bgzf_first<<<(unsigned)std::min<int64_t>((max_blocks + 255) / 256, 4096), 256, 0, st>>>(a);
    k_bgzf_ranges<<<(unsigned)((max_blocks + 7) / 8), 256, 0, st>>>(a);
    const unsigned grid = (unsigned)std::min<int64_t>(max_blocks, n_sms);
    k_bgzf_deflate<<<grid, BGZF_THREADS, bgzf_dyn_smem(), st>>>(a);
    if (a.hist) return; // symbol statistics of (at most the first 8192 blocks of) this record stream
    k_bgzf_scan<<<1, 1024, 0, st>>>(a);
    k_bgzf_pack<<<(unsigned)(n_sms * 8), 256, 0, st>>>(a);
}

} // namespace vgl
