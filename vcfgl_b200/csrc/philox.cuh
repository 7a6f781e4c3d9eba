// Philox4x32-10 counter-based RNG (Salmon et al., SC'11) and the keying used by
// the native simulator.  Every draw is a pure function of
//   key     = (seed_lo, seed_hi)
//   counter = (site_lo, site_hi8 | read << 8, sample, purpose << 24 | block)
// so a run is reproducible for any batch size, slot count or GPU count
// (north_star; replaces the reference's four sequential libc streams,
// SURVEY.md 3.4: rng.h:8-12, io.cpp:1047-1061).
#pragma once
#include <math.h>
#include <stdint.h>

namespace vgl {

enum Purpose : uint32_t {
    P_DEPTH = 0,   // per cell: Poisson depth
    P_READ = 1,    // per read: haplotype, error test, wrong base, strand, tail distance
    P_SITE = 2,    // per site: beta-distributed error rate (--error-qs 1)
    P_QS = 3,      // per read: beta-distributed error probability (--error-qs 2)
    P_SUBSAMPLE = 4, // per cell: which 255 reads errmod keeps when depth > 255
    P_COUNTS = 5,  // per cell: count-level sampler (binomial / multinomial splits)
    P_STRAND = 6,  // per cell, tile kernel with strand totals: bit r of the stream = read r (reads grouped A, C, G, T) is forward
    P_TAIL = 7,    // per cell, tile kernel with I16: tail distances, twelve reads per block
    P_LAST = 8     // per site, tile kernel with I16: which read of the site's last cell with reads is "the last read" (vcfgl.cpp:657)
};

struct u32x4 {
    uint32_t x, y, z, w;
};

__host__ __device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t b)
{
#ifdef __CUDA_ARCH__
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}

__host__ __device__ __forceinline__ u32x4 philox4x32_10(u32x4 c, uint32_t k0, uint32_t k1)
{
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = mulhi32(M0, c.x), lo0 = M0 * c.x;
        const uint32_t hi1 = mulhi32(M1, c.z), lo1 = M1 * c.z;
        u32x4 n;
        n.x = hi1 ^ c.y ^ k0;
        n.y = lo1;
        n.z = hi0 ^ c.w ^ k1;
        n.w = lo0;
        c = n;
        k0 += W0;
        k1 += W1;
    }
    return c;
}

struct Key {
    uint32_t k0, k1;
};

__host__ __device__ __forceinline__ u32x4 draw(Key key, int64_t site, uint32_t sample, uint32_t read,
                                               uint32_t purpose, uint32_t block)
{
    u32x4 c;
    c.x = (uint32_t)site;
    c.y = ((uint32_t)((uint64_t)site >> 32) & 0xFFu) | (read << 8);
    c.z = sample;
    c.w = (purpose << 24) | (block & 0xFFFFFFu);
    return philox4x32_10(c, key.k0, key.k1);
}

// uniform in (0,1), 32-bit resolution, never 0 or 1
__host__ __device__ __forceinline__ double u01_32(uint32_t w) { return ((double)w + 0.5) * 2.3283064365386963e-10; }
// uniform in (0,1), 53-bit resolution, never 0 or 1: 2^53 - 1 + 0.5 rounds to 2^53, so the top value is clamped to the
// largest double below 1 (no other value reaches it)
__host__ __device__ __forceinline__ double u01_53(uint32_t hi, uint32_t lo)
{
    const uint64_t v = ((uint64_t)hi << 21) ^ (uint64_t)(lo >> 11); // 53 bits
    return fmin(((double)v + 0.5) * 1.1102230246251565e-16, 0x1.fffffffffffffp-1);
}

// sequential stream of 32-bit words for rejection samplers (one Philox block per 4 words)
struct Stream {
    Key key;
    int64_t site;
    uint32_t sample, read, purpose, block;
    u32x4 buf;
    int have;
    __device__ __forceinline__ void init(Key k, int64_t s, uint32_t smp, uint32_t rd, uint32_t p)
    {
        key = k; site = s; sample = smp; read = rd; purpose = p; block = 0; have = 0;
    }
    __device__ __forceinline__ uint32_t next()
    {
        if (have == 0) {
            buf = draw(key, site, sample, read, purpose, block++);
            have = 4;
        }
        uint32_t v = buf.x;
        buf.x = buf.y; buf.y = buf.z; buf.z = buf.w;
        --have;
        return v;
    }
    __device__ __forceinline__ double uniform() { const uint32_t a = next(), b = next(); return u01_53(a, b); }
};

} // namespace vgl
