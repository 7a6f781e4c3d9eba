// Host-side constant tables.  Compiled with -ffp-contract=off: the table values
// must equal the reference's bit for bit (plain x86-64 SSE2 double arithmetic,
// separate multiply and add roundings), because GL model 1 likelihoods are sums
// of table entries.
#include "tables.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <utility>
#include <vector>

namespace vgl {

const double kLutLog10Gl[3][257] = {
#include "lut_log10_gl.inc"
};

namespace {
// log C(n, k), 1 <= k <= n < 256; 0 elsewhere (errmod.c:51-64)
std::vector<double> log_binomial()
{
    std::vector<double> t(256 * 256, 0.0);
    std::vector<double> lfact(256);
    for (int n = 0; n < 256; ++n) lfact[n] = lgamma(n + 1);
    for (int n = 1; n < 256; ++n)
        for (int k = 1; k <= n; ++k) t[n << 8 | k] = lfact[n] - lfact[k] - lfact[n - k];
    return t;
}
} // namespace

void ErrmodTables::build(double depcorr, double eta)
{
    const std::vector<double> lc = log_binomial();
    fk.assign(256, 0.0);
    fk[0] = 1.0;
    for (int n = 1; n < 256; ++n) fk[n] = pow(1. - depcorr, n) * (1.0 - eta) + eta; // errmod.c:75-77

    beta.assign((size_t)64 * 256 * 256, 0.0);
    for (int q = 1; q < 64; ++q) { // errmod.c:86-99
        const double e = pow(10.0, -q / 10.0);
        const double le = log(e), le1 = log(1.0 - e);
        for (int n = 1; n <= 255; ++n) {
            double* row = beta.data() + ((size_t)q << 16 | (size_t)n << 8);
            double upper = lc[n << 8 | n] + n * le; // log of the binomial tail P(K >= k+1)
            row[n] = HUGE_VAL;
            for (int k = n - 1; k >= 0; --k) {
                const double with_k = upper + log1p(exp(lc[n << 8 | k] + k * le + (n - k) * le1 - upper));
                row[k] = -10. / M_LN10 * (upper - with_k);
                upper = with_k;
            }
        }
    }
    lhet.assign(256 * 256, 0.0);
    for (int n = 0; n < 256; ++n) // errmod.c:107-109
        for (int k = 0; k < 256; ++k) lhet[n << 8 | k] = lc[n << 8 | k] - M_LN2 * n;
}

std::vector<double> ErrmodTables::fixed_q_bsum(int q) const
{
    if (q < 4) q = 4; // errmod.c:168-169
    if (q > 63) q = 63;
    std::vector<double> t(256 * 256, 0.0);
    for (int n = 1; n <= 255; ++n) {
        const double* row = beta.data() + ((size_t)q << 16 | (size_t)n << 8);
        double acc = 0.0;
        for (int c = 0; c < n; ++c) {
            acc += fk[c] * row[c]; // two roundings; must not be contracted into an FMA
            t[n << 8 | (c + 1)] = acc;
        }
    }
    return t;
}

std::vector<double> ErrmodTables::het_term() const
{
    std::vector<double> t(256 * 256);
    for (int i = 0; i < 256 * 256; ++i) t[i] = -4.343 * lhet[i];
    return t;
}

std::vector<unsigned long long> poisson_cdf_u64(double lambda, int max_n)
{
    std::vector<unsigned long long> t;
    const long double two64 = 18446744073709551616.0L;
    long double cdf = 0.0L;
    for (int k = 0; k < max_n; ++k) {
        long double pmf;
        if (lambda <= 0.0) pmf = k == 0 ? 1.0L : 0.0L;
        else pmf = expl(-(long double)lambda + k * logl((long double)lambda) - lgammal((long double)k + 1.0L));
        cdf += pmf;
        // stop once the remaining tail is below the 2^-64 resolution of the uniform
        if (cdf >= 1.0L - 1e-19L || (k > lambda && pmf < 1e-22L) || k == max_n - 1) {
            t.push_back(~0ull);
            break;
        }
        const long double scaled = cdf * two64;
        t.push_back(scaled >= two64 ? ~0ull : (unsigned long long)scaled);
    }
    return t;
}

std::vector<unsigned long long> poisson_alias_u64(const std::vector<unsigned long long>& cdf)
{
    typedef unsigned __int128 u128;
    const int K = 256;
    if (cdf.empty() || cdf.size() > (size_t)K) return {};
    const u128 one = (u128)1 << 64;
    // mass of outcome k scaled by K, in units of 2^-64 of a column: m[k] = K * pmf[k], sum = K * 2^64
    std::vector<u128> m(K, 0);
    u128 prev = 0;
    for (size_t k = 0; k < cdf.size(); ++k) {
        const u128 c = k + 1 == cdf.size() ? one : (u128)cdf[k];
        m[k] = (c - prev) * K;
        prev = c;
    }
    std::vector<unsigned long long> out(K);
    std::vector<int> small, large;
    for (int k = 0; k < K; ++k) (m[k] < one ? small : large).push_back(k);
    std::vector<u128> stay(K, one);
    std::vector<int> alias(K);
    for (int k = 0; k < K; ++k) alias[k] = k;
    while (!small.empty() && !large.empty()) {
        const int s = small.back(), l = large.back();
        small.pop_back();
        stay[s] = m[s];
        alias[s] = l;
        m[l] -= one - m[s];
        if (m[l] < one) {
            large.pop_back();
            small.push_back(l);
        }
    }
    // leftovers hold exactly one column each (integer arithmetic: no rounding residue)
    for (int k = 0; k < K; ++k) {
        if (alias[k] == k) { out[k] = (unsigned long long)k; continue; } // threshold irrelevant: both branches give k
        const u128 t56 = (stay[k] + 255) >> 8; // frac56 < ceil(stay / 256)  <=>  frac56 * 256 < stay
        out[k] = (unsigned long long)(t56 << 8) | (unsigned long long)alias[k];
    }
    return out;
}

std::vector<uint32_t> binomial_cdf4_u32(double e)
{
    std::vector<uint32_t> t(256 * 4, 0xFFFFFFFFu);
    if (!(e > 0.0)) return t; // never an error: every u < 2^32-1 gives E = 0
    // P(E = j) by the ratio recurrence from (1 - e)^n: every step is one rounded operation, so a CDF that is a short dyadic
    // fraction (e = 1/4, 1/2) comes out exact and its floor is not one short
    const long double E = e, Q = 1.0L - E;
    for (int n = 0; n < 256; ++n) {
        long double cdf = 0.0L, pj = powl(Q, n);
        for (int j = 0; j < 4 && j <= n; ++j) {
            if (j > 0) pj = pj * (n - j + 1) * E / (j * Q);
            cdf += pj;
            const long double sc = cdf * 4294967296.0L;
            t[n * 4 + j] = sc >= 4294967295.0L ? 0xFFFFFFFFu : (uint32_t)sc;
        }
    }
    return t;
}

double inc_beta(double a, double b, double x)
{
    if (!(x > 0.0)) return 0.0;
    if (!(x < 1.0)) return 1.0;
    // use the symmetry I_x(a,b) = 1 - I_{1-x}(b,a) where the continued fraction converges fast
    const bool flip = x > (a + 1.0) / (a + b + 2.0);
    const double aa = flip ? b : a, bb = flip ? a : b, xx = flip ? 1.0 - x : x;
    const double lfront = lgamma(aa + bb) - lgamma(aa) - lgamma(bb) + aa * log(xx) + bb * log1p(-xx);
    const double tiny = 1e-300;
    double c = 1.0, d = 1.0 - (aa + bb) * xx / (aa + 1.0);
    if (fabs(d) < tiny) d = tiny;
    d = 1.0 / d;
    double h = d;
    for (int m = 1; m <= 20000; ++m) {
        const double m2 = 2.0 * m;
        double num = m * (bb - m) * xx / ((aa + m2 - 1.0) * (aa + m2));
        d = 1.0 + num * d; if (fabs(d) < tiny) d = tiny;
        c = 1.0 + num / c; if (fabs(c) < tiny) c = tiny;
        d = 1.0 / d;
        h *= d * c;
        num = -(aa + m) * (aa + bb + m) * xx / ((aa + m2) * (aa + m2 + 1.0));
        d = 1.0 + num * d; if (fabs(d) < tiny) d = tiny;
        c = 1.0 + num / c; if (fabs(c) < tiny) c = tiny;
        d = 1.0 / d;
        const double del = d * c;
        h *= del;
        if (fabs(del - 1.0) < 1e-16) break;
    }
    const double v = exp(lfront) * h / aa;
    return flip ? 1.0 - v : v;
}

// Walker alias over 256 columns of capacity 2^24 each for integer weights that sum to 2^32 (exact integer arithmetic):
// entry = stay24 << 8 | alias; a draw keeps its column when its low 24 bits are below stay24
static std::vector<uint32_t> walker_alias24(const std::vector<unsigned long long>& w)
{
    typedef unsigned long long u64;
    const int K = 256;
    const u64 cap = 1ull << 24;
    std::vector<u64> m(K, 0);
    for (size_t i = 0; i < w.size() && i < (size_t)K; ++i) m[i] = w[i];
    std::vector<int> small, large, alias(K);
    std::vector<u64> stay(K, cap);
    for (int k = 0; k < K; ++k) { alias[k] = k; (m[k] < cap ? small : large).push_back(k); }
    while (!small.empty() && !large.empty()) {
        const int s = small.back(), l = large.back();
        small.pop_back();
        stay[s] = m[s];
        alias[s] = l;
        m[l] -= cap - m[s];
        if (m[l] < cap) { large.pop_back(); small.push_back(l); }
    }
    // leftovers hold exactly one column each (integer arithmetic): alias = itself, any threshold
    std::vector<uint32_t> out(K, 0u);
    for (int k = 0; k < K; ++k) {
        if (alias[k] == k) out[k] = (uint32_t)((cap - 1) << 8) | (uint32_t)k;
        else out[k] = (uint32_t)(stay[k] << 8) | (uint32_t)alias[k];
    }
    return out;
}

std::vector<uint32_t> qs_class_table(double a, double b, double shift, bool use_bins, const uint8_t* bin_lut, int bin_max,
                                     std::vector<double>* prob, std::vector<int>* q_values, int* dominant, double* p_minor)
{
    typedef unsigned long long u64;
    if (!(shift >= 0.0)) return {};
    const int KMAX = 420; // phred beyond this has no representable mass for any admissible Beta
    // mass[q] = P(final quality score q), q = 0..255; [256]: scores beyond the last --qs-bins range
    std::vector<long double> mass(257, 0.0L);
    for (int k = 0; k <= KMAX; ++k) {
        // q index k <=> phred + shift in [k, k+1) (k = 0 also takes the part below 0 of the shifted axis: (int) truncates)
        double lo = k == 0 ? 0.0 : (double)k - shift, hi = (double)k + 1.0 - shift;
        if (k == KMAX) hi = INFINITY;
        if (hi <= 0.0) continue;
        if (lo < 0.0) lo = 0.0;
        const double p_hi = pow(10.0, -lo / 10.0), p_lo = std::isinf(hi) ? 0.0 : pow(10.0, -hi / 10.0);
        const long double P = (long double)inc_beta(a, b, p_hi) - (long double)inc_beta(a, b, p_lo);
        if (!(P > 0.0L)) continue;
        int q;
        if (use_bins) q = k > bin_max ? 256 : bin_lut[k];
        else q = k > 63 ? 63 : k;
        mass[q] += P;
    }
    // classes with mass, quantised to 2^-32 with the rounding residue given to the heaviest class
    std::vector<int> cls_info;
    std::vector<u64> wq;
    long double total = 0.0L;
    for (long double m : mass) total += m;
    if (!(total > 0.5L)) return {};
    u64 sum = 0;
    int heavy = 0;
    for (int i = 0; i < 257; ++i) {
        const u64 w = (u64)(mass[i] / total * 4294967296.0L + 0.5L);
        if (w == 0) continue;
        cls_info.push_back(i < 256 ? i : (1 << 9)); // out of range: score 0 + flag (what bin_qs() of the per-read kernels returns)
        wq.push_back(w);
        if (w > wq[heavy]) heavy = (int)wq.size() - 1;
        sum += w;
    }
    const int K = 256;
    if (wq.empty() || (int)wq.size() > K) return {};
    const u64 one32 = 1ull << 32;
    if (sum > one32) { if (wq[heavy] <= sum - one32) return {}; wq[heavy] -= sum - one32; }
    else wq[heavy] += one32 - sum;
    if (prob) {
        prob->assign(257, 0.0);
        for (size_t i = 0; i < wq.size(); ++i) (*prob)[((cls_info[i] >> 9) & 1) ? 256 : (cls_info[i] & 0xFF)] = (double)wq[i] / 4294967296.0;
    }
    std::vector<uint32_t> out(768, 0u);
    {
        const std::vector<uint32_t> al = walker_alias24(wq);
        for (int k = 0; k < K; ++k) out[k] = al[k];
    }
    // the conditional law of the classes other than the heaviest one ("minor" classes), quantised to 2^-32 again:
    // the tile kernel draws how many reads of a cell are minor, then their classes from this table
    {
        std::vector<u64> wm(wq.size(), 0);
        const u64 rest = one32 - wq[heavy];
        if (rest == 0) {
            wm[heavy] = one32; // a single class: the table is never consulted
        } else {
            u64 s2 = 0;
            int big = -1;
            for (size_t i = 0; i < wq.size(); ++i) {
                if ((int)i == heavy) continue;
                wm[i] = (u64)((long double)wq[i] / (long double)rest * 4294967296.0L + 0.5L);
                s2 += wm[i];
                if (big < 0 || wm[i] > wm[big]) big = (int)i;
            }
            if (s2 > one32) wm[big] -= s2 - one32;
            else wm[big] += one32 - s2;
        }
        const std::vector<uint32_t> al = walker_alias24(wm);
        for (int k = 0; k < K; ++k) out[512 + k] = al[k];
    }
    if (dominant) *dominant = heavy;
    if (p_minor) *p_minor = (double)((long double)(one32 - wq[heavy]) / 4294967296.0L);
    // dense index of the quality scores in use (ascending)
    std::vector<int> qidx(256, -1), qv;
    for (int q = 0; q < 256; ++q)
        for (int ci : cls_info)
            if ((ci & 0xFF) == q && qidx[q] < 0) { qidx[q] = (int)qv.size(); qv.push_back(q); }
    if (q_values) *q_values = qv;
    for (size_t i = 0; i < cls_info.size(); ++i) out[256 + i] = (uint32_t)cls_info[i] | ((uint32_t)qidx[cls_info[i] & 0xFF] << 16);
    return out;
}

std::vector<double> m2_const_table(const std::vector<double>& c)
{
    const size_t nq = c.size() / 3;
    std::vector<double> t(nq * M2_TAB_DOUBLES, 0.0);
    for (size_t q = 0; q < nq; ++q) {
        const double c2 = c[3 * q], c1 = c[3 * q + 1], c0 = c[3 * q + 2];
        double* tq = t.data() + q * M2_TAB_DOUBLES;
        for (int b = 0; b < 4; ++b)
            for (int k = 0; k < 5; ++k)
                for (int j = 0; j <= k; ++j) {
                    const int hits = (j == b) + (k == b);
                    tq[b * 17 + k * (k + 1) / 2 + j] = hits == 2 ? c2 : (hits == 1 ? c1 : c0);
                }
        double* tc = tq + 68;
        // classes: 0 xx, 1 xy, 2 yy, 3 x., 4 y., 5 ..   [0]: the read is y, [1]: the read is x
        const double rx[6] = {c2, c1, c0, c1, c0, c0}, ry[6] = {c0, c1, c2, c0, c1, c0};
        for (int i = 0; i < 6; ++i) { tc[i] = ry[i]; tc[8 + i] = rx[i]; }
    }
    return t;
}

bool m2_pure_table(const std::vector<double>& c, std::vector<float>* out)
{
    const size_t nq = c.size() / 3;
    out->assign(nq * 65 * 2, 0.0f);
    for (size_t q = 0; q < nq; ++q) {
        const double c2 = c[3 * q], c1 = c[3 * q + 1], c0 = c[3 * q + 2];
        if (!(c2 >= c1 && c2 >= c0)) return false; // the matching homozygote would not be the running maximum
        float v2 = -0.0f, v1 = -0.0f, v0 = -0.0f; // bcf_utils.h:310
        for (int n = 0; n <= 64; ++n) {
            (*out)[(q * 65 + n) * 2] = v1;
            (*out)[(q * 65 + n) * 2 + 1] = v0;
            // one more read of x (gl_methods.cpp:27-58): float += double, then the maximum is subtracted in float
            const float a2 = (float)((double)v2 + c2), a1 = (float)((double)v1 + c1), a0 = (float)((double)v0 + c0);
            v2 = a2 - a2;
            v1 = a1 - a2;
            v0 = a0 - a2;
        }
    }
    return true;
}

std::vector<uint32_t> m2_class_map()
{
    std::vector<uint32_t> m(16 * 8, 0u);
    for (int x = 0; x < 4; ++x)
        for (int y = 0; y < 4; ++y) {
            if (x == y) continue;
            uint32_t* e = m.data() + (x * 4 + y) * 8;
            unsigned long long ids = 0;
            unsigned mask[6] = {0, 0, 0, 0, 0, 0};
            for (int k = 0; k < 5; ++k)
                for (int j = 0; j <= k; ++j) {
                    const int rj = j == x ? 0 : (j == y ? 1 : 2), rk = k == x ? 0 : (k == y ? 1 : 2);
                    const int hi = rj > rk ? rj : rk, lo = rj > rk ? rk : rj;
                    const int cls = hi * (hi + 1) / 2 + lo, pair = k * (k + 1) / 2 + j;
                    ids |= (unsigned long long)cls << (3 * pair);
                    mask[cls] |= 1u << pair;
                }
            e[0] = mask[0] | (mask[1] << 16);
            e[1] = mask[2] | (mask[3] << 16);
            e[2] = mask[4] | (mask[5] << 16);
            e[4] = (uint32_t)ids;
            e[5] = (uint32_t)(ids >> 32);
        }
    return m;
}

bool ErrmodTables::scores_safe_for_fast_div(const std::vector<double>& bsum, const std::vector<double>& het)
{
    const double lo = ldexp(1.0, -100), hi = ldexp(1.0, 100);
    for (const std::vector<double>* t : {&bsum, &het})
        for (double v : *t) {
            if (!(v >= 0.0) || v > hi) return false;        // negative, NaN or huge
            if (v != 0.0 && v < lo) return false;           // positive but tiny
        }
    return true;
}

static int bin_lookup(int n_bins, const uint8_t bins[][3], int qs)
{
    for (int i = 0; i < n_bins; ++i)
        if (qs >= bins[i][0] && qs <= bins[i][1]) return bins[i][2];
    return -1000;
}

int precalc(double error_rate, int error_qs, int gl_model, int precise_gl, int adjust_qs, double adjust_by,
            int n_bins, const uint8_t bins[][3], PreCalc* out)
{
    *out = PreCalc();
    if (error_qs == 2) return 0; // per-read quality scores: nothing to precompute
    int qs, adj = -1;
    if (error_rate == 0.0) {
        qs = adj = 63;
    } else if (error_rate == 1.0) {
        qs = adj = 0;
    } else {
        const double phred = -10.0 * log10(error_rate);
        qs = (int)phred;
        if (adjust_qs) adj = (int)(phred + adjust_by);
    }
    if (n_bins) {
        qs = bin_lookup(n_bins, bins, qs);
        if (adjust_qs) adj = bin_lookup(n_bins, bins, adj);
        if (qs < 0 || (adjust_qs && adj < 0)) return -1;
    } else {
        if (qs > 63) qs = 63;
        if (adjust_qs && adj > 63) adj = 63;
    }
    if (qs < 0 || (adjust_qs && adj < 0)) return -1; // a negative --adjust-by can push the score below 0: the tables have no such row
    out->qs = qs;
    if (adjust_qs) out->adj_qs = adj;
    if (gl_model == 2) {
        if (!precise_gl) {
            const int q = (adjust_qs & 1) ? out->adj_qs : out->qs;
            out->homT = kLutLog10Gl[0][q];
            out->het = kLutLog10Gl[1][q];
            out->homF = kLutLog10Gl[2][q];
        } else if (error_rate == 0.0) {
            out->homT = 0;
            out->het = -0.3010299956639812;
            out->homF = -INFINITY;
        } else {
            out->homT = log10(1.0 - error_rate);
            out->het = log10((1.0 - error_rate) / 2.0 + error_rate / 6.0);
            out->homF = log10(error_rate) - 0.47712125471966244;
        }
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// Prefix codes for csrc/bgzf.cu (RFC 1951)
namespace {

// code lengths of a Huffman code over the symbols with cnt > 0, none longer than max_bits (counts are halved until the
// tree is shallow enough: the classic fallback, a fraction of a percent from package-merge on skewed inputs)
std::vector<int> huff_lengths(std::vector<uint64_t> cnt, int max_bits)
{
    const int n = (int)cnt.size();
    std::vector<int> len(n, 0);
    int used = 0, one = -1;
    for (int i = 0; i < n; ++i)
        if (cnt[i]) { ++used; one = i; }
    if (used == 0) return len;
    if (used == 1) { // a complete code needs two codewords (zlib rejects incomplete literal / code-length codes)
        len[one] = 1;
        len[one == 0 ? 1 : 0] = 1;
        return len;
    }
    for (;;) {
        // two-queue construction over the sorted leaves
        std::vector<int> order;
        for (int i = 0; i < n; ++i)
            if (cnt[i]) order.push_back(i);
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return cnt[a] < cnt[b]; });
        const int m = (int)order.size();
        std::vector<uint64_t> w(2 * m - 1);
        std::vector<int> parent(2 * m - 1, -1);
        for (int i = 0; i < m; ++i) w[i] = cnt[order[i]];
        int leaf = 0, node = m, next = m;
        auto take = [&]() -> int {
            if (leaf < m && (node >= next || w[leaf] <= w[node])) return leaf++;
            return node++;
        };
        while (next < 2 * m - 1) {
            const int a = take(), b = take();
            w[next] = w[a] + w[b];
            parent[a] = parent[b] = next;
            ++next;
        }
        int deepest = 0;
        for (int i = 0; i < m; ++i) {
            int d = 0;
            for (int j = i; parent[j] >= 0; j = parent[j]) ++d;
            len[order[i]] = d;
            deepest = std::max(deepest, d);
        }
        if (deepest <= max_bits) return len;
        for (int i = 0; i < n; ++i)
            if (cnt[i]) cnt[i] = (cnt[i] + 1) / 2;
    }
}

// canonical codes (RFC 1951 3.2.2), bit-reversed
std::vector<uint32_t> canon_codes(const std::vector<int>& len)
{
    int bl_count[17] = {0};
    for (int l : len) ++bl_count[l];
    bl_count[0] = 0;
    uint32_t next[17] = {0}, code = 0;
    for (int b = 1; b <= 16; ++b) {
        code = (code + (uint32_t)bl_count[b - 1]) << 1;
        next[b] = code;
    }
    std::vector<uint32_t> out(len.size(), 0u);
    for (size_t i = 0; i < len.size(); ++i) {
        if (!len[i]) continue;
        const uint32_t c = next[len[i]]++;
        uint32_t r = 0;
        for (int k = 0; k < len[i]; ++k) r |= ((c >> k) & 1u) << (len[i] - 1 - k);
        out[i] = r;
    }
    return out;
}

struct BitOut {
    uint32_t* w;
    uint32_t cap_bits, n = 0;
    void put(uint32_t v, int bits)
    {
        for (int k = 0; k < bits; ++k, ++n)
            if (n < cap_bits && ((v >> k) & 1u)) w[n >> 5] |= 1u << (n & 31);
    }
};

} // namespace

void bgzf_build_code(const uint32_t* hist, bool fixed, BgzfCode* out)
{
    memset(out, 0, sizeof(*out));
    std::vector<int> ll(288, 0), dl(30, 5);
    if (fixed) {
        for (int i = 0; i < 288; ++i) ll[i] = i < 144 ? 8 : (i < 256 ? 9 : (i < 280 ? 7 : 8));
    } else {
        std::vector<uint64_t> c(286), d(30);
        for (int i = 0; i < 286; ++i) c[i] = (uint64_t)hist[i] + 1; // every byte value and length must stay codable
        for (int i = 0; i < 30; ++i) d[i] = (uint64_t)hist[288 + i] + 1;
        const std::vector<int> l1 = huff_lengths(c, 15);
        std::copy(l1.begin(), l1.end(), ll.begin());
        dl = huff_lengths(d, 15);
    }
    const std::vector<uint32_t> lc = canon_codes(ll);
    std::vector<int> dl32(dl);
    if (fixed) dl32.resize(32, 5); // the fixed distance code has 32 codewords of 5 bits
    const std::vector<uint32_t> dc = canon_codes(dl32);
    for (int i = 0; i < 256; ++i) out->lit[i] = lc[i] | ((uint32_t)ll[i] << 16);
    out->eob = lc[256] | ((uint32_t)ll[256] << 16);
    for (int L = 3; L <= 258; ++L) {
        int idx, eb;
        uint32_t ev;
        const int t = L - 3;
        if (t < 8) { idx = t; eb = 0; ev = 0; }
        else if (L == 258) { idx = 28; eb = 0; ev = 0; }
        else {
            int hb = 0;
            while ((t >> (hb + 1)) != 0) ++hb;
            eb = hb - 2;
            idx = 4 * (hb - 1) + ((t >> eb) & 3);
            ev = (uint32_t)t & ((1u << eb) - 1u);
        }
        const int sym = 257 + idx, nb = ll[sym];
        out->len[t] = (lc[sym] | (ev << nb)) | ((uint32_t)(nb + eb) << 24);
    }
    for (int i = 0; i < 30; ++i) out->dist[i] = dc[i] | ((uint32_t)dl[i] << 16);
    BitOut bo{out->hdr, (uint32_t)(sizeof(out->hdr) * 8)};
    bo.put(1, 1); // BFINAL: every BGZF block is one deflate block
    if (fixed) {
        bo.put(1, 2);
    } else {
        bo.put(2, 2);
        // the 316 code lengths, run-length coded with the symbols 16 / 17 / 18 (3.2.7)
        std::vector<int> seq(ll.begin(), ll.begin() + 286);
        seq.insert(seq.end(), dl.begin(), dl.end());
        std::vector<std::pair<int, int>> rle; // symbol, extra value
        for (size_t i = 0; i < seq.size();) {
            size_t j = i;
            while (j < seq.size() && seq[j] == seq[i]) ++j;
            int run = (int)(j - i);
            const int v = seq[i];
            if (v == 0) {
                while (run >= 11) { const int r = std::min(run, 138); rle.push_back({18, r - 11}); run -= r; }
                if (run >= 3) { rle.push_back({17, run - 3}); run = 0; }
                while (run-- > 0) rle.push_back({0, 0});
            } else {
                rle.push_back({v, 0});
                --run;
                while (run >= 3) { const int r = std::min(run, 6); rle.push_back({16, r - 3}); run -= r; }
                while (run-- > 0) rle.push_back({v, 0});
            }
            i = j;
        }
        std::vector<uint64_t> cc(19, 0);
        for (auto& e : rle) ++cc[e.first];
        const std::vector<int> cl = huff_lengths(cc, 7);
        const std::vector<uint32_t> ccode = canon_codes(cl);
        static const int order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
        int hclen = 19;
        while (hclen > 4 && cl[order[hclen - 1]] == 0) --hclen;
        bo.put(286 - 257, 5);
        bo.put(30 - 1, 5);
        bo.put((uint32_t)(hclen - 4), 4);
        for (int i = 0; i < hclen; ++i) bo.put((uint32_t)cl[order[i]], 3);
        for (auto& e : rle) {
            bo.put(ccode[e.first], cl[e.first]);
            if (e.first == 16) bo.put((uint32_t)e.second, 2);
            else if (e.first == 17) bo.put((uint32_t)e.second, 3);
            else if (e.first == 18) bo.put((uint32_t)e.second, 7);
        }
    }
    out->hdr_bits = bo.n;
}

namespace {
// a BCF typed integer (bcf_enc_int1: type byte, then 1 / 2 / 4 little-endian bytes; other type codes take 4 bytes, as the
// device's parser reads them, bcf.cu read_typed_int); false when it runs past `end`
bool read_typed_int(const uint8_t*& p, const uint8_t* end, int64_t& v)
{
    if (p >= end) return false;
    const int t = *p & 0xF, w = t == 1 ? 1 : (t == 2 ? 2 : 4);
    if (end - p < 1 + w) return false;
    const uint8_t* r = p + 1;
    v = w == 1 ? (int8_t)r[0] : (w == 2 ? (int16_t)(r[0] | (r[1] << 8)) : (int32_t)(r[0] | (r[1] << 8) | (r[2] << 16) | ((uint32_t)r[3] << 24)));
    p += 1 + w;
    return true;
}
} // namespace

bool bcf_fmt_blocks_tile(const uint8_t* p, uint64_t len, uint32_t n_fmt, int64_t n_samples)
{
    if (n_samples < 1) return false;
    const uint8_t* const end = p + len;
    for (uint32_t k = 0; k < n_fmt; ++k) {
        int64_t key = 0, n = 0;
        if (!read_typed_int(p, end, key) || p >= end) return false;
        const int d = *p++, ty = d & 0xF;
        n = d >> 4;
        if (n == 15 && !read_typed_int(p, end, n)) return false;
        if (n < 0) return false;
        const uint64_t w = ty == 1 || ty == 7 ? 1 : (ty == 2 ? 2 : (ty == 0 ? 0 : 4)), rest = (uint64_t)(end - p);
        if (w && n && (uint64_t)n > rest / w / (uint64_t)n_samples) return false; // n x w x S > the bytes left (no overflow)
        p += (uint64_t)n * w * (uint64_t)n_samples;
    }
    return p == end;
}

// ---------------------------------------------------------------------------------------------------------------
// The kernel set of a context
const char* kernel_set_name(KernelSet k)
{
    static const char* const names[] = {"k_sim+k_site+k_scan+k_emit", "k_fused_m1f", "k_tile_m1f", "k_tile_m2", "k_truth_site+k_scan+k_truth_emit"};
    return names[k];
}

namespace {
// the model-2 tile kernel's tables: false when it cannot take the run (the per-read kernels keep the reference's behaviour)
bool plan_tile_m2(const vgl_params& p, RunPlan* k, PlanTables* tab)
{
    std::vector<double> consts; // (homT, het, homF) per quality score in use
    if (p.error_qs == 2) {
        std::vector<int> qv;
        tab->qcls = qs_class_table(k->beta_a, k->beta_b, (p.adjust_qs & 1) ? p.adjust_by : 0.0, p.n_qs_bins > 0, k->bin_lut, k->bin_max, nullptr,
                                   &qv, &k->q_dom, &k->q_minor);
        if (tab->qcls.empty()) return false; // classes outside the bins / too many
        k->q_dom_idx = (int)((tab->qcls[256 + k->q_dom] >> 16) & 0xFFu);
        for (int q : qv) consts.insert(consts.end(), {kLutLog10Gl[0][q], kLutLog10Gl[1][q], kLutLog10Gl[2][q]});
    } else
        consts = {k->pre.homT, k->pre.het, k->pre.homF};
    // the table-driven update needs constants that are negative (finite and non-zero, or -inf): see m2_f2d() in tile_m2.cu.
    // Not so e.g. under --precise-gl 1 with --error-rate 0 (homT = 0).
    if (!std::all_of(consts.begin(), consts.end(), [](double c) { return c < 0.0; })) return false;
    k->m2_nq = (int)consts.size() / 3;
    tab->m2_tab = m2_const_table(consts);
    if (!m2_pure_table(consts, &tab->m2_pure)) tab->m2_pure.clear();
    return true;
}
} // namespace

int plan_run(const vgl_params& p, const double* depth_means, bool allow_tile, RunPlan* k, PlanTables* tab, const char** why)
{
    auto fail = [why](int rc, const char* msg) { *why = msg; return rc; };
    // ---- derived run constants (vcfgl.cpp:1661-1766, rng.h:368-371)
    if (precalc(p.error_rate, p.error_qs, p.gl_model, p.precise_gl, p.adjust_qs, p.adjust_by, p.n_qs_bins, p.qs_bins, &k->pre) != 0)
        return fail(VGL_ERANGE, "the fixed quality score falls outside every --qs-bins range");
    if (p.error_qs != 2) k->gl_mode = p.gl_model == 1 ? GL_M1_FIXED : GL_M2_FIXED;
    else k->gl_mode = p.gl_model == 1 ? GL_M1_PERREAD : (p.precise_gl ? GL_M2_PRECISE : GL_M2_LUT);
    if (p.error_qs != 0) {
        const double m = p.error_rate, one_over = 1.0 / m;
        k->beta_a = (((1.0 - m) / p.beta_variance) - one_over) * pow(m, 2);
        k->beta_b = k->beta_a * (one_over - 1);
        if (!(k->beta_a > 0.0) || !(k->beta_b > 0.0)) return fail(VGL_EINVAL, "beta shape parameters must be positive (rng.h:373-388)");
    }
    const uint32_t t = p.tag_mask;
    k->sample_strand = (t & (VGL_TAG_I16 | VGL_TAG_FMT_ADF | VGL_TAG_FMT_ADR | VGL_TAG_INFO_ADF | VGL_TAG_INFO_ADR)) != 0;
    k->need_cellq = p.error_qs == 2 && (t & (VGL_TAG_QS | VGL_TAG_I16));
    k->need_tail = (t & VGL_TAG_I16) != 0;
    for (int i = 0; i < p.n_qs_bins; ++i) // first matching range wins (vcfgl.cpp:57-64)
        for (int q = p.qs_bins[i][0]; q <= p.qs_bins[i][1]; ++q)
            if (q > k->bin_max) { k->bin_lut[q] = p.qs_bins[i][2]; k->bin_max = q; }
    if (p.gl_model == 1) {
        ErrmodTables em;
        em.build(1.0 - p.gl1_theta); // io.cpp:1276
        tab->m1_het = em.het_term();
        if (k->gl_mode == GL_M1_FIXED) {
            tab->m1_bsum = em.fixed_q_bsum((p.adjust_qs & 1) ? k->pre.adj_qs : k->pre.qs); // gl_methods.cpp:318
            k->fast_div = ErrmodTables::scores_safe_for_fast_div(tab->m1_bsum, tab->m1_het) ? 1 : 0;
        } else {
            tab->fk = std::move(em.fk);
            tab->beta = std::move(em.beta);
        }
    }
    // ---- the depth law: 256-column alias tables when no cell can get more than 255 reads
    tab->alias.assign(256, 0ull);
    k->alias_ok = p.depth_mode == VGL_DEPTH_FIXED && p.depth_mean < 256.0;
    if (p.depth_mode == VGL_DEPTH_POISSON) {
        tab->pois_cdf = poisson_cdf_u64(p.depth_mean, 1024);
        std::vector<unsigned long long> al = poisson_alias_u64(tab->pois_cdf); // empty: depth can exceed 255
        if (!al.empty()) { tab->alias = std::move(al); k->alias_ok = true; }
    }
    if (p.depth_mode == VGL_DEPTH_POISSON_PER_SAMPLE) { // --depths-file: one alias table per distinct mean, a row index per sample
        std::vector<double> means;
        std::vector<unsigned long long> all;
        k->alias_ok = true;
        for (int sidx = 0; sidx < p.n_samples && k->alias_ok; ++sidx) {
            const double m = depth_means[sidx];
            size_t row = 0;
            while (row < means.size() && means[row] != m) ++row;
            if (row == means.size()) {
                const std::vector<unsigned long long> al = poisson_alias_u64(poisson_cdf_u64(m, 1024));
                if (al.empty() || means.size() >= 65535) { k->alias_ok = false; break; }
                means.push_back(m);
                all.insert(all.end(), al.begin(), al.end());
            }
            tab->alias_row.push_back((uint16_t)row);
        }
        if (k->alias_ok) tab->alias = std::move(all);
        else tab->alias_row.clear();
    }
    // ---- the kernel set
    const bool plane_ok = (size_t)p.max_batch_sites * (((size_t)p.n_samples * 15 + 3) & ~(size_t)3) < (1ull << 31); // G-shaped plane
    // the fused single-kernel path: native RNG, GL model 1 with a run-constant qs, count-level sampler
    const bool fused = k->gl_mode == GL_M1_FIXED && p.sampler != VGL_SAMPLER_PER_READ && !(t & (VGL_TAG_QS | VGL_TAG_I16)) && plane_ok;
    if (p.sampler == VGL_SAMPLER_COUNTS && !fused) return fail(VGL_EINVAL, "count-level sampler unavailable for this configuration (plane too large)");
    const bool tile = allow_tile && plane_ok && k->alias_ok && p.n_samples <= TILE_M1F_MAX_SAMPLES;
    // k_tile_m1f takes the fused path's runs without strand tags, and its AUX variant those with QS / I16 / INFO ADF, ADR / GP /
    // FORMAT ADF, ADR
    const bool tile_m1f = tile && k->gl_mode == GL_M1_FIXED && p.sampler != VGL_SAMPLER_PER_READ && p.error_qs == 0 && k->fast_div &&
                          ((t & TILE_M1F_AUX_TAGS) || (fused && !k->sample_strand));
    // k_tile_m2: native RNG, GL model 2 with run constants or the qs class table (not --precise-gl 1 with --error-qs 2), tags
    // within GL / PL / AD / DP / INFO AD, DP
    const uint32_t m2_tags = VGL_TAG_GL | VGL_TAG_PL | VGL_TAG_FMT_AD | VGL_TAG_FMT_DP | VGL_TAG_INFO_AD | VGL_TAG_INFO_DP;
    const bool tile_m2 = tile && p.gl_model == 2 && p.sampler == VGL_SAMPLER_AUTO && !(p.error_qs == 2 && p.precise_gl) && !(t & ~m2_tags);
    if (p.depth_mode == VGL_DEPTH_INF) k->set = KS_TRUTH;
    else if (tile_m1f) k->set = KS_TILE_M1F;
    else if (tile_m2 && plan_tile_m2(p, k, tab)) k->set = KS_TILE_M2;
    else if (fused) k->set = KS_FUSED_M1F;
    k->aux = k->set == KS_TILE_M1F && (t & TILE_M1F_AUX_TAGS);
    return VGL_OK;
}

} // namespace vgl
