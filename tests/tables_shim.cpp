// tests/tables_shim.cpp -- test-only C shim over the PRODUCT's host tables (vcfgl_b200/csrc/tables.cpp),
// so that tests can compare them bit-for-bit with the reference's (oracle/_ref) without widening the C ABI.
#include "../vcfgl_b200/csrc/tables.h"
#include <cstring>
// philox.cuh on the host: the same Philox4x32-10 and counter layout the kernels use
#define __host__
#define __device__
#define __forceinline__ inline
#include "../vcfgl_b200/csrc/philox.cuh"
extern "C" {
const double* shim_lut() { return &vgl::kLutLog10Gl[0][0]; }
void* shim_errmod(double depcorr) { auto* t = new vgl::ErrmodTables(); t->build(depcorr); return t; }
const double* shim_fk(void* t) { return ((vgl::ErrmodTables*)t)->fk.data(); }
const double* shim_beta(void* t) { return ((vgl::ErrmodTables*)t)->beta.data(); }
const double* shim_lhet(void* t) { return ((vgl::ErrmodTables*)t)->lhet.data(); }
void shim_fixed_bsum(void* t, int q, double* out) { auto v = ((vgl::ErrmodTables*)t)->fixed_q_bsum(q); memcpy(out, v.data(), v.size() * 8); }
void shim_free(void* t) { delete (vgl::ErrmodTables*)t; }
int shim_precalc(double e, int eq, int gl, int precise, int adj, double adjby, int* qs, int* adjqs, double* g3)
{
    vgl::PreCalc pc;
    const uint8_t none[1][3] = {{0, 0, 0}};
    int rc = vgl::precalc(e, eq, gl, precise, adj, adjby, 0, none, &pc);
    *qs = pc.qs; *adjqs = pc.adj_qs; g3[0] = pc.homT; g3[1] = pc.het; g3[2] = pc.homF;
    return rc;
}
double shim_inc_beta(double a, double b, double x) { return vgl::inc_beta(a, b, x); }
// returns the number of table words (0: no table); prob512[2q + err]
int shim_qs_classes(double a, double b, double shift, int use_bins, const uint8_t* bin_lut, int bin_max, uint32_t* words, double* prob512)
{
    std::vector<double> pr;
    auto w = vgl::qs_class_table(a, b, shift, use_bins != 0, bin_lut, bin_max, &pr);
    if (w.empty()) return 0;
    memcpy(words, w.data(), w.size() * 4);
    memcpy(prob512, pr.data(), 257 * 8);
    return (int)w.size();
}
// 640 words: lit[256], len[256], dist[32], eob, hdr_bits, hdr[94]
void shim_bgzf_code(const uint32_t* hist, int fixed, uint32_t* out)
{
    vgl::BgzfCode c;
    vgl::bgzf_build_code(hist, fixed != 0, &c);
    memcpy(out, &c, sizeof(c));
}
int shim_bgzf_code_words() { return (int)(sizeof(vgl::BgzfCode) / 4); }
// 1 when exactly n_fmt FORMAT blocks of S samples tile the len bytes at p (the check vgl_submit runs on VGL_HOST_BCF input)
int shim_bcf_fmt_blocks_tile(const uint8_t* p, uint64_t len, uint32_t n_fmt, int64_t n_samples)
{
    return vgl::bcf_fmt_blocks_tile(p, len, n_fmt, n_samples) ? 1 : 0;
}
// the kernel set vgl_create picks for *p (p->depth_means: the --depths-file means); *status receives plan_run's status
const char* shim_kernel_set(const vgl_params* p, int allow_tile, int* status)
{
    vgl::RunPlan plan;
    vgl::PlanTables tab;
    const char* why = "";
    *status = vgl::plan_run(*p, p->depth_means, allow_tile != 0, &plan, &tab, &why);
    return vgl::kernel_set_name(plan.set);
}
// ---- the draw keying and the sampler tables (tests/test_sampler_laws.py, tests/test_gpu_sampler_draws.py)
void shim_philox(uint32_t k0, uint32_t k1, const uint32_t* ctr4, int64_t n, uint32_t* out4)
{
    for (int64_t i = 0; i < n; ++i) {
        const vgl::u32x4 c = {ctr4[4 * i], ctr4[4 * i + 1], ctr4[4 * i + 2], ctr4[4 * i + 3]};
        const vgl::u32x4 o = vgl::philox4x32_10(c, k0, k1);
        out4[4 * i] = o.x; out4[4 * i + 1] = o.y; out4[4 * i + 2] = o.z; out4[4 * i + 3] = o.w;
    }
}
static vgl::Key shim_key(uint64_t seed) { return vgl::Key{(uint32_t)(seed & 0xFFFFFFFFu), (uint32_t)(seed >> 32)}; }
// blocks 0 and 1 of the P_COUNTS counter of every (site, sample), site-major: out8[cell] = block 0 words, block 1 words
void shim_counts_b01(uint64_t seed, int64_t first_site, int64_t n_sites, int64_t S, uint32_t* out8)
{
    const vgl::Key key = shim_key(seed);
    for (int64_t sl = 0; sl < n_sites; ++sl)
        for (int64_t s = 0; s < S; ++s) {
            uint32_t* o = out8 + 8 * (sl * S + s);
            const vgl::u32x4 b0 = vgl::draw(key, first_site + sl, (uint32_t)s, 0, vgl::P_COUNTS, 0);
            const vgl::u32x4 b1 = vgl::draw(key, first_site + sl, (uint32_t)s, 0, vgl::P_COUNTS, 1);
            o[0] = b0.x; o[1] = b0.y; o[2] = b0.z; o[3] = b0.w; o[4] = b1.x; o[5] = b1.y; o[6] = b1.z; o[7] = b1.w;
        }
}
// one block per entry: draw(seed, site[i], sample[i], read[i], purpose, block[i])
void shim_draws(uint64_t seed, const int64_t* site, const uint32_t* sample, const uint32_t* read, uint32_t purpose, const uint32_t* block,
                int64_t n, uint32_t* out4)
{
    const vgl::Key key = shim_key(seed);
    for (int64_t i = 0; i < n; ++i) {
        const vgl::u32x4 o = vgl::draw(key, site[i], sample[i], read[i], purpose, block[i]);
        out4[4 * i] = o.x; out4[4 * i + 1] = o.y; out4[4 * i + 2] = o.z; out4[4 * i + 3] = o.w;
    }
}
// the sites of [first_site, first_site + n_sites) where some sample's word `word` of P_COUNTS block 0 is >= lo; returns their
// number (at most cap are stored)
int64_t shim_scan_counts_word(uint64_t seed, int64_t first_site, int64_t n_sites, int64_t S, int word, uint32_t lo, int64_t* out, int64_t cap)
{
    const vgl::Key key = shim_key(seed);
    int64_t k = 0;
    for (int64_t sl = 0; sl < n_sites && k < cap; ++sl)
        for (int64_t s = 0; s < S; ++s) {
            const vgl::u32x4 b0 = vgl::draw(key, first_site + sl, (uint32_t)s, 0, vgl::P_COUNTS, 0);
            const uint32_t w[4] = {b0.x, b0.y, b0.z, b0.w};
            if (w[word] >= lo) { out[k++] = first_site + sl; break; }
        }
    return k;
}
double shim_u01_32(uint32_t w) { return vgl::u01_32(w); }
double shim_u01_53(uint32_t hi, uint32_t lo) { return vgl::u01_53(hi, lo); }
// returns the number of entries written (at most cap)
int shim_poisson_cdf_u64(double lambda, int max_n, uint64_t* out, int cap)
{
    const auto t = vgl::poisson_cdf_u64(lambda, max_n);
    const int n = (int)t.size() < cap ? (int)t.size() : cap;
    memcpy(out, t.data(), (size_t)n * 8);
    return (int)t.size();
}
// 256 entries, or 0 when the law does not fit the table
int shim_poisson_alias_u64(const uint64_t* cdf, int n, uint64_t* out256)
{
    const auto t = vgl::poisson_alias_u64(std::vector<unsigned long long>(cdf, cdf + n));
    if (!t.empty()) memcpy(out256, t.data(), 256 * 8);
    return (int)t.size();
}
void shim_binomial_cdf4_u32(double e, uint32_t* out1024)
{
    const auto t = vgl::binomial_cdf4_u32(e);
    memcpy(out1024, t.data(), 1024 * 4);
}
// the sampler tables vgl_create uploads for *p: the alias rows (returned: their number; at most cap_rows stored), each sample's
// row under --depths-file (n_samples entries, else untouched), the qs class table (768 words, --error-qs 2 under k_tile_m2),
// its dominant class and the probability of the other classes
int shim_plan_tables(const vgl_params* p, uint64_t* alias, int cap_rows, uint16_t* alias_row, uint32_t* qcls, int* q_dom, double* q_minor)
{
    vgl::RunPlan plan;
    vgl::PlanTables tab;
    const char* why = "";
    if (vgl::plan_run(*p, p->depth_means, true, &plan, &tab, &why) != VGL_OK) return -1;
    const int rows = (int)(tab.alias.size() / 256);
    memcpy(alias, tab.alias.data(), (size_t)(rows < cap_rows ? rows : cap_rows) * 256 * 8);
    if (!tab.alias_row.empty()) memcpy(alias_row, tab.alias_row.data(), tab.alias_row.size() * 2);
    if (tab.qcls.size() == 768) memcpy(qcls, tab.qcls.data(), 768 * 4);
    *q_dom = plan.q_dom;
    *q_minor = plan.q_minor;
    return rows;
}
}
