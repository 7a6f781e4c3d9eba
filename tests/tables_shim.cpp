// tests/tables_shim.cpp -- test-only C shim over the PRODUCT's host tables (vcfgl_b200/csrc/tables.cpp),
// so that tests can compare them bit-for-bit with the reference's (oracle/_ref) without widening the C ABI.
#include "../vcfgl_b200/csrc/tables.h"
#include <cstring>
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
}
