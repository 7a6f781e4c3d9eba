// Host-side constant tables of the simulation core (built once in vgl_create()).
#pragma once
#include <stdint.h>
#include <vector>

#include "../../include/vgl.h"

namespace vgl {

enum GlMode : int {
    GL_M1_FIXED = 0,   // gl_methods.cpp:304-369  model 1, one qs for every read -> depends on base counts only
    GL_M1_PERREAD = 1, // gl_methods.cpp:233-302  model 1, per-read qs
    GL_M2_FIXED = 2,   // gl_methods.cpp:4-69     model 2, run-constant homT/het/homF
    GL_M2_LUT = 3,     // gl_methods.cpp:71-150   model 2, qs -> LUT
    GL_M2_PRECISE = 4  // gl_methods.cpp:152-231  model 2, log10 of the per-read error probability
};

// samtools/bcftools "revised MAQ" error-model coefficients
// (reference: htslib/errmod.c:51-125, errmod_init(1 - theta) at io.cpp:1276)
struct ErrmodTables {
    std::vector<double> fk;   // [256]          dependency decay  fk[n] = (1-depcorr)^n (1-eta) + eta
    std::vector<double> beta; // [64][256][256] phred-scaled binomial tail ratios, index q<<16 | n<<8 | k
    std::vector<double> lhet; // [256][256]     log C(n,k) - n ln 2, index n<<8 | k
    void build(double depcorr, double eta = 0.03);
    // for a FIXED quality score q: the running sum errmod_cal() would reach after walking
    // c reads of one base at depth n:  bsum[n<<8 | c] = sum_{i<c} fk[i] * beta[q][n][i]
    // (errmod.c:174-177 with w == c because the strand bit is never set, gl_methods.cpp:329)
    std::vector<double> fixed_q_bsum(int q) const;
    // -4.343 * lhet[n<<8 | k]  (errmod.c:200)
    std::vector<double> het_term() const;
    // true when every errmod score (a float sum of non-negative table terms) is +0 or >= 2^-100 and
    // finite: each positive term of both tables is itself >= 2^-100, and all are finite and >= 0
    static bool scores_safe_for_fast_div(const std::vector<double>& bsum, const std::vector<double>& het);
};

// Poisson(lambda) CDF as 2^64 fixed-point thresholds: n = smallest k with u < cdf[k] for a 64-bit
// uniform u.  At most max_n entries; the last entry is 2^64-1.  (native count-level sampler)
std::vector<unsigned long long> poisson_cdf_u64(double lambda, int max_n);

// Walker alias table over 256 columns for the same distribution (tile kernel): with a 64-bit uniform u,
// column = u >> 56; the cell keeps `column` when (u << 8) < (entry & ~0xFF), else takes entry & 0xFF.
// Built in exact integer arithmetic from the CDF above, so P(n) is reproduced to 2^-64.
// Returns an empty vector when the support does not fit 256 outcomes.
std::vector<unsigned long long> poisson_alias_u64(const std::vector<unsigned long long>& cdf);

// number of mis-called reads E ~ Binomial(n, e): thresholds floor(P(E <= j | n) * 2^32), j = 0..3, n = 0..255
// (saturated at 2^32-1); E = #{j : u >= t[n][j]} for a 32-bit uniform u, 4 = "beyond the table".
std::vector<uint32_t> binomial_cdf4_u32(double e);

// regularized incomplete beta function I_x(a, b) (continued fraction, Lentz), x in [0, 1]
double inc_beta(double a, double b, double x);

// Law of the per-read quality score the GL uses under --error-qs 2 (vcfgl.cpp:494-523): the read's error probability p
// is Beta(a, b), phred = -10 log10 p, q = (int)(phred + shift) (shift = --adjust-by when the GL uses the adjusted score,
// else 0), then --qs-bins or the cap at 63; P(q) = I(p_hi) - I(p_lo).  (The read is mis-called with the run-constant
// --error-rate, independently of its quality score: vcfgl.cpp:485 draws before and apart from :495.)
// Returned: 768 words = a Walker alias table over 256 columns (threshold24 << 8 | alias; probabilities quantised to
// 2^-32) followed by the class info words: q | out-of-range << 9 | dense index of q << 16 (ascending q; `q_values`
// receives the scores).  Scores beyond the last --qs-bins range (the reference exits when it draws one, vcfgl.cpp:63)
// form a class of their own (score 0, bit 9) so that the kernel can raise VGL_ERANGE.  `prob` receives the quantised
// probabilities ([q], out of range at [256]; for tests).  Empty when the classes do not fit 256 columns.
// Words 512..767: the Walker alias table of the conditional law of the classes other than the heaviest ("dominant") one;
// `dominant` receives that class's index (into the info words), `p_minor` the probability that a read is not of it.
std::vector<uint32_t> qs_class_table(double a, double b, double shift, bool use_bins, const uint8_t* bin_lut, int bin_max,
                                     std::vector<double>* prob = nullptr, std::vector<int>* q_values = nullptr, int* dominant = nullptr,
                                     double* p_minor = nullptr);

// Constant tables of the model-2 tile kernel for each (homT, het, homF) triple: per triple M2_TAB_DOUBLES doubles =
// [4 read bases][17] the constant each of the 15 base pairs (k*(k+1)/2 + j, 4 = unobserved allele) receives from a
// read of that base (gl_methods.cpp:27-48), then [2][8] the constants of the six classes {xx, xy, yy, x., y., ..} of
// a cell whose reads show two bases x, y for a read of y ([0]) or x ([1]).
enum { M2_TAB_DOUBLES = 84 };
std::vector<double> m2_const_table(const std::vector<double>& homT_het_homF);
// GL of a cell whose n <= 64 reads all show the same base x and share one quality score ("pure" cell): the matching
// homozygote is the maximum after every read, so the vector is a function of n alone: out[(q * 65 + n) * 2 + {0, 1}] = the
// value of the base pairs that contain x once / not at all (the pair xx holds +0), computed with the reference's
// float += double, float -= max sequence (gl_methods.cpp:27-58).  False when a triple does not have homT >= het, homF
// (error rates >= 0.5): the shortcut is then not valid.
bool m2_pure_table(const std::vector<double>& homT_het_homF, std::vector<float>* out);
// [16 = x*4+y][8 words]: words 0..2 = six 16-bit masks of the base pairs in each class, words 4,5 = the class of
// every base pair (3 bits each, pair k at bits 3k)
std::vector<uint32_t> m2_class_map();

// qScore_to_log10_gl[3][257] (shared.cpp:110-114)
extern const double kLutLog10Gl[3][257];

// derived per-run constants (reference: preCalcStruct io.h:22-32, filled at vcfgl.cpp:1661-1743)
struct PreCalc {
    int qs = -1, adj_qs = -1;
    double homT = -1.0, het = -1.0, homF = -1.0;
};

// returns 0, or -1 when a qs falls outside the --qs-bins ranges (vcfgl.cpp:63)
int precalc(double error_rate, int error_qs, int gl_model, int precise_gl, int adjust_qs, double adjust_by,
            int n_bins, const uint8_t bins[][3], PreCalc* out);

// ---- the prefix codes of the device's BGZF compressor (csrc/bgzf.cu), RFC 1951.  One code per context: either deflate's fixed
// code (3.2.6) or a "dynamic" code (3.2.7) built once from the symbol counts of the context's first record stream; every block
// then starts with the same precomputed header bits.  All codes are stored bit-reversed (deflate packs Huffman codes most
// significant bit first into a stream that is otherwise filled from the least significant bit).
struct BgzfCode {
    uint32_t lit[256];  // literal byte: code | bits << 16
    uint32_t len[256];  // match length - 3: (code | extra bits << code bits) | total bits << 24   (<= 15 + 5 bits)
    uint32_t dist[32];  // distance code 0..29: code | bits << 16   (the extra bits follow, computed by the kernel)
    uint32_t eob;       // end of block: code | bits << 16
    uint32_t hdr_bits;  // bits of the block header (BFINAL, BTYPE, and for a dynamic code the code lengths)
    uint32_t hdr[94];   // the header bits, least significant bit first
};
enum { BGZF_HIST = 320 }; // symbol counts: [0..285] literal / length symbols, [288..317] distance symbols
// fixed = deflate's fixed code; else from the counts (every symbol gets a code, whatever its count)
void bgzf_build_code(const uint32_t* hist, bool fixed, BgzfCode* out);

// ---- input records of VGL_HOST_BCF (vgl_bcf_site_in): true when exactly n_fmt FORMAT blocks (a typed-integer key, a type
// descriptor with the vector size, n_samples vectors) tile the `len` bytes at p.  Every byte read lies inside them, and the
// device's parser (bcf.cu in_fmt_block) then walks n_fmt blocks without leaving the range.
bool bcf_fmt_blocks_tile(const uint8_t* p, uint64_t len, uint32_t n_fmt, int64_t n_samples);

// ---- the kernel set of a context (vgl_create), chosen from its parameters alone
enum { TILE_M1F_MAX_SAMPLES = 60000 }; // largest S the tile kernels take (the slot arithmetic needs (S4 + block) * S4 < 2^32)
// tags the AUX variant adds to the tile kernel's GL / PL / AD / DP / INFO AD, DP
enum : uint32_t { TILE_M1F_AUX_TAGS = VGL_TAG_QS | VGL_TAG_I16 | VGL_TAG_INFO_ADF | VGL_TAG_INFO_ADR | VGL_TAG_GP | VGL_TAG_FMT_ADF | VGL_TAG_FMT_ADR };
enum KernelSet : int {
    KS_PER_READ,  // k_sim, k_site, k_scan, k_emit: every configuration (and every replayed batch)
    KS_FUSED_M1F, // k_fused_m1f: GL model 1 with a run-constant qs, count-level sampler
    KS_TILE_M1F,  // k_tile_m1f (tile_m1f.cu): the fused path's headline special case, depths from the alias table, --error-qs 0
    KS_TILE_M2,   // k_tile_m2 (tile_m2.cu): GL model 2 with run constants (--error-qs 0/1) or the qs class table (--error-qs 2)
    KS_TRUTH      // --depth inf (truth.cu): k_truth_site, k_scan, k_truth_emit
};
const char* kernel_set_name(KernelSet k); // as vgl_native_kernels() reports it

struct RunPlan { // the run constants of a context and its kernel set
    KernelSet set = KS_PER_READ;
    bool aux = false; // KS_TILE_M1F: the AUX variant (a tag of TILE_M1F_AUX_TAGS is on)
    int gl_mode = GL_M1_FIXED;
    PreCalc pre;
    double beta_a = 0, beta_b = 0;
    int sample_strand = 0, need_cellq = 0, need_tail = 0;
    uint8_t bin_lut[256] = {};
    int bin_max = -1;
    int fast_div = 0;             // GL_M1_FIXED: the 3-instruction /10 is exact for every score
    bool alias_ok = false;        // the depth law fits a 256-column alias table: no cell holds more than 255 reads
    int q_dom = 0, q_dom_idx = 0; // KS_TILE_M2 with --error-qs 2: the dominant quality class (qs_class_table)
    double q_minor = 0.0;
    int m2_nq = 0;                // KS_TILE_M2: quality scores in m2_tab
};
struct PlanTables { // host tables the context uploads for its kernel set
    std::vector<double> m1_het, m1_bsum, fk, beta; // GL model 1 (ErrmodTables)
    std::vector<unsigned long long> pois_cdf;      // VGL_DEPTH_POISSON
    std::vector<unsigned long long> alias;         // tile kernels: [rows][256] Walker alias tables of the depth law
    std::vector<uint16_t> alias_row;               // --depths-file: each sample's row in alias
    std::vector<uint32_t> qcls;                    // KS_TILE_M2, --error-qs 2: qs_class_table()
    std::vector<double> m2_tab;                    // KS_TILE_M2: m2_const_table()
    std::vector<float> m2_pure;                    // KS_TILE_M2: m2_pure_table(), when valid
};
// Fills the default-constructed *plan and *tab.  VGL_OK, or VGL_ERANGE / VGL_EINVAL with the reason in *why.  depth_means:
// [n_samples] under VGL_DEPTH_POISSON_PER_SAMPLE.  allow_tile = false keeps the tile kernels out.
int plan_run(const vgl_params& p, const double* depth_means, bool allow_tile, RunPlan* plan, PlanTables* tab, const char** why);

} // namespace vgl
