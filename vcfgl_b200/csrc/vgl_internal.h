// Internal declarations shared by the kernels and the C-ABI layer.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/vgl.h"
#include "tables.h"

namespace vgl {

// per-cell record written by the simulate kernel, read by the site and emit kernels (16 B)
struct __align__(16) CellRec {
    uint16_t ad[4];  // reads per observed base A,C,G,T
    uint16_t fwd[4]; // of those, forward-strand reads (0 when the strand is not sampled)
};

// per-cell quality sums, only when per-read qs AND (QS or I16) are on (32 B)
struct __align__(16) CellQ {
    int32_t qsum[4];
    int32_t qsumsq[4];
};

// per-cell tail-distance sums, only with I16 (16 B)
struct __align__(16) CellTail {
    uint32_t sum, sumsq;
    int32_t last_base; // base of the cell's last read, -1 if no reads
    uint32_t _pad;
};

// GL / PL of the two non-trivial classes of a pure cell (tile_m1f.cu): base pairs that hold the cell's base once / not at all
struct __align__(16) M1Pure {
    float gl1, gl0;
    int32_t pl1, pl0;
};

struct DevParams {
    // geometry
    int32_t S, n_sites;
    int64_t first_site;
    int64_t n_cells;
    uint32_t k0, k1; // Philox key
    uint32_t rk[20]; // its ten round keys {k0 + r*W0, k1 + r*W1}
    // simulation parameters
    int32_t depth_mode;
    double depth_mean;
    const double* depth_means;
    double error_rate;
    int32_t error_qs;
    double beta_a, beta_b;
    int32_t gl_mode;
    int32_t adjust_qs;
    double adjust_by;
    int32_t use_bins, bin_max;
    uint8_t bin_lut[256];
    int32_t do_unobserved, rm_invar_sim, rm_empty, do_gvcf;
    uint32_t tag_mask;
    int32_t i16_mapq;
    int32_t pre_qs, pre_adj_qs; // fixed-qs runs (vcfgl.cpp:1697-1703)
    double homT, het, homF;     // GL_M2_FIXED constants
    int32_t sample_strand;      // shared.h:160 PROGRAM_WILL_SAMPLE_STRAND
    int32_t need_cellq, need_tail;
    int32_t fast_div;           // table-derived proof that the 3-instruction /10 is exact for every score
    int32_t zero_holes;         // tile kernels: zero the unused tail of every tile's plane span (planes that cross PCIe whole)
    // tables
    const double* lut_log10;  // [3*257]
    const double* m1_bsum;    // [256*256] fixed-qs running sums
    const double* m1_het;     // [256*256] -4.343*lhet
    const double* em_fk;      // [256]
    const double* em_beta;    // [64*256*256]
    // buffers
    const uint8_t* gt;
    int32_t* dp;
    CellRec* cell;
    CellQ* cellq;
    CellTail* celltail;
    vgl_site_out* sites;
    int64_t* totals; // [2] used G / R elements
    int64_t* totals_host; // the same two words in pinned host memory (device-accessible)
    uint64_t* pairmap; // [n_sites] base-pair -> genotype-slot map (GL model 1), written by k_site
    float* gl;
    int32_t* pl;
    float* gp;
    int32_t *ad, *adf, *adr;
    int32_t* status;
    // fused tile kernel (native, GL model 1 fixed qs, count-level sampler)
    const unsigned long long* pois_cdf; // [pois_n] Poisson CDF, 2^64 fixed point
    int32_t pois_n;
    int32_t sites_per_tile, n_tiles;
    unsigned long long* tile_state;     // [n_tiles] decoupled look-back words
    uint32_t* ticket;                   // dynamic tile counter
    // tile kernel (tile_m1f.cu)
    const unsigned long long* pois_alias; // [256] Walker alias table of the depth distribution: t56 << 8 | alias
    const uint16_t* alias_row;            // --depths-file: [S] row of each sample's own table in pois_alias ([rows][256]); null: one table
    const uint32_t* err_cdf;              // [256][4] P(E <= j | n reads) * 2^32, j = 0..3
    uint32_t* cnt_scratch;                // per-CTA rows of packed counts when a site does not fit shared memory
    const void* m1_pure;                  // [256] M1Pure: GL / PL of a cell whose reads all show one base, by depth; null: not usable
    // model-2 tile kernel (tile_m2.cu), --error-qs 2: alias table + info words of the per-read (quality score, error) classes
    const uint32_t* qcls;                 // [512], tables.h qs_class_table()
    const double* m2_tab;                 // [m2_nq][M2_TAB_DOUBLES] constants per quality score in use, tables.h m2_const_table(); null: none
    int32_t m2_nq;
    const uint32_t* m2_cmap;              // [16][8], tables.h m2_class_map()
    const uint32_t* qm_cdf;               // [256][4] P(M <= j | n) * 2^32: reads of a cell whose quality class is not the dominant one
    double q_minor;                       // P(a read is not of the dominant class)
    int32_t q_dom, q_dom_idx;             // the dominant class (index into the info words) and the dense index of its score
    const float* m2_pure;                 // [m2_nq][65][2] tables.h m2_pure_table(); null: no closed form for pure cells
    float* m2_park;                       // per-CTA rows of parked results of mixed cells (16 floats each)
    // replay
    int32_t replay;
    const int32_t* rp_depths;
    const int64_t* rp_off;
    const uint8_t *rp_bases, *rp_strands, *rp_qs, *rp_adjqs, *rp_tails;
    const double* rp_eprob;
    const int64_t* rp_deep_cells; // sorted cell ids with depth > 255 (GL model 1)
    int64_t rp_n_deep;
    const uint16_t* rp_deep_codes;
};

// VGL_HOST_BCF (bcf.cu): device serialisation of the kept sites as BCF records
struct BcfSiteMinMax {
    int32_t mn[5], mx[5]; // dp, pl, ad, adf, adr
};
struct BcfArgs {
    int32_t S, n_sites;
    uint32_t tag_mask;
    int32_t do_unobserved, do_gvcf;
    vgl_bcf_dict dict;
    const vgl_site_out* sites;
    const vgl_bcf_site_in* site_in;
    const uint8_t* blob;
    const int32_t* dp;
    const float *gl, *gp;
    const int32_t *pl, *ad, *adf, *adr;
    BcfSiteMinMax* minmax; // [n_sites]
    uint32_t* rec_len;     // [n_sites]
    long long* rec_off;    // [n_sites + 1]
    uint8_t* out;
    long long out_cap;
    int64_t* totals;       // [3] receives the total
    int32_t* status;
    struct BcfRecPlanes* planes; // [n_sites] or null: FORMAT plane layout of every record (for the BGZF compressor)
    // -doGVCF 1: the records are those of the block merger (gvcf.cu), in its order; null: one record per kept site
    const vgl_gvcf_rec* recs;    // [counts[0]]
    const int32_t* rec_counts;   // [0] records
    const int32_t *blk_dp, *blk_pl; // planes of the blocks' per-sample minima
};
void launch_bcf(const BcfArgs& a, cudaStream_t st);

// VGL_HOST_BGZF (bgzf.cu): the record stream compressed into BGZF blocks on the device
struct BcfRecPlanes { // where the FORMAT planes of a serialised record lie (written by k_bcf_emit)
    uint32_t off[7];  // byte offset of the plane's first value within the record
    uint16_t cell[7]; // bytes per sample
    uint16_t n;       // planes
};
enum { BGZF_STRIDE = 36992, BGZF_RNG_LIST = 63, BGZF_RNG_WORDS = 4 * (1 + BGZF_RNG_LIST) }; // bytes of a block's slot in the staging buffer (>= 18 + 32768 * 9 / 8 + 2 + 8)
struct BgzfArgs {
    int32_t S, n_sites;
    const uint8_t* in;          // the uncompressed record stream
    long long in_cap;
    const long long* rec_off;   // [n_sites + 1]
    const BcfRecPlanes* planes; // [n_sites]
    const uint32_t* crc_pow;    // [2048] bgzf_crc_pow_table(): chunk shifts, slicing tables
    uint8_t* stage;             // [max blocks][BGZF_STRIDE]
    uint32_t* blk_size;         // [max blocks]
    long long* blk_off;         // [max blocks]
    int32_t* blk_first;         // [max blocks] first record that reaches into the block
    uint32_t* rng_g;            // [max blocks][BGZF_RNG_WORDS] k_bgzf_ranges -> k_bgzf_deflate: {ranges, segments, state, -}, the ranges
    uint8_t* out;               // the compressed stream, blocks back to back
    int64_t* totals;            // [3] bytes of the record stream (in); [4] compressed bytes, [5] blocks (out)
    const BgzfCode* code;       // the context's prefix code (tables.h): deflate's fixed code until the statistics pass has run
    uint32_t* hist;             // non-null: statistics pass -- [BGZF_HIST] symbol counts of the parse, no output
};
size_t bgzf_dyn_smem();
int64_t bgzf_blocks_for(int64_t bytes);
void bgzf_crc_pow_table(uint32_t* t);
void launch_bgzf(const BgzfArgs& a, int64_t max_blocks, cudaStream_t st, int n_sms);

void launch_sim(const DevParams& p, cudaStream_t st);
void launch_site(const DevParams& p, cudaStream_t st);
void launch_scan(const DevParams& p, cudaStream_t st);
void launch_emit(const DevParams& p, cudaStream_t st);
int run_selftest(unsigned long long* n_bad, unsigned int* first_bad);
void launch_fused_m1f(const DevParams& p, cudaStream_t st, int n_sms);
void launch_tile_m1f(const DevParams& p, cudaStream_t st, int n_sms, bool aux);
int build_m1f_pure_table(const double* d_bsum, const double* d_het, void* out, cudaStream_t st);
void launch_tile_m1f_draws(const DevParams& p, cudaStream_t st, int pass, int32_t* depths, const int64_t* off, uint8_t* bases, uint8_t* strands,
                           uint8_t* tails);
void launch_tile_m2(const DevParams& p, cudaStream_t st, int n_sms, int mode);
size_t tile_m2_row_words(int S, int n_sms);
size_t tile_m2_park_floats(int S, int n_sms);
void launch_tile_m2_draws(const DevParams& p, cudaStream_t st, int mode, int pass, int32_t* depths, const int64_t* off, uint8_t* bases,
                          uint8_t* qs, double* eprob);
void launch_narrow(const int32_t* src, void* dst, int bits, bool is_pl, const int64_t* n_dev, int64_t n_fixed, int64_t cap, int32_t* status,
                   cudaStream_t st, int n_sms);
int tile_m1f_sites_per_tile(int S);
size_t tile_m1f_scratch_words(int S, int n_sms);
void launch_draws(const DevParams& p, cudaStream_t st, const int64_t* off, uint8_t* bases, uint8_t* strands, uint8_t* qs,
                  uint8_t* adjqs, uint8_t* tails, double* eprob);

// --depth inf (truth.cu)
void launch_truth_site(const DevParams& p, cudaStream_t st, int n_sms);
void launch_truth_emit(const DevParams& p, cudaStream_t st, int n_sms);

// discordance summary (discord.cu)
void launch_discordance(const vgl_site_out* sites, const uint8_t* gt, const int32_t* dp, const float* gl, int32_t S, int32_t n_sites,
                        unsigned long long* counts, cudaStream_t st, int n_sms);

// gVCF block merger (gvcf.cu)
struct GvcfDps {
    int32_t n;
    int32_t v[VGL_MAX_GVCF_DPS];
};
struct GvcfArgs {
    int32_t S, n_sites;
    GvcfDps dps;
    const vgl_site_out* sites;
    const int32_t *dp, *pl;
    const vgl_gvcf_site_in* sin;
    int2* key;
    vgl_gvcf_rec* recs;
    int32_t *prev_kept, *kept_idx, *counts, *blk_rec;
    unsigned long long *local, *block_sum;
    int32_t *out_dp, *out_pl;
};
void launch_gvcf(const GvcfArgs& a, cudaStream_t st, int n_sms);
void launch_gvcf_sin_from_bcf(const vgl_bcf_site_in* in, vgl_gvcf_site_in* out, int32_t n, cudaStream_t st);

// input path (vcfin.cu)
void launch_place_rows(const uint8_t* rows, const int32_t* d_row_map, int32_t first_record, int32_t n_sites, int32_t S, uint8_t fill, uint8_t* gt,
                       cudaStream_t st, int n_sms);
int parser_create(int device, int S, int rm_invar, int n_sms, int64_t max_text, int32_t max_records, vgl_parser** out, std::string& err);
void parser_destroy(vgl_parser* ps);

} // namespace vgl

// VCF text parser object of the input path (include/vgl.h); owned by the caller, tied to a context's device and geometry
struct vgl_parser {
    int device = 0, S = 0, rm_invar = 0, n_sms = 148;
    int32_t max_records = 0, n_records = 0;
    size_t text_cap = 0, d_text_bytes = 0;
    uint32_t max_tiles = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[3] = {};
    cudaEvent_t ev_done = nullptr; // rows of the last parse are complete
    cudaEvent_t ev_placed = nullptr; // the last vgl_place_rows() that read them has run
    bool placed = false;
    uint8_t *h_text = nullptr, *d_text = nullptr, *d_rows = nullptr;
    uint32_t *d_line_end = nullptr, *d_counters = nullptr, *h_counters = nullptr;
    uint32_t *d_tile_count = nullptr, *d_block_base = nullptr, *d_work = nullptr;
    uint16_t* d_tile_masks = nullptr; // one line-feed mask per 16 bytes of text
    vgl_in_site *d_sites = nullptr, *h_sites = nullptr;
    int32_t* d_row_map = nullptr;
    void* d_meta = nullptr; // RecMeta [max_records] (vcfin.cu)
    int64_t launches = 0;
    std::string err;
};
