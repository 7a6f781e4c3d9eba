/*
 * vgl.h -- C ABI of the B200-native vcfgl simulation core (libvgl.so).
 *
 * Drop-in boundary for the reference's per-site hot path.  The reference has
 * no plugin ABI; its operator interface for this path is internal:
 *
 *   static int simulate_record_values(simRecord*)          vcfgl.cpp:327
 *   void (*calculate_gls)(simRecord*)                      vcfgl.cpp:222, gl_methods.h:6-10
 *   inputs through globals: args (io.h:40-148), true_gts_acgt_int and
 *   n_sim_reads_arr (vcfgl.cpp:66-67), libc RNG state (vcfgl.cpp:214-219)
 *   outputs: the simRecord tag arrays handed to htslib by
 *   simRecord::add_tags()                                  bcf_utils.cpp:426-507
 *
 * The replacement works on BATCHES of sites: the host driver loop
 * (vcfgl.cpp:1469-1565) appends each site's packed true genotypes to a pinned
 * input buffer instead of calling simulate_record_values(), submits the batch,
 * and one batch later walks vgl_batch_out in site order feeding the returned
 * arrays to bcf_update_format_* / bcf_update_info_* with zero repacking (see INTEGRATION.md).
 *
 * Conventions: every function returns VGL_OK (0) or a negative vgl_status and
 * never exits the process (the reference's ERROR()/ASSERT() exit(1),
 * shared.h:292-327; the host maps codes back to that).  All memory handed out
 * is owned by the context and stays valid until the slot is submitted again
 * or the context is destroyed.  One host thread per context; one context per
 * GPU.  Site ids are global running indices, so results do not depend on batch
 * size or on how sites are sharded over GPUs.
 *
 * There is no CPU fallback: vgl_create() fails with VGL_ENODEV without a CUDA
 * device.
 */
#ifndef VGL_H
#define VGL_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VGL_ABI_VERSION 9 /* 2: VGL_HOST_NARROW; 3: VGL_HOST_BCF; 4: input path (vgl_parser_*, vgl_parse_vcf, vgl_place_rows); 5: vgl_gvcf_merge;
                          * 6: VGL_DEPTH_INF; 7: vgl_discordance; 8: vgl_parse_bcf 
                          * 9: VGL_HOST_BGZF (device-side BGZF compression of the record stream); vgl_bcf_site_in::fmt_off/fmt_len/n_fmt */

#define VGL_MAX_ALLELES 5    /* shared.h:220 MAX_NALLELES */
#define VGL_MAX_GENOTYPES 15 /* shared.h:228 MAX_NGTS */

/* packed true genotype of one (site, sample) cell: low nibble = first
 * haplotype, high nibble = second; value = ACGT int 0..3 (what
 * check_rec_alleles() stores in true_gts_acgt_int, vcfgl.cpp:133-146),
 * 0xF = missing (-1 there). */
#define VGL_GT_MISSING 0xF
#define VGL_GT_PACK(h0, h1) ((uint8_t)(((h0) & 0xF) | (((h1) & 0xF) << 4)))

/* missing sentinels, identical to htslib's (htslib/vcf.c:56, htslib/htslib/vcf.h:1325) */
#define VGL_F32_MISSING_BITS 0x7F800001u
#define VGL_I32_MISSING INT32_MIN

typedef enum vgl_status {
    VGL_OK = 0,
    VGL_EINVAL = -1,  /* bad argument / unsupported option combination (io.cpp:860-1000) */
    VGL_ENOMEM = -2,
    VGL_ECUDA = -3,   /* CUDA runtime error; vgl_last_error() has the text */
    VGL_ESTATE = -4,  /* slot busy / not submitted */
    VGL_ERANGE = -5,  /* a quality score fell outside every --qs-bins range (vcfgl.cpp:63) */
    VGL_ENODEV = -6,  /* no CUDA device: there is no CPU path */
    VGL_EOVERFLOW = -7, /* batch status with VGL_HOST_NARROW: a depth / allelic depth did not fit narrow_bits (values were saturated) */
    VGL_EMISSING = -8   /* batch status with VGL_DEPTH_INF: a true genotype is missing (the reference asserts, vcfgl.cpp:1196) */
} vgl_status;

/* vgl_params.tag_mask: which tags add_tags() would emit (io.h:90-102) */
enum {
    VGL_TAG_GL = 1 << 0, VGL_TAG_GP = 1 << 1, VGL_TAG_PL = 1 << 2, VGL_TAG_I16 = 1 << 3,
    VGL_TAG_QS = 1 << 4, VGL_TAG_FMT_DP = 1 << 5, VGL_TAG_INFO_DP = 1 << 6,
    VGL_TAG_FMT_AD = 1 << 7, VGL_TAG_INFO_AD = 1 << 8, VGL_TAG_FMT_ADF = 1 << 9,
    VGL_TAG_INFO_ADF = 1 << 10, VGL_TAG_FMT_ADR = 1 << 11, VGL_TAG_INFO_ADR = 1 << 12
};

enum { VGL_DEPTH_POISSON = 0,            /* --depth x        rng.h:284 */
       VGL_DEPTH_POISSON_PER_SAMPLE = 1, /* --depths-file    rng.h:318 */
       VGL_DEPTH_FIXED = 2,              /* every cell gets exactly (int)depth_mean reads */
       VGL_DEPTH_INF = 3 };              /* --depth inf: no reads; GL / GP / PL state the true genotype (vcfgl.cpp:1089-1262).
                                          * Only those three tags; vgl_site_out::info_dp is -1; not with replay, -doGVCF or
                                          * --rm-invar-sites 4 (io.cpp:783-800, 1012-1019) */

/* vgl_params.host_output: what vgl_wait() brings to pinned host memory */
enum { VGL_HOST_NONE = 0,    /* nothing but the totals and the status word: results stay in HBM */
       VGL_HOST_I32 = 1,     /* every plane exactly as add_tags() hands it to htslib (int32 / float32, bcf_utils.cpp:426-507) */
       VGL_HOST_NARROW = 2,  /* GL / GP as float32; PL, AD, ADF, ADR and DP narrowed on the device to the width BCF stores them
                              * in anyway (htslib/vcf.c:2249-2294 bcf_enc_vint): 1.8x fewer bytes over PCIe (see vgl_batch_out) */
       VGL_HOST_BCF = 3,     /* complete uncompressed BCF records, serialised on the device byte-for-byte as the reference's
                              * add_tags() + bcf_write() would (bcf_utils.cpp:426-507, htslib/vcf.c:1773-1917, 1951-2001): the
                              * host appends vgl_batch_out.bcf to the output stream (see vgl_bcf_site_in).  Not with -doGVCF:
                              * the block merger (bcf_utils.cpp:662-942) consumes arrays. */
       VGL_HOST_BGZF = 4 };  /* the same records, compressed on the device into BGZF blocks (the reference's default output,
                              * -O b; htslib/bgzf.c, vcfgl.cpp:1791-1803): vgl_batch_out.bgzf.  Input as for VGL_HOST_BCF. */

/* VGL_HOST_BCF: dictionary ids of the simulator's tags in the OUTPUT header, bcf_hdr_id2int(hdr, BCF_DT_ID, "DP") etc.
 * (FORMAT and INFO tags of the same name share one id).  Only ids of tags enabled in tag_mask are read. */
typedef struct vgl_bcf_dict {
    int32_t dp, gl, pl, gp, ad, adf, adr, qs, i16;
    int32_t end, min_dp; /* -doGVCF 1: INFO/END and INFO/MIN_DP of the block records (bcf_utils.cpp:905-912) */
} vgl_bcf_dict;

/* VGL_HOST_BCF: what the input record passes through to the output record unchanged (the reference edits a bcf_copy of
 * the input record: vcfgl.cpp:1540, bcf1_sync keeps the untouched pieces verbatim, htslib/vcf.c:1802-1838).
 * The byte ranges index the slot's pass-through blob (vgl_bcf_input_buffer); with in_rec unpacked,
 *   ID           = in_rec->shared.s[0 .. unpack_size[0])
 *   FILTER+INFO  = in_rec->shared.s[unpack_size[0] + unpack_size[1] .. shared.l)
 * A length of 0 selects the encoding of "." (ID: 0x07, FILTER: 0x00, no INFO). */
typedef struct vgl_bcf_site_in {
    int32_t rid, pos;             /* bcf1_t::rid, ::pos (0-based) */
    uint32_t qual_bits;           /* bcf1_t::qual as raw bits; VGL_F32_MISSING_BITS for "." */
    uint32_t n_info;              /* INFO fields the input record carries (they precede the simulator's) */
    uint32_t id_off, id_len;
    uint32_t flt_info_off, flt_info_len;
    /* FORMAT blocks the input record carries besides GT, concatenated in the record's order (typed key, size/type descriptor,
     * n_samples vectors each -- the bytes of in_rec->indiv.s with the GT block taken out); n_fmt of them.  The reference keeps
     * them: bcf_update_genotypes(NULL) removes only GT (vcfgl.cpp:793), a block whose key one of the simulated tags has is
     * replaced IN PLACE by that tag (an input FORMAT/DP), the other simulated tags follow the input's blocks
     * (htslib/vcf.c bcf_update_format).  n_fmt = 0: the input FORMAT is GT alone. */
    uint32_t fmt_off, fmt_len, n_fmt;
    uint32_t _pad;
} vgl_bcf_site_in;

/* how the native simulator draws a cell (replay ignores this) */
enum { VGL_SAMPLER_AUTO = 0,     /* COUNTS when the GL depends on base counts only, else PER_READ */
       VGL_SAMPLER_PER_READ = 1, /* one Philox block per read; ordered reads (all modes) */
       VGL_SAMPLER_COUNTS = 2 }; /* binomial/multinomial per cell: GL model 1 with --error-qs 0/1 only */

/* = the argStruct fields the hot path reads (io.h:40-148) */
typedef struct vgl_params {
    int32_t abi_version;  /* VGL_ABI_VERSION */
    int32_t n_samples;
    int64_t seed;         /* --seed */
    int32_t depth_mode;
    double depth_mean;          /* --depth (io.h:63) */
    const double* depth_means;  /* [n_samples] for PER_SAMPLE (io.h:125), else NULL */
    double error_rate;    /* --error-rate (io.h:66) */
    int32_t error_qs;     /* --error-qs 0|1|2 (io.h:67) */
    double beta_variance; /* --beta-variance (io.h:68); shape from rng.h:370-371 */
    int32_t gl_model;     /* --gl-model 1|2 (io.h:69) */
    double gl1_theta;     /* --gl1-theta (io.h:70) */
    int32_t precise_gl;   /* --precise-gl (io.h:72) */
    int32_t adjust_qs;    /* --adjust-qs bitmask (io.h:75, shared.h:103-117) */
    double adjust_by;     /* --adjust-by (io.h:76) */
    int32_t n_qs_bins;    /* --qs-bins (io.h:145-146): [start, end, value] */
    uint8_t qs_bins[255][3];
    int32_t do_unobserved;  /* -doUnobserved 0..5 (io.h:81) */
    int32_t rm_invar_sites; /* --rm-invar-sites bitmask; only bit 4 (simulated invariant) is device-side */
    int32_t rm_empty_sites; /* --rm-empty-sites */
    int32_t do_gvcf;        /* -doGVCF (only changes the no-reads site, vcfgl.cpp:242-246) */
    uint32_t tag_mask;
    int32_t i16_mapq;       /* --i16-mapq (io.h:73) */
    /* engine configuration (no reference counterpart) */
    int32_t device_id;       /* CUDA device ordinal */
    int32_t max_batch_sites; /* capacity of one slot */
    int32_t n_slots;         /* >= 1; 2 = double buffering */
    int32_t sampler;         /* VGL_SAMPLER_* */
    int32_t host_output;     /* VGL_HOST_* */
    /* VGL_HOST_BCF only */
    vgl_bcf_dict bcf_dict;
    int32_t bcf_blob_bytes_per_site; /* capacity of a slot's pass-through blob = max_batch_sites * this (0: 16) */
} vgl_params;

/* Replay input: the reference's own draws for a batch (from the instrumented
 * reference, oracle/ref_dump_hooks.h), all HOST pointers.  Cells are indexed
 * c = site_in_batch * n_samples + sample; reads of all cells are concatenated
 * in (cell, read) order and cover only cells whose genotype is not missing. */
typedef struct vgl_replay {
    const int32_t* depths;       /* [n_sites*S] depth drawn per cell, also for missing-GT cells (vcfgl.cpp:364-368) */
    const int64_t* read_offsets; /* [n_sites*S + 1] start of each cell's reads */
    int64_t n_reads;
    const uint8_t* bases;        /* [n_reads] observed base 0..3 (vcfgl.cpp:485-488) */
    const uint8_t* strands;      /* [n_reads] 0 fwd / 1 rev (vcfgl.cpp:581-586) or NULL */
    const uint8_t* qs;           /* [n_reads] per-read qs, --error-qs 2 (vcfgl.cpp:506-523) or NULL */
    const uint8_t* adj_qs;       /* [n_reads] adjusted qs (--adjust-qs != 0) or NULL */
    const double* error_probs;   /* [n_reads] beta-drawn error prob (--precise-gl 1, vcfgl.cpp:544) or NULL */
    const uint8_t* tail_dists;   /* [n_reads] capped tail distance, -addI16 (vcfgl.cpp:653-656) or NULL */
    /* GL model 1 cells deeper than 255 reads: the 255 read codes (qs<<5|base) kept by
     * errmod_cal's shuffle (htslib/errmod.c:156-159), 255 per such cell in cell order */
    int64_t n_deep_cells;
    const uint16_t* deep_codes;  /* [n_deep_cells*255] or NULL */
} vgl_replay;

/* per-site results: everything INFO-level plus where the site's FORMAT blocks start */
typedef struct vgl_site_out {
    int32_t skip_code;          /* 0 keep; -3 simulated invariant (vcfgl.cpp:677); -4 empty (vcfgl.cpp:401) */
    int32_t n_alleles;          /* sim->nAlleles */
    int32_t n_alleles_observed; /* sim->nAllelesObserved */
    int32_t n_genotypes;        /* sim->nGenotypes */
    int8_t alleles2acgt[8];     /* [5] used; 4 = <*>/<NON_REF>, -1 = none (bcf_utils.h:167-180) */
    int8_t acgt2alleles[8];     /* [5] used */
    int32_t info_dp;            /* INFO/DP; 0 => "no reads" record (vcfgl.cpp:228-315) */
    int32_t info_ad[5], info_adf[5], info_adr[5];
    float qs[5];                /* INFO/QS */
    float i16[16];              /* INFO/I16 */
    int32_t _pad;
    int64_t g_off; /* element offset of this site's [n_samples][n_genotypes] block in gl/pl/gp */
    int64_t r_off; /* element offset of this site's [n_samples][n_alleles] block in ad/adf/adr */
} vgl_site_out;

/* results of one batch.  With host_output=1 every pointer is pinned host memory,
 * with host_output=0 every pointer (also `sites`) is device memory and nothing but
 * the two totals and the status word crosses PCIe.  Planes not requested by
 * tag_mask are NULL. */
typedef struct vgl_batch_out {
    int32_t n_sites;
    int32_t n_samples;
    const vgl_site_out* sites; /* [n_sites] */
    const int32_t* dp;         /* FORMAT/DP [n_sites][n_samples] */
    const float* gl;           /* per site: [n_samples][n_genotypes] at sites[i].g_off */
    const int32_t* pl;
    const float* gp;
    const int32_t* ad;         /* per site: [n_samples][n_alleles] at sites[i].r_off */
    const int32_t* adf;
    const int32_t* adr;
    int64_t g_elems, r_elems;  /* used elements of the G- and R-shaped planes */
    int32_t status;            /* VGL_OK or e.g. VGL_ERANGE raised on the device */
    /* VGL_HOST_NARROW only (else 0 / NULL; then dp / pl / ad / adf / adr above are NULL and gl / gp are host pointers).
     * Same element order and the same g_off / r_off element offsets as the int32 planes.
     *   pl_u8   PL is 0..255 by construction (vcfgl.cpp:931-934); a MISSING PL (bcf_int32_missing: cells with FORMAT/DP == 0,
     *           gl_methods.cpp:60-66, 359-366, and every cell of a site with INFO/DP == 0) is stored as 0 -- test dp_n.
     *   dp_n, ad_n, adf_n, adr_n   unsigned, narrow_bits wide: 8 when the depth law is bounded by 255 reads per cell (fixed
     *           depth < 256, or a same-mean Poisson depth with P(n > 255) < 2^-64), else 16.  A value that does not fit is
     *           saturated and the batch status becomes VGL_EOVERFLOW. */
    int32_t narrow_bits;
    const uint8_t* pl_u8;
    const void *dp_n, *ad_n, *adf_n, *adr_n;
    /* VGL_HOST_BCF only (then every plane pointer above is NULL; `sites` is still filled): the records of the kept sites
     * (skip_code == 0) back to back in site order, each one the bytes bcf_write() emits (l_shared, l_indiv, the six
     * fixed words, shared block, FORMAT block).  Site i's record is bcf[bcf_off[i] .. bcf_off[i + 1]) (empty if skipped). */
    const uint8_t* bcf;
    const int64_t* bcf_off;    /* [n_sites + 1] */
    int64_t bcf_bytes;         /* = bcf_off[n_sites] */
    /* VGL_HOST_BGZF only: the same record stream compressed on the device into BGZF blocks (htslib/bgzf.c; the reference's
     * default container, -O b), each block a gzip member holding 32 KiB of the stream.  `bgzf` holds the blocks back to back:
     * the host appends the bytes to the output file after its own (BGZF-compressed) header and closes the file with the 28-byte
     * BGZF EOF block.  `bcf` is NULL in this mode; bcf_off / bcf_bytes still describe the UNCOMPRESSED stream (record i starts at
     * uncompressed offset bcf_off[i], e.g. for an index), bgzf_bytes the compressed one.  The blocks of a context share one
     * dynamic Huffman code built by the first vgl_submit from the symbol statistics of its record stream (that call synchronises
     * the slot's stream once); blocks that would not shrink to three quarters are stored (RFC 1951 3.2.4). */
    const uint8_t* bgzf;
    int64_t bgzf_bytes;
    int32_t bgzf_blocks;
    /* VGL_HOST_BCF with -doGVCF 1 (after vgl_set_gvcf_dps): the batch went through the block merger on the device
     * (prepare_gvcf_block, bcf_utils.cpp:662-942) and `bcf` holds its n_recs records in output order -- regular records and
     * block records (END, MIN_DP, the founder's alleles and QS, per-sample minima of PL and DP) -- with the seam to the
     * neighbouring batches already stitched: a block open at the end of a batch is held back and comes out (merged, if the
     * next batch continues it) in front of the next batch's records, or from vgl_gvcf_flush() after the last batch.  Batches
     * must be waited in submission order (vgl_wait returns VGL_ESTATE for a slot while an older one is still in flight);
     * bcf_off is NULL in this mode. */
    int32_t n_recs;
} vgl_batch_out;

/* timing of a slot's last completed submit, CUDA events on the slot's stream (ms) */
enum { VGL_T_H2D = 0, VGL_T_SIM = 1, VGL_T_SITE = 2, VGL_T_SCAN = 3, VGL_T_EMIT = 4, VGL_T_D2H = 5,
       VGL_T_TOTAL = 6, VGL_T_COUNT = 7 };

/* submit flags */
enum { VGL_SUBMIT_GT_ON_DEVICE = 1 << 0 }; /* skip the H2D copy: reuse the genotypes already in the slot's device buffer */

typedef struct vgl_ctx vgl_ctx;

/* builds the errmod / LUT tables, device buffers, streams and pinned rings */
int vgl_create(const vgl_params* params, vgl_ctx** out);

void vgl_destroy(vgl_ctx* ctx);

/* pinned host input buffer of a slot: uint8 [max_batch_sites][n_samples] packed genotypes */
int vgl_input_buffer(vgl_ctx* ctx, int slot, uint8_t** gt, int64_t* capacity_sites);

/* VGL_HOST_BCF: pinned per-site pass-through records [max_batch_sites] and the blob their byte ranges index.  Fill them
 * for the sites of a batch before vgl_submit(). */
int vgl_bcf_input_buffer(vgl_ctx* ctx, int slot, vgl_bcf_site_in** sites, uint8_t** blob, int64_t* blob_capacity);

/* asynchronous: H2D of the slot's genotypes, all kernels, (host_output) D2H of site records */
int vgl_submit(vgl_ctx* ctx, int slot, int64_t first_site_id, int32_t n_sites,
               const vgl_replay* replay /* NULL = native Philox simulation */, uint32_t flags);

/* blocks until the slot's batch is complete and describes it */
int vgl_wait(vgl_ctx* ctx, int slot, vgl_batch_out* out);

/* make the slot run on a caller-owned cudaStream_t (e.g. torch's current stream); NULL restores the slot's own */
int vgl_set_stream(vgl_ctx* ctx, int slot, void* cuda_stream);

int vgl_slot_timing(vgl_ctx* ctx, int slot, float ms[VGL_T_COUNT]);

/* host_output=0 only: fetch the per-site records of a waited slot into host memory */
int vgl_copy_sites(vgl_ctx* ctx, int slot, vgl_site_out* host_dst);

/* The native simulator's own draws for a range of sites, in exactly the layout of vgl_replay
 * (so they can be replayed, fed to the CPU oracle, or printed as a pileup like the reference's
 * -printPileup, vcfgl.cpp:616-634).  Uses the genotypes currently in the slot's input buffer.
 * Synchronous; host arrays are owned by the context and valid until the next call on the slot. */
typedef struct vgl_draws {
    int64_t n_cells, n_reads;
    const int32_t* depths;       /* [n_cells] (0 where the genotype is missing) */
    const int64_t* read_offsets; /* [n_cells + 1] */
    const uint8_t *bases, *strands, *qs, *adj_qs, *tail_dists; /* [n_reads]; qs/adj_qs only with --error-qs 2 */
    const double* error_probs;   /* [n_reads]: --error-qs 2 the read's own, --error-qs 1 its site's error rate */
} vgl_draws;
int vgl_native_draws(vgl_ctx* ctx, int slot, int64_t first_site_id, int32_t n_sites, vgl_draws* out);

/* number of kernel launches issued by this context so far */
int64_t vgl_launch_count(const vgl_ctx* ctx);

/* which kernel set a native (non-replay) submit of this context runs: "k_tile_m1f" (one kernel: GL model 1 with a
 * run-constant quality score, every tag, one Poisson mean, --depths-file or fixed depth), "k_tile_m2" (one kernel: GL model 2
 * with run constants or the quality-score LUT; GL / PL / AD / DP tags), "k_fused_m1f" (one kernel: remaining GL model 1 /
 * fixed-qs options -- --error-qs 1, cells deeper than 255 reads) or "k_sim+k_site+k_scan+k_emit" (general path; also every
 * replay submit) */
const char* vgl_native_kernels(const vgl_ctx* ctx);

/* algorithmic bytes of a finished batch as defined in DESIGN.md / SURVEY.md 8(d) */
int64_t vgl_algorithmic_bytes(const vgl_batch_out* out, uint32_t tag_mask);

/* Exhaustive on-device check (all 2^32 float bit patterns) that the kernels' arithmetic shortcuts --
 * the 3-instruction /10 and the branch-free lroundf -- equal the reference's expressions
 * (gl_methods.cpp:343, vcfgl.cpp:931).  *n_mismatch must come back 0. */
int vgl_selftest(int device_id, int64_t* n_mismatch, uint32_t* first_mismatch_bits);

/* ------------------------------------------------------------------------------------------------------------------
 * Input path (SURVEY.md 8(f) row 1): VCF text records -> packed true genotypes, on the device.
 *
 * Replaces, for the records of a batch, what the reference's driver loop does per record before the hot path:
 *   bcf_read -> vcf_parse / vcf_parse_format (GT vector)      htslib/vcf.c:3041-3110, 2425-2790
 *   bcf_get_genotypes + check_rec_alleles()                   vcfgl.cpp:75-163
 * The host keeps the header (it supplies record lines only) and everything dictionary-shaped (CHROM -> rid, ID, FILTER,
 * INFO); per record the device returns POS, the allele map, the skip decision of --rm-invar-sites bits 1 / 2 and the
 * byte ranges of the line the host may still want to look at, and leaves the record's genotypes as one row of packed
 * bytes in HBM.  vgl_place_rows() then builds a slot's genotype matrix from those rows -- dropping skipped records and
 * inserting the all-hom-ref sites of -explode 1 (vcfgl.cpp:1480-1538, 1567-1611) -- and the batch is submitted with
 * VGL_SUBMIT_GT_ON_DEVICE: genotypes never exist on the host in unpacked form.
 */
enum { VGL_SOURCE_BINARY = 0, /* --source 0: REF=0 ALT=1, simulated as A / C (vcfgl.cpp:103-127) */
       VGL_SOURCE_ACGT = 1 }; /* --source 1: alleles are bases (vcfgl.cpp:98-101) */

/* per-record status: where the reference would exit (ERROR / ASSERT) the parser reports a code; if a line has several
 * defects the smallest code wins */
typedef enum vgl_in_status {
    VGL_IN_OK = 0,
    VGL_IN_ENCOLS = 1,     /* fewer than 10 columns */
    VGL_IN_EPOS = 2,       /* POS beyond int32 */
    VGL_IN_ENALLELE = 3,   /* > 5 alleles (vcfgl.cpp:90-92) or > 2 with --source 0 (vcfgl.cpp:123-125) */
    VGL_IN_EALLELE = 4,    /* allele not a base (vcfgl.cpp:99-101) / not 0 or 1 (vcfgl.cpp:113-115) */
    VGL_IN_ENOGT = 5,      /* no GT in FORMAT (vcfgl.cpp:83-85) */
    VGL_IN_ENSAMPLES = 6,  /* fewer sample columns than n_samples (htslib/vcf.c:2777-2783) */
    VGL_IN_EGTCHAR = 7,    /* GT not a number or '.', or an invalid character after it (htslib/vcf.c:2666-2669, 2729-2737) */
    VGL_IN_EPLOIDY = 8,    /* a sample is not diploid (the reference reads gt_arr as [2 * n_samples], vcfgl.cpp:131-146) */
    VGL_IN_EALLELEIDX = 9, /* GT allele index >= n_allele (vcfgl.cpp:144) */
    VGL_IN_ESYMBOLIC = 10  /* GT points at <*> / <NON_REF> */
} vgl_in_status;

typedef struct vgl_in_site {
    int32_t status;        /* vgl_in_status */
    int32_t skip_code;     /* 0; -1 all true genotypes hom-ref, -2 all hom-alt (check_rec_alleles, vcfgl.cpp:150-160) */
    int64_t pos;           /* bcf1_t::pos, 0-based */
    int64_t allele_sum;    /* sum of the GT allele indices (vcfgl.cpp:145); computed only when --rm-invar-sites has bit 1 or 2
                            * set (its only use, vcfgl.cpp:150-160), else 0 */
    uint64_t line_off;     /* the record's line in the text chunk ... */
    uint32_t line_len;     /* ... without its LF (and CR) */
    int32_t n_allele;      /* bcf1_t::n_allele */
    int8_t allele_acgt[8]; /* [5] used: rec_alleles[] of check_rec_alleles (4 = <*> / <NON_REF>, -1 = none / invalid) */
    uint32_t id_off, fmt_off, samples_off; /* start of the ID, FORMAT and first sample column, relative to line_off */
    uint32_t _pad;
} vgl_in_site;

typedef struct vgl_parser vgl_parser;

/* a parser belongs to a context (device, n_samples, --rm-invar-sites); it owns a pinned text staging buffer, the device
 * copy of the text, the record index and the genotype rows [max_records][n_samples], and its own stream */
int vgl_parser_create(vgl_ctx* ctx, int64_t max_text_bytes /* < 4 GiB */, int32_t max_records, vgl_parser** out);
void vgl_parser_destroy(vgl_parser* ps);
int vgl_parser_text_buffer(vgl_parser* ps, uint8_t** text, int64_t* capacity);

enum { VGL_PARSE_FINAL = 1 << 0,           /* last chunk of the file: a tail without LF is a record too */
       VGL_PARSE_TEXT_ON_DEVICE = 1 << 1 }; /* reuse the text already on the device (skips the H2D copy) */

typedef struct vgl_parse_out {
    int32_t n_records;           /* complete lines parsed (at most max_records) */
    int32_t n_errors;            /* records with status != VGL_IN_OK */
    int32_t first_error_record;  /* -1 if none */
    int32_t n_kept;              /* records with status OK and skip_code 0 */
    int64_t bytes_consumed;      /* text bytes covered by those records: carry the rest over to the next chunk */
    const vgl_in_site* sites;    /* [n_records], pinned host memory owned by the parser */
    float ms_h2d, ms_kernels;    /* CUDA events on the parser's stream */
} vgl_parse_out;

/* synchronous: H2D of the text, k_vcf_lines (record index), k_vcf_gt (columns, alleles, genotypes), D2H of the site records */
int vgl_parse_vcf(vgl_parser* ps, int64_t n_bytes, int32_t gt_source, uint32_t flags, vgl_parse_out* out);

/* The same for uncompressed BCF records (the reference reads VCF and BCF through the same bcf_read, vcfgl.cpp:1479): the text
 * buffer holds the records' bytes as they follow the BCF header (BGZF already inflated by the host), rec_off[0 .. n_records]
 * their byte offsets (record i = [rec_off[i], rec_off[i + 1]); the host finds them by hopping l_shared + l_indiv + 8), gt_key the
 * dictionary id of FORMAT/GT in the input header (bcf_hdr_id2int(hdr, BCF_DT_ID, "GT")).  k_bcf_gt decodes the fixed fields, the
 * allele strings and the typed GT vector (htslib/vcf.c:1535-1600 bcf_unpack, bcf_get_genotypes) and applies
 * check_rec_alleles (vcfgl.cpp:75-163).  vgl_in_site: line_off / line_len = the record's bytes, id_off = 32,
 * fmt_off = start of the FORMAT block, samples_off = start of the GT values; everything else as for text. */
int vgl_parse_bcf(vgl_parser* ps, int64_t n_bytes, const uint32_t* rec_off, int32_t n_records, int32_t gt_source, int32_t gt_key, uint32_t flags,
                  vgl_parse_out* out);

/* copies genotype rows of the last parse to host memory (tests, debugging): host_dst [n_records][n_samples] */
int vgl_parser_rows(vgl_parser* ps, int32_t first_record, int32_t n_records, uint8_t* host_dst);

/* builds slot `slot`'s device genotype matrix: site r takes the row of record row_map[r], or fill_gt in every sample when
 * row_map[r] < 0 (an -explode 1 site: the blank record's GT is 0|0, i.e. VGL_GT_PACK(ref, ref)).  row_map == NULL selects
 * records first_record .. first_record + n_sites - 1.  Asynchronous on the slot's stream; follow with
 * vgl_submit(..., VGL_SUBMIT_GT_ON_DEVICE). */
int vgl_place_rows(vgl_ctx* ctx, int slot, vgl_parser* ps, const int32_t* row_map, int32_t first_record, int32_t n_sites, uint8_t fill_gt);

/* ------------------------------------------------------------------------------------------------------------------
 * gVCF block merging on the device (SURVEY.md 8(f) row 3): what prepare_gvcf_block() (bcf_utils.cpp:662-942) decides
 * and accumulates while write_record_values() (vcfgl.cpp:165-207) walks the written sites of a -doGVCF 1 run.
 *
 * Call after vgl_wait() on a slot (its planes are still in HBM): the device classifies every written site (skip_code 0)
 * as a block member or not (one observed allele and min FORMAT/DP inside a --gvcf-dps range, bcf_utils.cpp:692, 741-765),
 * cuts the site sequence into records (a member joins the block before it iff same contig, pos <= end + 1, same range:
 * bcf_utils.cpp:711, 719, 790) and reduces each block: MIN_DP, DP[s] = min over members, PL[s] = the founder's PL[3s] and the
 * lexicographic minimum of (PL[3s+1], PL[3s+2]) (bcf_utils.cpp:838-866).  The host writes regular records as before and
 * block records from the founder's alleles / QS plus these arrays (bcf_utils.cpp:876-905).  A batch's first block may
 * continue the previous batch's last one: same three conditions, the same minima (vgl_host.hpp GvcfStitcher).
 * Needs -doUnobserved 1 or 2 (members then have REF + <*>, three genotypes), FORMAT/DP and int32 planes on the device
 * (any host_output except VGL_HOST_BCF).
 */
#define VGL_MAX_GVCF_DPS 16

typedef struct vgl_gvcf_site_in {
    int32_t rid, pos; /* bcf1_t::rid, ::pos of every site of the batch, written or not */
} vgl_gvcf_site_in;

typedef struct vgl_gvcf_rec {
    int32_t first_site, last_site; /* batch indices of the first / last member; a regular record: both the site itself */
    int32_t n_members;             /* 0: write the site as it is (GVCF_WRITE_SIMREC); >= 1: a block of that many written sites */
    int32_t min_dp;                /* INFO/MIN_DP of a block (a regular record: the site's minimum FORMAT/DP) */
    int32_t dp_range;              /* 1-based --gvcf-dps range of a block, 0 for a regular record */
    int32_t plane;                 /* block: its DP at dp + plane * n_samples, its PL at pl + plane * 3 * n_samples; else -1 */
} vgl_gvcf_rec;

typedef struct vgl_gvcf_out {
    int32_t n_recs, n_blocks;
    const vgl_gvcf_rec* recs; /* [n_recs] in output order, pinned host memory owned by the context */
    const int32_t* dp;        /* [n_blocks][n_samples] */
    const int32_t* pl;        /* [n_blocks][n_samples][3], NULL without the PL tag */
    float ms_kernels;
} vgl_gvcf_out;

/* VGL_HOST_BCF with -doGVCF 1: the ascending --gvcf-dps thresholds, once, before the first vgl_submit; and, after the last
 * vgl_wait, the block that was still open (write_record_values(NULL), vcfgl.cpp:169-177): *n_bytes = 0 when there is none.
 * The returned bytes stay valid until the next call on the context. */
int vgl_set_gvcf_dps(vgl_ctx* ctx, const int32_t* gvcf_dps, int32_t n_gvcf_dps);
int vgl_gvcf_flush(vgl_ctx* ctx, const uint8_t** rec, int64_t* n_bytes);

/* synchronous; sites: host array [n_sites of the slot's last batch]; gvcf_dps: ascending thresholds of --gvcf-dps */
int vgl_gvcf_merge(vgl_ctx* ctx, int slot, const vgl_gvcf_site_in* sites, const int32_t* gvcf_dps, int32_t n_gvcf_dps, vgl_gvcf_out* out);

/* On-device genotype-call discordance of the slot's last (waited) batch (SURVEY.md 8(f) row 4): the hom / het comparison of
 * misc/gtDiscordance.cpp:11-15 between the call implied by the simulated likelihoods -- the genotype with the single largest
 * GL; a tie is no call and counts as discordant -- and the true genotype, over the cells of written sites with INFO/DP > 0 and
 * FORMAT/DP > 0.  Needs the GL tag and FORMAT/DP.  Synchronous; 60 bytes read per cell, 32 bytes returned. */
typedef struct vgl_discordance_out {
    int64_t n_hom, n_hom_discordant; /* cells whose true genotype is homozygous / of those, calls that differ */
    int64_t n_het, n_het_discordant;
    float ms_kernel;
} vgl_discordance_out;
int vgl_discordance(vgl_ctx* ctx, int slot, vgl_discordance_out* out);

const char* vgl_strerror(int status);
const char* vgl_last_error(const vgl_ctx* ctx);
int vgl_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* VGL_H */
