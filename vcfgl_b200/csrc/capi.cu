// C-ABI layer of libvgl.so (include/vgl.h): context, slots, pinned rings, streams,
// batch submit / wait.  Host code here only moves data and launches kernels; every
// per-cell computation happens in kernels.cu.  There is no CPU path.
#include "tables.h"
#include "vgl_internal.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <thread>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

using namespace vgl;

namespace {

enum { EV_START = 0, EV_H2D, EV_SIM, EV_SITE, EV_SCAN, EV_EMIT, EV_META, EV_D2H0, EV_D2H1, EV_KDONE, EV_BCF, EV_COUNT };

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

// The FORMAT planes of a batch.  GL and GP hold floats, the others int32; both are 4 bytes wide.
enum { P_DP, P_GL, P_GP, P_PL, P_AD, P_ADF, P_ADR, P_COUNT };
enum PlaneShape { PER_CELL, PER_GENOTYPE, PER_ALLELE };
enum PlaneNarrow { NARROW_NONE, NARROW_DEPTH, NARROW_PL }; // VGL_HOST_NARROW: not narrowed, to narrow_bits, to 8 bits (0..255)
struct PlaneDesc { uint32_t tag; PlaneShape shape; PlaneNarrow narrow; };
const PlaneDesc kPlanes[P_COUNT] = {
    {0, PER_CELL, NARROW_DEPTH}, // always there: the kernels write the depths whatever the tags
    {VGL_TAG_GL, PER_GENOTYPE, NARROW_NONE},
    {VGL_TAG_GP, PER_GENOTYPE, NARROW_NONE},
    {VGL_TAG_PL, PER_GENOTYPE, NARROW_PL},
    {VGL_TAG_FMT_AD, PER_ALLELE, NARROW_DEPTH},
    {VGL_TAG_FMT_ADF, PER_ALLELE, NARROW_DEPTH},
    {VGL_TAG_FMT_ADR, PER_ALLELE, NARROW_DEPTH},
};
// elements of plane i when the batch has `cells` cells and g / r elements in the G- / R-shaped planes
size_t plane_elems(int i, size_t cells, size_t g, size_t r)
{
    return kPlanes[i].shape == PER_CELL ? cells : kPlanes[i].shape == PER_GENOTYPE ? g : r;
}
struct PlaneBufs {
    void* d = nullptr;  // device, zeroed once at creation
    void* dn = nullptr; // VGL_HOST_NARROW: device, narrowed
    void* h = nullptr;  // pinned host: VGL_HOST_I32, and the planes VGL_HOST_NARROW does not narrow
    void* hn = nullptr; // VGL_HOST_NARROW: pinned host, narrowed
};

struct Slot {
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaEvent_t ev[EV_COUNT] = {};
    bool submitted = false;
    bool waited = false;
    int32_t n_sites = 0;
    int64_t seq = 0; // the context's submit count when this slot was last submitted (the order of the batches in flight)
    // host (pinned)
    uint8_t* h_gt = nullptr;
    vgl_site_out* h_sites = nullptr;
    int64_t* h_totals = nullptr; // [0..1] plane extents, [2] status, [3] record-stream bytes, [4] BGZF bytes, [5] BGZF blocks
    PlaneBufs plane[P_COUNT];
    template <typename T = int32_t> T* dev(int i) const { return static_cast<T*>(plane[i].d); }
    // VGL_HOST_BCF: pass-through input (pinned + device), plan arrays, the record stream (device + pinned)
    vgl_bcf_site_in *h_bcf_in = nullptr, *d_bcf_in = nullptr;
    uint8_t *h_blob = nullptr, *d_blob = nullptr, *d_bcf = nullptr, *h_bcf = nullptr;
    BcfSiteMinMax* d_minmax = nullptr;
    uint32_t* d_rec_len = nullptr;
    long long *d_rec_off = nullptr, *h_rec_off = nullptr;
    // VGL_HOST_BGZF: plane layout of every record, block staging, block sizes / offsets, the compressed stream (device + pinned)
    BcfRecPlanes* d_planes = nullptr;
    uint8_t *d_stage = nullptr, *d_bgzf = nullptr, *h_bgzf = nullptr;
    uint32_t* d_blk_rng = nullptr;
    uint32_t* d_blk_size = nullptr;
    long long* d_blk_off = nullptr;
    int32_t* d_blk_first = nullptr;
    // device
    uint8_t* d_gt = nullptr;
    CellRec* d_cell = nullptr;
    CellQ* d_cellq = nullptr;
    CellTail* d_celltail = nullptr;
    vgl_site_out* d_sites = nullptr;
    int64_t* d_totals = nullptr; // [2] totals, then int32 status at [2]
    uint64_t* d_pairmap = nullptr;
    unsigned long long* d_tile_state = nullptr; // fused: [max tiles] look-back words, then the ticket
    // vgl_gvcf_merge(): allocated on first use
    vgl_gvcf_site_in* g_sin = nullptr;
    int2* g_key = nullptr;
    vgl_gvcf_rec *g_recs = nullptr, *hg_recs = nullptr;
    int32_t *g_prev = nullptr, *g_kidx = nullptr, *g_counts = nullptr, *hg_counts = nullptr, *g_blast = nullptr;
    unsigned long long *g_local = nullptr, *g_bsum = nullptr;
    int32_t *g_dp = nullptr, *g_pl = nullptr, *hg_dp = nullptr, *hg_pl = nullptr;
    cudaEvent_t g_ev[2] = {};
    unsigned long long *d_disc = nullptr, *h_disc = nullptr; // vgl_discordance()
    // replay uploads (grown on demand)
    DevBuf r_depths, r_off, r_bases, r_strands, r_qs, r_adjqs, r_eprob, r_tails, r_deep_cells, r_deep_codes;
    float ms[VGL_T_COUNT] = {};
    bool had_d2h = false;
    bool early_d2h = false; // the plane copies were enqueued by vgl_submit (tile kernels: the spans are known on the host)
    int64_t stream_copied = 0; // VGL_HOST_BCF / BGZF: bytes of the record stream vgl_submit already copied on a prediction
    const uint8_t* seam_ptr = nullptr; // -doGVCF: the stream vgl_wait hands out after the seam was stitched
    int64_t seam_bytes = 0;
    int32_t seam_recs = 0;
    // vgl_native_draws() results (host)
    std::vector<int32_t> dr_depths;
    std::vector<int64_t> dr_off;
    std::vector<uint8_t> dr_bases, dr_strands, dr_qs, dr_adjqs, dr_tails;
    std::vector<double> dr_eprob;
};

} // namespace

struct vgl_ctx {
    vgl_params prm;
    std::vector<double> depth_means;
    RunPlan plan; // the run constants and the kernel set (plan_run)
    int n_sms = 148;
    int narrow_bits = 0;                   // VGL_HOST_NARROW: width of the DP / AD planes (8 or 16), 0 = int32 planes
    size_t bcf_cap = 0, blob_cap = 0;      // VGL_HOST_BCF: bytes per slot of the record stream / the pass-through blob
    int64_t bgzf_max_blocks = 0;           // VGL_HOST_BGZF: blocks a full record stream makes
    BgzfCode* d_bgzf_code = nullptr;       // the context's prefix code (deflate's fixed code until the statistics pass)
    uint32_t* d_bgzf_hist = nullptr;       // symbol counts of the statistics pass
    bool bgzf_code_ready = false;          // built from the first batch's record stream (vgl_submit)
    double stream_bytes_per_site = 0.0;    // VGL_HOST_BCF / BGZF: bytes per site of the last finished batch (predicts the next copy)
    // VGL_HOST_BCF with -doGVCF: thresholds, and the block still open at the end of the last waited batch (the seam)
    std::vector<int32_t> gvcf_dps;
    struct Carry {
        bool open = false;
        int32_t rid = 0, start = 0, end = 0, range = 0, min_dp = 0, n_alleles = 0;
        int8_t a2b[8] = {0};
        float qs[5] = {0};
        std::vector<int32_t> dp, pl;
        std::vector<uint8_t> rec; // its record as it stands
    } carry;
    size_t bcf_headroom = 0;               // bytes in front of a slot's pinned record stream (a re-encoded seam block goes there)
    std::vector<uint8_t> flush_rec;
    cudaEvent_t chain_ev = nullptr;        // kernels of the previous submit are done (see vgl_submit)
    int64_t submit_seq = 0;                // submits so far (Slot::seq)
    uint32_t* d_crc_pow = nullptr;
    uint32_t *d_qcls = nullptr, *d_m2_cmap = nullptr, *d_qm_cdf = nullptr;
    float *d_m2_pure = nullptr, *d_m2_park = nullptr;
    void* d_m1_pure = nullptr;
    double* d_m2_tab = nullptr;
    unsigned long long *d_pois = nullptr, *d_alias = nullptr;
    uint16_t* d_alias_row = nullptr; // --depths-file: each sample's row in d_alias
    uint32_t *d_errcdf = nullptr, *d_cnt_scratch = nullptr;
    int pois_n = 0;
    double *d_lut = nullptr, *d_m1_bsum = nullptr, *d_m1_het = nullptr, *d_fk = nullptr, *d_beta = nullptr, *d_depth_means = nullptr;
    std::vector<Slot> slots;
    size_t g_cap = 0, r_cap = 0; // per-slot plane capacity in elements
    int64_t launches = 0;
    std::string err;
};

#define CK(call)                                                                           \
    do {                                                                                   \
        cudaError_t e_ = (call);                                                           \
        if (e_ != cudaSuccess) {                                                           \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                \
            return VGL_ECUDA;                                                              \
        }                                                                                  \
    } while (0)

static int fail(vgl_ctx* ctx, int code, const char* msg)
{
    if (ctx) ctx->err = msg;
    return code;
}

// bytes per element of plane i narrowed (VGL_HOST_NARROW)
static size_t narrow_bytes(const vgl_ctx* ctx, int i) { return kPlanes[i].narrow == NARROW_PL ? 1 : (size_t)ctx->narrow_bits / 8; }

// kernel sets that run one kernel per batch (a tile state: look-back words and the ticket)
static bool one_kernel(KernelSet k) { return k == KS_FUSED_M1F || k == KS_TILE_M1F || k == KS_TILE_M2; }

extern "C" int vgl_abi_version(void) { return VGL_ABI_VERSION; }

extern "C" const char* vgl_strerror(int s)
{
    switch (s) {
    case VGL_OK: return "ok";
    case VGL_EINVAL: return "invalid argument or unsupported option combination";
    case VGL_ENOMEM: return "out of memory";
    case VGL_ECUDA: return "CUDA runtime error";
    case VGL_ESTATE: return "slot in wrong state";
    case VGL_ERANGE: return "quality score outside every --qs-bins range";
    case VGL_ENODEV: return "no CUDA device available (libvgl has no CPU path)";
    case VGL_EOVERFLOW: return "a depth did not fit the narrow planes (VGL_HOST_NARROW)";
    case VGL_EMISSING: return "missing true genotype with --depth inf";
    default: return "unknown status";
    }
}

extern "C" const char* vgl_last_error(const vgl_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

extern "C" int64_t vgl_launch_count(const vgl_ctx* ctx) { return ctx ? ctx->launches : 0; }

extern "C" const char* vgl_native_kernels(const vgl_ctx* ctx)
{
    return ctx ? kernel_set_name(ctx->plan.set) : "";
}

extern "C" int64_t vgl_algorithmic_bytes(const vgl_batch_out* o, uint32_t tag_mask)
{
    // SURVEY.md 8(d): 1 B packed genotype in + int32/float32 planes as handed to htslib
    int64_t b = 0;
    const int64_t S = o->n_samples;
    for (int i = 0; i < o->n_sites; ++i) {
        const vgl_site_out& s = o->sites[i];
        b += S; // genotypes are read for every site, also skipped ones
        if (s.skip_code != 0) continue;
        const int64_t G = s.n_genotypes, A = s.n_alleles;
        const int ng = !!(tag_mask & VGL_TAG_GL) + !!(tag_mask & VGL_TAG_PL) + !!(tag_mask & VGL_TAG_GP);
        const int na = !!(tag_mask & VGL_TAG_FMT_AD) + !!(tag_mask & VGL_TAG_FMT_ADF) + !!(tag_mask & VGL_TAG_FMT_ADR);
        b += 4 * S * (G * ng + A * na + !!(tag_mask & VGL_TAG_FMT_DP));
        b += 4 * (16 * !!(tag_mask & VGL_TAG_I16) + A * (!!(tag_mask & VGL_TAG_QS) + !!(tag_mask & VGL_TAG_INFO_AD) +
                                                          !!(tag_mask & VGL_TAG_INFO_ADF) + !!(tag_mask & VGL_TAG_INFO_ADR)) +
                  !!(tag_mask & VGL_TAG_INFO_DP));
    }
    return b;
}

static int validate(const vgl_params* p, std::string& why)
{
    // the option rules of io.cpp:860-1000 that concern the hot path
    if (p->abi_version != VGL_ABI_VERSION) { why = "abi_version mismatch"; return VGL_EINVAL; }
    if (p->n_samples < 1) { why = "n_samples < 1"; return VGL_EINVAL; }
    if (p->max_batch_sites < 1 || p->n_slots < 1 || p->n_slots > 8) { why = "bad max_batch_sites / n_slots"; return VGL_EINVAL; }
    if (p->depth_mode < 0 || p->depth_mode > 3) { why = "bad depth_mode"; return VGL_EINVAL; }
    if (p->depth_mode == VGL_DEPTH_INF) { // io.cpp:783-800, 1012-1019
        if (p->tag_mask & ~(uint32_t)(VGL_TAG_GL | VGL_TAG_GP | VGL_TAG_PL)) { why = "--depth inf: only GL, GP and PL exist (no reads: -addFormatDP 0 etc.)"; return VGL_EINVAL; }
        if (p->do_gvcf || (p->rm_invar_sites & 4)) { why = "--depth inf cannot be used with -doGVCF 1 or --rm-invar-sites 4"; return VGL_EINVAL; }
        if (p->error_rate != 0.0) { why = "--depth inf requires --error-rate 0 (io.cpp:847-853)"; return VGL_EINVAL; }
        if (p->host_output == VGL_HOST_BCF || p->host_output == VGL_HOST_BGZF || p->host_output == VGL_HOST_NARROW) { why = "--depth inf: host_output must be VGL_HOST_NONE or VGL_HOST_I32"; return VGL_EINVAL; }
    }
    if (p->depth_mode == VGL_DEPTH_POISSON_PER_SAMPLE && !p->depth_means) { why = "depth_means missing"; return VGL_EINVAL; }
    if (p->depth_mode != VGL_DEPTH_POISSON_PER_SAMPLE && p->depth_mode != VGL_DEPTH_INF && !(p->depth_mean >= 0.0 && p->depth_mean <= 500.0)) { why = "--depth out of [0,500]"; return VGL_EINVAL; }
    if (!(p->error_rate >= 0.0 && p->error_rate < 1.0)) { why = "--error-rate out of [0,1)"; return VGL_EINVAL; }
    if (p->error_qs < 0 || p->error_qs > 2) { why = "--error-qs out of [0,2]"; return VGL_EINVAL; }
    if (p->gl_model < 1 || p->gl_model > 2) { why = "--gl-model out of [1,2]"; return VGL_EINVAL; }
    if (!(p->gl1_theta >= 0.0 && p->gl1_theta <= 1.0)) { why = "--gl1-theta out of [0,1]"; return VGL_EINVAL; }
    if (p->precise_gl && p->gl_model == 1) { why = "--precise-gl 1 is not supported with --gl-model 1"; return VGL_EINVAL; }
    if (p->adjust_qs < 0 || p->adjust_qs > 31) { why = "--adjust-qs out of range"; return VGL_EINVAL; }
    if (p->adjust_qs && p->adjust_by == 0.0) { why = "--adjust-qs requires non-zero --adjust-by"; return VGL_EINVAL; }
    if ((p->adjust_qs & 1) && p->precise_gl) { why = "--adjust-qs 1 requires --precise-gl 0"; return VGL_EINVAL; }
    if ((p->adjust_qs & 2) && !(p->tag_mask & VGL_TAG_QS)) { why = "--adjust-qs 2 requires -addQS 1"; return VGL_EINVAL; }
    if (p->error_qs != 0) {
        if (!(p->error_rate > 0.0)) { why = "--error-qs 1|2 requires --error-rate > 0"; return VGL_EINVAL; }
        if (!(p->beta_variance > 0.0)) { why = "--error-qs 1|2 requires --beta-variance > 0"; return VGL_EINVAL; }
    }
    if (p->do_unobserved < 0 || p->do_unobserved > 5) { why = "-doUnobserved out of [0,5]"; return VGL_EINVAL; }
    if (p->i16_mapq < 0 || p->i16_mapq > 60) { why = "--i16-mapq out of [0,60]"; return VGL_EINVAL; }
    if (p->n_qs_bins < 0 || p->n_qs_bins > 255) { why = "bad n_qs_bins"; return VGL_EINVAL; }
    if (p->sampler < 0 || p->sampler > 2) { why = "bad sampler"; return VGL_EINVAL; }
    if (p->host_output < 0 || p->host_output > 4) { why = "bad host_output"; return VGL_EINVAL; }
    if (p->host_output == VGL_HOST_BCF && p->do_gvcf && ((p->do_unobserved != 1 && p->do_unobserved != 2) || !(p->tag_mask & VGL_TAG_FMT_DP))) {
        why = "VGL_HOST_BCF with -doGVCF needs -doUnobserved 1|2 and FORMAT/DP (the block merger's requirements)";
        return VGL_EINVAL;
    }
    if (p->host_output == VGL_HOST_BGZF && p->do_gvcf) { why = "VGL_HOST_BCF does not take -doGVCF (the block merger consumes arrays)"; return VGL_EINVAL; }
    if ((p->host_output == VGL_HOST_BCF || p->host_output == VGL_HOST_BGZF) && (p->bcf_blob_bytes_per_site < 0 || p->bcf_blob_bytes_per_site > 65536)) { why = "bad bcf_blob_bytes_per_site"; return VGL_EINVAL; }
    if (p->sampler == VGL_SAMPLER_COUNTS && !(p->gl_model == 1 && p->error_qs != 2)) { why = "count-level sampler needs --gl-model 1 and --error-qs 0|1"; return VGL_EINVAL; }
    if (p->sampler == VGL_SAMPLER_COUNTS && (p->tag_mask & (VGL_TAG_QS | VGL_TAG_I16))) { why = "count-level sampler does not produce QS / I16 (use VGL_SAMPLER_PER_READ)"; return VGL_EINVAL; }
    return VGL_OK;
}

template <typename T>
static cudaError_t upload(T** d, const std::vector<T>& h) // an empty table leaves *d null
{
    if (h.empty()) return cudaSuccess;
    cudaError_t e = cudaMalloc((void**)d, h.size() * sizeof(T));
    if (e != cudaSuccess) return e;
    return cudaMemcpy(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice);
}

extern "C" void vgl_destroy(vgl_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->prm.device_id);
    for (Slot& s : ctx->slots) {
        if (s.own_stream) cudaStreamSynchronize(s.own_stream);
        for (auto& e : s.ev)
            if (e) cudaEventDestroy(e);
        cudaFree(s.g_sin); cudaFree(s.g_key); cudaFree(s.g_recs); cudaFreeHost(s.hg_recs); cudaFree(s.g_prev); cudaFree(s.g_kidx);
        cudaFree(s.g_counts); cudaFreeHost(s.hg_counts); cudaFree(s.g_blast); cudaFree(s.g_local); cudaFree(s.g_bsum); cudaFree(s.g_dp); cudaFree(s.g_pl); cudaFreeHost(s.hg_dp); cudaFreeHost(s.hg_pl);
        for (auto& e : s.g_ev)
            if (e) cudaEventDestroy(e);
        cudaFree(s.d_disc); cudaFreeHost(s.h_disc);
        cudaFreeHost(s.h_gt); cudaFreeHost(s.h_sites); cudaFreeHost(s.h_totals);
        for (PlaneBufs& b : s.plane) {
            cudaFree(b.d); cudaFree(b.dn); cudaFreeHost(b.h); cudaFreeHost(b.hn);
        }
        cudaFreeHost(s.h_bcf_in); cudaFreeHost(s.h_blob); cudaFreeHost(s.h_bcf); cudaFreeHost(s.h_rec_off);
        cudaFree(s.d_bcf_in); cudaFree(s.d_blob); cudaFree(s.d_bcf); cudaFree(s.d_minmax); cudaFree(s.d_rec_len); cudaFree(s.d_rec_off);
        cudaFree(s.d_planes); cudaFree(s.d_stage); cudaFree(s.d_bgzf); cudaFreeHost(s.h_bgzf); cudaFree(s.d_blk_size); cudaFree(s.d_blk_off); cudaFree(s.d_blk_first); cudaFree(s.d_blk_rng);
        cudaFree(s.d_gt); cudaFree(s.d_cell); cudaFree(s.d_cellq); cudaFree(s.d_celltail);
        cudaFree(s.d_sites); cudaFree(s.d_totals); cudaFree(s.d_pairmap); cudaFree(s.d_tile_state);
        for (DevBuf* b : {&s.r_depths, &s.r_off, &s.r_bases, &s.r_strands, &s.r_qs, &s.r_adjqs, &s.r_eprob, &s.r_tails, &s.r_deep_cells, &s.r_deep_codes})
            cudaFree(b->p);
        if (s.own_stream) cudaStreamDestroy(s.own_stream);
    }
    cudaFree(ctx->d_lut); cudaFree(ctx->d_m1_bsum); cudaFree(ctx->d_m1_het); cudaFree(ctx->d_fk); cudaFree(ctx->d_beta);
    cudaFree(ctx->d_depth_means); cudaFree(ctx->d_pois); cudaFree(ctx->d_alias); cudaFree(ctx->d_alias_row); cudaFree(ctx->d_bgzf_code); cudaFree(ctx->d_bgzf_hist); cudaFree(ctx->d_errcdf); cudaFree(ctx->d_cnt_scratch); cudaFree(ctx->d_qcls); cudaFree(ctx->d_m2_cmap); cudaFree(ctx->d_m2_tab); cudaFree(ctx->d_qm_cdf); cudaFree(ctx->d_m2_pure); cudaFree(ctx->d_m2_park); cudaFree(ctx->d_m1_pure); cudaFree(ctx->d_crc_pow);
    delete ctx;
}

static int create_impl(vgl_ctx* ctx)
{
    const vgl_params& p = ctx->prm;
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) return fail(ctx, VGL_ENODEV, "no CUDA device");
    if (p.device_id < 0 || p.device_id >= n_dev) return fail(ctx, VGL_EINVAL, "device_id out of range");
    CK(cudaSetDevice(p.device_id));

    PlanTables tab;
    const char* why = "";
    const int rc = plan_run(p, ctx->depth_means.data(), !getenv("VGL_NO_TILE"), &ctx->plan, &tab, &why);
    if (rc != VGL_OK) return fail(ctx, rc, why);
    const KernelSet ks = ctx->plan.set;
    const uint32_t t = p.tag_mask;

    // ---- tables
    CK(upload(&ctx->d_lut, std::vector<double>(&kLutLog10Gl[0][0], &kLutLog10Gl[0][0] + 3 * 257)));
    CK(upload(&ctx->d_m1_het, tab.m1_het));
    CK(upload(&ctx->d_m1_bsum, tab.m1_bsum));
    CK(upload(&ctx->d_fk, tab.fk));
    CK(upload(&ctx->d_beta, tab.beta));
    CK(upload(&ctx->d_depth_means, ctx->depth_means));
    CK(upload(&ctx->d_pois, tab.pois_cdf));
    ctx->pois_n = (int)tab.pois_cdf.size();
    CK(cudaDeviceGetAttribute(&ctx->n_sms, cudaDevAttrMultiProcessorCount, p.device_id));
    if (ks == KS_TILE_M2) {
        CK(upload(&ctx->d_qcls, tab.qcls));
        if (p.error_qs == 2) CK(upload(&ctx->d_qm_cdf, binomial_cdf4_u32(ctx->plan.q_minor)));
        CK(upload(&ctx->d_m2_tab, tab.m2_tab));
        CK(upload(&ctx->d_m2_cmap, m2_class_map()));
        CK(upload(&ctx->d_m2_pure, tab.m2_pure));
    }
    // closed form of cells whose reads all show one base: worth its branch when most 32-cell chunks hold no mis-called read
    // (expected mis-called reads per chunk = 32 x depth x error rate below ~1/2; heterozygous cells are the input's business)
    double exp_depth = p.depth_mode == VGL_DEPTH_POISSON || p.depth_mode == VGL_DEPTH_FIXED ? p.depth_mean : 0.0;
    for (double d : ctx->depth_means) exp_depth = std::max(exp_depth, d);
    if (ks == KS_TILE_M1F && 32.0 * exp_depth * p.error_rate < 0.5 && !getenv("VGL_NO_PURE")) {
        CK(cudaMalloc(&ctx->d_m1_pure, 256 * sizeof(M1Pure)));
        if (!build_m1f_pure_table(ctx->d_m1_bsum, ctx->d_m1_het, ctx->d_m1_pure, nullptr)) {
            cudaFree(ctx->d_m1_pure);
            ctx->d_m1_pure = nullptr;
        }
    }
    // narrow host planes: 8 bits when no cell can hold more than 255 reads (the truncated tail of the Poisson law is below 2^-64)
    if (p.host_output == VGL_HOST_NARROW) ctx->narrow_bits = ctx->plan.alias_ok ? 8 : 16;
    if (ks == KS_TILE_M1F || ks == KS_TILE_M2) {
        CK(upload(&ctx->d_alias, tab.alias));
        CK(upload(&ctx->d_alias_row, tab.alias_row));
        CK(upload(&ctx->d_errcdf, binomial_cdf4_u32(p.error_rate)));
        const size_t words = ks == KS_TILE_M2 ? tile_m2_row_words(p.n_samples, ctx->n_sms) : tile_m1f_scratch_words(p.n_samples, ctx->n_sms);
        if (words) CK(cudaMalloc((void**)&ctx->d_cnt_scratch, words * 4));
        if (ks == KS_TILE_M2) CK(cudaMalloc((void**)&ctx->d_m2_park, tile_m2_park_floats(p.n_samples, ctx->n_sms) * sizeof(float)));
    }

    // ---- slots
    const size_t B = (size_t)p.max_batch_sites, S = (size_t)p.n_samples, cells = B * S, cells4 = (cells + 3) & ~(size_t)3;
    ctx->g_cap = B * ((S * 15 + 3) & ~(size_t)3);
    ctx->r_cap = B * ((S * 5 + 3) & ~(size_t)3);
    ctx->slots.resize(p.n_slots);
    for (Slot& s : ctx->slots) {
        CK(cudaStreamCreateWithFlags(&s.own_stream, cudaStreamNonBlocking));
        s.stream = s.own_stream;
        for (auto& e : s.ev) CK(cudaEventCreate(&e));
        CK(cudaHostAlloc((void**)&s.h_gt, cells, cudaHostAllocDefault));
        CK(cudaHostAlloc((void**)&s.h_sites, B * sizeof(vgl_site_out), cudaHostAllocDefault));
        CK(cudaHostAlloc((void**)&s.h_totals, 8 * sizeof(int64_t), cudaHostAllocDefault));
        CK(cudaMalloc((void**)&s.d_gt, cells));
        CK(cudaMalloc((void**)&s.d_cell, cells * sizeof(CellRec)));
        if (ctx->plan.need_cellq) CK(cudaMalloc((void**)&s.d_cellq, cells * sizeof(CellQ)));
        if (ctx->plan.need_tail) CK(cudaMalloc((void**)&s.d_celltail, cells * sizeof(CellTail)));
        CK(cudaMalloc((void**)&s.d_sites, B * sizeof(vgl_site_out)));
        CK(cudaMalloc((void**)&s.d_totals, 8 * sizeof(int64_t)));
        CK(cudaMalloc((void**)&s.d_pairmap, B * sizeof(uint64_t)));
        if (one_kernel(ks)) {
            CK(cudaMalloc((void**)&s.d_tile_state, (B + 2) * sizeof(unsigned long long)));
            CK(cudaMemset(s.d_tile_state, 0, (B + 2) * sizeof(unsigned long long)));
        }
        CK(cudaMemset(s.d_totals, 0, 8 * sizeof(int64_t)));
        for (int i = 0; i < P_COUNT; ++i) {
            if (kPlanes[i].tag && !(t & kPlanes[i].tag)) continue;
            PlaneBufs& b = s.plane[i];
            const size_t n = plane_elems(i, cells4, ctx->g_cap, ctx->r_cap);
            // zeroed once: words the kernels never write (block padding of the general path, tile-end holes) must not hold
            // another allocation's bits when a whole span is narrowed or copied to the host
            CK(cudaMalloc(&b.d, n * 4));
            CK(cudaMemset(b.d, 0, n * 4));
            if (p.host_output == VGL_HOST_NARROW && kPlanes[i].narrow != NARROW_NONE) {
                CK(cudaMalloc(&b.dn, n * narrow_bytes(ctx, i)));
                CK(cudaHostAlloc(&b.hn, n * narrow_bytes(ctx, i), cudaHostAllocDefault));
            } else if (p.host_output == VGL_HOST_I32 || p.host_output == VGL_HOST_NARROW) {
                CK(cudaHostAlloc(&b.h, n * 4, cudaHostAllocDefault));
            }
        }
        if (p.host_output == VGL_HOST_BCF || p.host_output == VGL_HOST_BGZF) {
            const bool bgzf = p.host_output == VGL_HOST_BGZF;
            // worst case per record: every integer tag at the widest type its values can need (PL <= 255 -> int16; depths
            // bounded by 255 reads under the alias-table law -> int16, else int32) + literals + the pass-through bytes
            const size_t wc = ctx->plan.alias_ok ? 2 : 4, per_site_blob = p.bcf_blob_bytes_per_site ? (size_t)p.bcf_blob_bytes_per_site : 16;
            const size_t per_cell = ((t & VGL_TAG_FMT_DP) ? wc : 0) + ((t & VGL_TAG_GL) ? 60 : 0) + ((t & VGL_TAG_GP) ? 60 : 0) +
                                    ((t & VGL_TAG_PL) ? 30 : 0) + 5 * wc * (!!(t & VGL_TAG_FMT_AD) + !!(t & VGL_TAG_FMT_ADF) + !!(t & VGL_TAG_FMT_ADR));
            ctx->bcf_cap = ((cells * per_cell + B * (512 + per_site_blob)) + 15) & ~(size_t)15;
            ctx->blob_cap = B * per_site_blob;
            CK(cudaHostAlloc((void**)&s.h_bcf_in, B * sizeof(vgl_bcf_site_in), cudaHostAllocDefault));
            CK(cudaHostAlloc((void**)&s.h_blob, ctx->blob_cap, cudaHostAllocDefault));
            ctx->bcf_headroom = (!bgzf && p.do_gvcf) ? (((size_t)4096 + 16 * S + 15) & ~(size_t)15) : 0;
            if (!bgzf) CK(cudaHostAlloc((void**)&s.h_bcf, ctx->bcf_cap + ctx->bcf_headroom, cudaHostAllocDefault));
            else { // the record stream stays on the device; the host receives the compressed blocks
                ctx->bgzf_max_blocks = bgzf_blocks_for((int64_t)ctx->bcf_cap);
                const size_t worst = (size_t)ctx->bgzf_max_blocks * BGZF_STRIDE;
                CK(cudaMalloc((void**)&s.d_planes, B * sizeof(BcfRecPlanes)));
                CK(cudaMalloc((void**)&s.d_stage, worst));
                CK(cudaMalloc((void**)&s.d_bgzf, worst));
                CK(cudaHostAlloc((void**)&s.h_bgzf, worst, cudaHostAllocDefault));
                CK(cudaMalloc((void**)&s.d_blk_size, (size_t)ctx->bgzf_max_blocks * sizeof(uint32_t)));
                CK(cudaMalloc((void**)&s.d_blk_off, (size_t)ctx->bgzf_max_blocks * sizeof(long long)));
                CK(cudaMalloc((void**)&s.d_blk_first, (size_t)ctx->bgzf_max_blocks * sizeof(int32_t)));
                CK(cudaMalloc((void**)&s.d_blk_rng, (size_t)ctx->bgzf_max_blocks * BGZF_RNG_WORDS * sizeof(uint32_t)));
                if (!ctx->d_bgzf_code) {
                    std::vector<BgzfCode> codes(1);
                    bgzf_build_code(nullptr, true, &codes[0]);
                    CK(upload(&ctx->d_bgzf_code, codes));
                    CK(cudaMalloc((void**)&ctx->d_bgzf_hist, BGZF_HIST * sizeof(uint32_t)));
                    ctx->bgzf_code_ready = getenv("VGL_BGZF_FIXED") != nullptr; // development: keep the fixed code
                }
                if (!ctx->d_crc_pow) {
                    std::vector<uint32_t> pw(2048);
                    bgzf_crc_pow_table(pw.data());
                    CK(upload(&ctx->d_crc_pow, pw));
                }
            }
            CK(cudaHostAlloc((void**)&s.h_rec_off, (B + 1) * sizeof(long long), cudaHostAllocDefault));
            memset(s.h_bcf_in, 0, B * sizeof(vgl_bcf_site_in));
            CK(cudaMalloc((void**)&s.d_bcf_in, B * sizeof(vgl_bcf_site_in)));
            CK(cudaMalloc((void**)&s.d_blob, ctx->blob_cap));
            CK(cudaMalloc((void**)&s.d_bcf, ctx->bcf_cap));
            CK(cudaMalloc((void**)&s.d_minmax, B * sizeof(BcfSiteMinMax)));
            CK(cudaMalloc((void**)&s.d_rec_len, B * sizeof(uint32_t)));
            CK(cudaMalloc((void**)&s.d_rec_off, (B + 1) * sizeof(long long)));
        }
    }
    return VGL_OK;
}

extern "C" int vgl_create(const vgl_params* params, vgl_ctx** out)
{
    if (!params || !out) return VGL_EINVAL;
    *out = nullptr;
    std::string why;
    const int v = validate(params, why);
    if (v != VGL_OK) {
        fprintf(stderr, "[vgl] invalid parameters: %s\n", why.c_str());
        return v;
    }
    vgl_ctx* ctx = new (std::nothrow) vgl_ctx();
    if (!ctx) return VGL_ENOMEM;
    ctx->prm = *params;
    if (params->depth_mode == VGL_DEPTH_POISSON_PER_SAMPLE) {
        ctx->depth_means.assign(params->depth_means, params->depth_means + params->n_samples);
        for (double d : ctx->depth_means)
            if (!(d >= 0.0 && d <= 500.0)) {
                delete ctx;
                return VGL_EINVAL;
            }
    }
    ctx->prm.depth_means = nullptr;
    const int rc = create_impl(ctx);
    if (rc != VGL_OK) {
        fprintf(stderr, "[vgl] vgl_create failed: %s (%s)\n", vgl_strerror(rc), ctx->err.c_str());
        vgl_destroy(ctx);
        return rc;
    }
    *out = ctx;
    return VGL_OK;
}

extern "C" int vgl_input_buffer(vgl_ctx* ctx, int slot, uint8_t** gt, int64_t* capacity_sites)
{
    if (!ctx || slot < 0 || slot >= (int)ctx->slots.size()) return VGL_EINVAL;
    if (gt) *gt = ctx->slots[slot].h_gt;
    if (capacity_sites) *capacity_sites = ctx->prm.max_batch_sites;
    return VGL_OK;
}

extern "C" int vgl_bcf_input_buffer(vgl_ctx* ctx, int slot, vgl_bcf_site_in** sites, uint8_t** blob, int64_t* blob_capacity)
{
    if (!ctx || slot < 0 || slot >= (int)ctx->slots.size()) return VGL_EINVAL;
    if (ctx->prm.host_output != VGL_HOST_BCF && ctx->prm.host_output != VGL_HOST_BGZF) return fail(ctx, VGL_ESTATE, "vgl_bcf_input_buffer: the context was not created with VGL_HOST_BCF");
    if (sites) *sites = ctx->slots[slot].h_bcf_in;
    if (blob) *blob = ctx->slots[slot].h_blob;
    if (blob_capacity) *blob_capacity = (int64_t)ctx->blob_cap;
    return VGL_OK;
}

extern "C" int vgl_set_stream(vgl_ctx* ctx, int slot, void* cuda_stream)
{
    if (!ctx || slot < 0 || slot >= (int)ctx->slots.size()) return VGL_EINVAL;
    Slot& s = ctx->slots[slot];
    if (s.submitted && !s.waited) return VGL_ESTATE;
    s.stream = cuda_stream ? (cudaStream_t)cuda_stream : s.own_stream;
    return VGL_OK;
}

// ---- discordance summary (discord.cu) ----
extern "C" int vgl_discordance(vgl_ctx* ctx, int slot, vgl_discordance_out* out)
{
    if (!ctx || !out || slot < 0 || slot >= (int)ctx->slots.size()) return VGL_EINVAL;
    const vgl_params& prm = ctx->prm;
    Slot& s = ctx->slots[slot];
    if (!s.submitted || !s.waited) return fail(ctx, VGL_ESTATE, "vgl_discordance: call vgl_wait on the slot first");
    if (!s.plane[P_GL].d || !(prm.tag_mask & VGL_TAG_FMT_DP) || prm.depth_mode == VGL_DEPTH_INF)
        return fail(ctx, VGL_EINVAL, "vgl_discordance: needs the GL tag and FORMAT/DP of a simulated batch");
    CK(cudaSetDevice(prm.device_id));
    cudaStream_t st = s.stream;
    if (!s.g_ev[0]) for (auto& e : s.g_ev) CK(cudaEventCreate(&e));
    if (!s.d_disc) {
        CK(cudaMalloc((void**)&s.d_disc, 4 * sizeof(unsigned long long)));
        CK(cudaHostAlloc((void**)&s.h_disc, 4 * sizeof(unsigned long long), cudaHostAllocDefault));
    }
    CK(cudaMemsetAsync(s.d_disc, 0, 4 * sizeof(unsigned long long), st));
    CK(cudaEventRecord(s.g_ev[0], st));
    launch_discordance(s.d_sites, s.d_gt, s.dev(P_DP), s.dev<float>(P_GL), prm.n_samples, s.n_sites, s.d_disc, st, ctx->n_sms);
    ctx->launches += 1;
    CK(cudaGetLastError());
    CK(cudaEventRecord(s.g_ev[1], st));
    CK(cudaMemcpyAsync(s.h_disc, s.d_disc, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    out->n_hom = (int64_t)s.h_disc[0], out->n_hom_discordant = (int64_t)s.h_disc[1];
    out->n_het = (int64_t)s.h_disc[2], out->n_het_discordant = (int64_t)s.h_disc[3];
    cudaEventElapsedTime(&out->ms_kernel, s.g_ev[0], s.g_ev[1]);
    return VGL_OK;
}

static int ensure_gvcf_buffers(vgl_ctx* ctx, Slot& s)
{
    if (s.g_sin) return VGL_OK;
    const size_t B = (size_t)ctx->prm.max_batch_sites, S = (size_t)ctx->prm.n_samples;
    CK(cudaMalloc((void**)&s.g_sin, B * sizeof(vgl_gvcf_site_in)));
    CK(cudaMalloc((void**)&s.g_key, B * sizeof(int2)));
    CK(cudaMalloc((void**)&s.g_recs, B * sizeof(vgl_gvcf_rec)));
    CK(cudaHostAlloc((void**)&s.hg_recs, B * sizeof(vgl_gvcf_rec), cudaHostAllocDefault));
    CK(cudaMalloc((void**)&s.g_prev, B * sizeof(int32_t)));
    CK(cudaMalloc((void**)&s.g_kidx, B * sizeof(int32_t)));
    CK(cudaMalloc((void**)&s.g_counts, 4 * sizeof(int32_t)));
    CK(cudaMalloc((void**)&s.g_blast, B * sizeof(int32_t))); // block ordinal -> record
    CK(cudaMalloc((void**)&s.g_bsum, (B / 1024 + 2) * sizeof(unsigned long long)));
    CK(cudaMalloc((void**)&s.g_local, B * sizeof(unsigned long long)));
    CK(cudaHostAlloc((void**)&s.hg_counts, 4 * sizeof(int32_t), cudaHostAllocDefault));
    CK(cudaMalloc((void**)&s.g_dp, B * S * sizeof(int32_t)));
    CK(cudaHostAlloc((void**)&s.hg_dp, B * S * sizeof(int32_t), cudaHostAllocDefault));
    if (s.plane[P_PL].d) {
        CK(cudaMalloc((void**)&s.g_pl, B * S * 3 * sizeof(int32_t)));
        CK(cudaHostAlloc((void**)&s.hg_pl, B * S * 3 * sizeof(int32_t), cudaHostAllocDefault));
    }
    return VGL_OK;
}

// ---- gVCF block merger (gvcf.cu) ----
static GvcfArgs gvcf_args(const vgl_ctx* ctx, const Slot& s, int32_t n_sites, const int32_t* gvcf_dps, int32_t n_gvcf_dps)
{
    GvcfArgs a;
    memset(&a, 0, sizeof a);
    a.S = ctx->prm.n_samples, a.n_sites = n_sites;
    a.dps.n = n_gvcf_dps;
    for (int i = 0; i < n_gvcf_dps; ++i) a.dps.v[i] = gvcf_dps[i];
    a.sites = s.d_sites, a.dp = s.dev(P_DP), a.pl = s.dev(P_PL), a.sin = s.g_sin, a.key = s.g_key, a.recs = s.g_recs;
    a.prev_kept = s.g_prev, a.kept_idx = s.g_kidx, a.counts = s.g_counts, a.out_dp = s.g_dp, a.out_pl = s.g_pl;
    a.blk_rec = s.g_blast, a.local = s.g_local, a.block_sum = s.g_bsum;
    return a;
}

extern "C" int vgl_gvcf_merge(vgl_ctx* ctx, int slot, const vgl_gvcf_site_in* sites, const int32_t* gvcf_dps, int32_t n_gvcf_dps, vgl_gvcf_out* out)
{
    if (!ctx || !sites || !gvcf_dps || !out || slot < 0 || slot >= (int)ctx->slots.size()) return VGL_EINVAL;
    const vgl_params& prm = ctx->prm;
    if (n_gvcf_dps < 1 || n_gvcf_dps > VGL_MAX_GVCF_DPS) return fail(ctx, VGL_EINVAL, "vgl_gvcf_merge: 1..16 --gvcf-dps thresholds");
    for (int i = 0; i < n_gvcf_dps; ++i)
        if (gvcf_dps[i] < 1 || (i && gvcf_dps[i] <= gvcf_dps[i - 1])) return fail(ctx, VGL_EINVAL, "vgl_gvcf_merge: --gvcf-dps must be >= 1 and ascending");
    if (prm.do_unobserved != 1 && prm.do_unobserved != 2) return fail(ctx, VGL_EINVAL, "vgl_gvcf_merge: needs -doUnobserved 1 or 2 (block members carry REF + one unobserved allele)");
    if (!(prm.tag_mask & VGL_TAG_FMT_DP) || prm.host_output == VGL_HOST_BCF) return fail(ctx, VGL_EINVAL, "vgl_gvcf_merge: needs FORMAT/DP and the tag planes on the device");
    Slot& s = ctx->slots[slot];
    if (!s.submitted || !s.waited) return fail(ctx, VGL_ESTATE, "vgl_gvcf_merge: call vgl_wait on the slot first");
    if (s.n_sites >= (1 << 21)) return fail(ctx, VGL_EINVAL, "vgl_gvcf_merge: at most 2^21 - 1 sites per batch");
    CK(cudaSetDevice(prm.device_id));
    const size_t S = (size_t)prm.n_samples;
    { const int rc = ensure_gvcf_buffers(ctx, s); if (rc != VGL_OK) return rc; }
    if (!s.g_ev[0]) for (auto& e : s.g_ev) CK(cudaEventCreate(&e));
    cudaStream_t st = s.stream;
    const int32_t n = s.n_sites;
    CK(cudaMemcpyAsync(s.g_sin, sites, (size_t)n * sizeof(vgl_gvcf_site_in), cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(s.g_ev[0], st));
    launch_gvcf(gvcf_args(ctx, s, n, gvcf_dps, n_gvcf_dps), st, ctx->n_sms);
    ctx->launches += 5;
    CK(cudaGetLastError());
    CK(cudaEventRecord(s.g_ev[1], st));
    CK(cudaMemcpyAsync(s.hg_counts, s.g_counts, 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const int32_t n_recs = s.hg_counts[0], n_blocks = s.hg_counts[1];
    if (n_recs) CK(cudaMemcpyAsync(s.hg_recs, s.g_recs, (size_t)n_recs * sizeof(vgl_gvcf_rec), cudaMemcpyDeviceToHost, st));
    if (n_blocks) {
        CK(cudaMemcpyAsync(s.hg_dp, s.g_dp, (size_t)n_blocks * S * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        if (s.g_pl) CK(cudaMemcpyAsync(s.hg_pl, s.g_pl, (size_t)n_blocks * S * 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    memset(out, 0, sizeof *out);
    out->n_recs = n_recs, out->n_blocks = n_blocks;
    out->recs = s.hg_recs, out->dp = s.hg_dp, out->pl = s.g_pl ? s.hg_pl : nullptr;
    cudaEventElapsedTime(&out->ms_kernels, s.g_ev[0], s.g_ev[1]);
    return VGL_OK;
}

// ---- input path (vcfin.cu) ----
extern "C" int vgl_parser_create(vgl_ctx* ctx, int64_t max_text_bytes, int32_t max_records, vgl_parser** out)
{
    if (!ctx || !out) return VGL_EINVAL;
    const int rc = parser_create(ctx->prm.device_id, ctx->prm.n_samples, ctx->prm.rm_invar_sites, ctx->n_sms, max_text_bytes, max_records, out, ctx->err);
    return rc;
}

extern "C" int vgl_place_rows(vgl_ctx* ctx, int slot, vgl_parser* ps, const int32_t* row_map, int32_t first_record, int32_t n_sites, uint8_t fill_gt)
{
    if (!ctx || !ps || slot < 0 || slot >= (int)ctx->slots.size()) return VGL_EINVAL;
    if (ps->S != ctx->prm.n_samples || ps->device != ctx->prm.device_id) return fail(ctx, VGL_EINVAL, "vgl_place_rows: parser belongs to another context geometry");
    if (n_sites < 1 || n_sites > ctx->prm.max_batch_sites) return fail(ctx, VGL_EINVAL, "vgl_place_rows: n_sites out of range");
    Slot& s = ctx->slots[slot];
    if (s.submitted && !s.waited) return fail(ctx, VGL_ESTATE, "slot still in flight: call vgl_wait first");
    if (row_map) {
        if (n_sites > ps->max_records) return fail(ctx, VGL_EINVAL, "vgl_place_rows: a row map holds at most the parser's max_records entries");
        for (int32_t i = 0; i < n_sites; ++i)
            if (row_map[i] >= ps->n_records) return fail(ctx, VGL_EINVAL, "vgl_place_rows: row_map entry beyond the parsed records");
    } else if (first_record < 0 || first_record + n_sites > ps->n_records)
        return fail(ctx, VGL_EINVAL, "vgl_place_rows: record range beyond the parsed records");
    CK(cudaSetDevice(ctx->prm.device_id));
    cudaStream_t st = s.stream;
    CK(cudaStreamWaitEvent(st, ps->ev_done, 0));
    if (ps->placed) CK(cudaStreamWaitEvent(st, ps->ev_placed, 0)); // the shared row-map buffer may still be read by the previous placement
    const int32_t* d_map = nullptr;
    if (row_map) {
        CK(cudaMemcpyAsync(ps->d_row_map, row_map, (size_t)n_sites * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st)); // row_map is the caller's (pageable) memory
        d_map = ps->d_row_map;
    }
    launch_place_rows(ps->d_rows, d_map, first_record, n_sites, ctx->prm.n_samples, fill_gt, s.d_gt, st, ctx->n_sms);
    ctx->launches += 1;
    CK(cudaGetLastError());
    CK(cudaEventRecord(ps->ev_placed, st));
    ps->placed = true;
    return VGL_OK;
}

template <typename T>
static int stage_replay(vgl_ctx* ctx, DevBuf& b, const T* h, size_t n, cudaStream_t st, const T** d_out)
{
    *d_out = nullptr;
    if (!h || n == 0) return VGL_OK;
    const size_t bytes = n * sizeof(T);
    if (b.cap < bytes) {
        CK(cudaStreamSynchronize(st));
        cudaFree(b.p);
        b.p = nullptr;
        b.cap = 0;
        CK(cudaMalloc(&b.p, bytes));
        b.cap = bytes;
    }
    CK(cudaMemcpyAsync(b.p, h, bytes, cudaMemcpyHostToDevice, st));
    *d_out = (const T*)b.p;
    return VGL_OK;
}

static void fill_params(const vgl_ctx* ctx, const Slot& s, int64_t first_site_id, int32_t n_sites, DevParams& p)
{
    const vgl_params& prm = ctx->prm;
    const int64_t S = prm.n_samples, cells = (int64_t)n_sites * S;
    memset(&p, 0, sizeof p);
    p.S = (int32_t)S;
    p.n_sites = n_sites;
    p.first_site = first_site_id;
    p.n_cells = cells;
    p.k0 = (uint32_t)((uint64_t)prm.seed & 0xFFFFFFFFu);
    p.k1 = (uint32_t)((uint64_t)prm.seed >> 32);
    for (int r = 0; r < 10; ++r) {
        p.rk[2 * r] = p.k0 + (uint32_t)r * 0x9E3779B9u;
        p.rk[2 * r + 1] = p.k1 + (uint32_t)r * 0xBB67AE85u;
    }
    p.depth_mode = prm.depth_mode;
    p.depth_mean = prm.depth_mean;
    p.depth_means = ctx->d_depth_means;
    p.error_rate = prm.error_rate;
    p.error_qs = prm.error_qs;
    p.beta_a = ctx->plan.beta_a;
    p.beta_b = ctx->plan.beta_b;
    p.gl_mode = ctx->plan.gl_mode;
    p.adjust_qs = prm.adjust_qs;
    p.adjust_by = prm.adjust_by;
    p.use_bins = prm.n_qs_bins > 0;
    p.bin_max = ctx->plan.bin_max;
    memcpy(p.bin_lut, ctx->plan.bin_lut, 256);
    p.do_unobserved = prm.do_unobserved;
    p.rm_invar_sim = (prm.rm_invar_sites & 4) != 0;
    p.rm_empty = prm.rm_empty_sites != 0;
    p.do_gvcf = prm.do_gvcf != 0;
    p.tag_mask = prm.tag_mask;
    p.i16_mapq = prm.i16_mapq;
    p.pre_qs = ctx->plan.pre.qs;
    p.pre_adj_qs = ctx->plan.pre.adj_qs;
    p.homT = ctx->plan.pre.homT;
    p.het = ctx->plan.pre.het;
    p.homF = ctx->plan.pre.homF;
    p.sample_strand = ctx->plan.sample_strand;
    p.need_cellq = ctx->plan.need_cellq;
    p.need_tail = ctx->plan.need_tail;
    p.fast_div = ctx->plan.fast_div;
    p.zero_holes = prm.host_output == VGL_HOST_I32 || prm.host_output == VGL_HOST_NARROW;
    p.lut_log10 = ctx->d_lut;
    p.m1_bsum = ctx->d_m1_bsum;
    p.m1_het = ctx->d_m1_het;
    p.em_fk = ctx->d_fk;
    p.em_beta = ctx->d_beta;
    p.gt = s.d_gt;
    p.dp = s.dev(P_DP);
    p.cell = s.d_cell;
    p.cellq = s.d_cellq;
    p.celltail = s.d_celltail;
    p.sites = s.d_sites;
    p.totals = s.d_totals;
    p.totals_host = s.h_totals; // pinned + mapped (UVA): the tile kernel also posts the totals there, sparing the tiny D2H copy
    p.pairmap = s.d_pairmap;
    p.pois_cdf = ctx->d_pois;
    p.pois_n = ctx->pois_n;
    p.pois_alias = ctx->d_alias;
    p.alias_row = ctx->d_alias_row;
    p.err_cdf = ctx->d_errcdf;
    p.cnt_scratch = ctx->d_cnt_scratch;
    p.m1_pure = ctx->d_m1_pure;
    p.qcls = ctx->d_qcls;
    p.m2_tab = ctx->d_m2_tab;
    p.m2_nq = ctx->plan.m2_nq;
    p.m2_cmap = ctx->d_m2_cmap;
    p.qm_cdf = ctx->d_qm_cdf;
    p.q_minor = ctx->plan.q_minor;
    p.q_dom = ctx->plan.q_dom;
    p.q_dom_idx = ctx->plan.q_dom_idx;
    p.m2_pure = ctx->d_m2_pure;
    p.m2_park = ctx->d_m2_park;
    {
        int T = 1024 / (int)S;
        T = T < 1 ? 1 : (T > 128 ? 128 : T);
        const bool tile = ctx->plan.set == KS_TILE_M1F || ctx->plan.set == KS_TILE_M2;
        if (tile) T = tile_m1f_sites_per_tile((int)S);
        p.sites_per_tile = T;
        p.n_tiles = (n_sites + T - 1) / T;
        p.tile_state = s.d_tile_state;
        p.ticket = s.d_tile_state ? reinterpret_cast<uint32_t*>(s.d_tile_state + (tile ? 0 : p.n_tiles)) : nullptr;
    }
    p.status = reinterpret_cast<int32_t*>(s.d_totals + 2);
    p.gl = s.dev<float>(P_GL); p.pl = s.dev(P_PL); p.gp = s.dev<float>(P_GP);
    p.ad = s.dev(P_AD); p.adf = s.dev(P_ADF); p.adr = s.dev(P_ADR);
}

extern "C" int vgl_set_gvcf_dps(vgl_ctx* ctx, const int32_t* gvcf_dps, int32_t n)
{
    if (!ctx || !gvcf_dps || n < 1 || n > VGL_MAX_GVCF_DPS) return VGL_EINVAL;
    for (int i = 0; i < n; ++i)
        if (gvcf_dps[i] < 1 || (i && gvcf_dps[i] <= gvcf_dps[i - 1])) return fail(ctx, VGL_EINVAL, "vgl_set_gvcf_dps: --gvcf-dps must be >= 1 and ascending");
    ctx->gvcf_dps.assign(gvcf_dps, gvcf_dps + n);
    return VGL_OK;
}

// ---- host-side encoding of ONE gVCF block record: only the block that straddles two batches is encoded here (its halves were
// reduced on the device); same bytes as bcf_layout_block() in bcf.cu / GVCF_FLUSH_BLOCK in bcf_utils.cpp:896-925
namespace {
struct ByteOut {
    std::vector<uint8_t>& v;
    void put(uint8_t b) { v.push_back(b); }
    void put16(uint32_t x) { put((uint8_t)x); put((uint8_t)(x >> 8)); }
    void put32(uint32_t x) { put16(x); put16(x >> 16); }
    void size(int n, int type)
    {
        if (n >= 15) {
            put((uint8_t)(15 << 4 | type));
            if (n >= 128) {
                if (n >= 32768) { put(1 << 4 | 3); put32((uint32_t)n); }
                else { put(1 << 4 | 2); put16((uint32_t)n); }
            } else { put(1 << 4 | 1); put((uint8_t)n); }
        } else put((uint8_t)(n << 4 | type));
    }
    void int1(int32_t x)
    {
        if (x == VGL_I32_MISSING) { size(1, 1); put(0x80); }
        else if (x == VGL_I32_MISSING + 1) { size(1, 1); put(0x81); }
        else if (x <= 127 && x >= -120) { size(1, 1); put((uint8_t)x); }
        else if (x <= 32767 && x >= -32760) { size(1, 2); put16((uint32_t)x); }
        else { size(1, 3); put32((uint32_t)x); }
    }
    void vint(const int32_t* a, size_t n, int nps)
    {
        int32_t mx = INT32_MIN, mn = INT32_MAX;
        for (size_t i = 0; i < n; ++i) {
            if (a[i] == VGL_I32_MISSING || a[i] == VGL_I32_MISSING + 1) continue;
            mx = std::max(mx, a[i]);
            mn = std::min(mn, a[i]);
        }
        const int t = (mx <= 127 && mn >= -120) ? 1 : ((mx <= 32767 && mn >= -32760) ? 2 : 3);
        size(nps, t);
        for (size_t i = 0; i < n; ++i) {
            const int32_t x = a[i];
            if (t == 1) put(x == VGL_I32_MISSING ? 0x80 : (x == VGL_I32_MISSING + 1 ? 0x81 : (uint8_t)x));
            else if (t == 2) put16(x == VGL_I32_MISSING ? 0x8000u : (x == VGL_I32_MISSING + 1 ? 0x8001u : (uint32_t)x));
            else put32((uint32_t)x);
        }
    }
};
} // namespace

static void encode_gvcf_block(const vgl_ctx* ctx, const vgl_ctx::Carry& c, std::vector<uint8_t>& out)
{
    const vgl_params& prm = ctx->prm;
    const int S = prm.n_samples;
    out.clear();
    ByteOut b{out};
    const int32_t end1 = c.end + 1;
    const bool has_end = end1 - c.start >= 2, has_qs = (prm.tag_mask & VGL_TAG_QS) != 0, has_pl = !c.pl.empty();
    b.put32(0); b.put32(0);
    b.put32((uint32_t)c.rid);
    b.put32((uint32_t)c.start);
    b.put32((uint32_t)(end1 - c.start));
    b.put32(VGL_F32_MISSING_BITS);
    b.put16((uint32_t)((has_end ? 1 : 0) + 1 + (has_qs ? 1 : 0)));
    b.put16((uint32_t)c.n_alleles);
    b.put32(((uint32_t)((has_pl ? 1 : 0) + 1) << 24) | ((uint32_t)S & 0xFFFFFFu));
    b.put(0x07);
    const bool nonref_name = prm.do_unobserved == 2 || prm.do_unobserved == 5;
    for (int k = 0; k < c.n_alleles; ++k) {
        const int code = c.a2b[k];
        const char* str = code == 4 ? (nonref_name ? "<NON_REF>" : "<*>") : (code == 0 ? "A" : code == 1 ? "C" : code == 2 ? "G" : "T");
        const int n = (int)strlen(str);
        b.size(n, 7);
        for (int i = 0; i < n; ++i) b.put((uint8_t)str[i]);
    }
    b.put(0x00);
    if (has_end) { b.int1(prm.bcf_dict.end); b.int1(end1); }
    b.int1(prm.bcf_dict.min_dp); b.int1(c.min_dp);
    if (has_qs) {
        b.int1(prm.bcf_dict.qs);
        b.size(c.n_alleles, 5);
        for (int k = 0; k < c.n_alleles; ++k) { uint32_t u; memcpy(&u, &c.qs[k], 4); b.put32(u); }
    }
    const uint32_t l_shared = (uint32_t)out.size() - 8;
    if (has_pl) { b.int1(prm.bcf_dict.pl); b.vint(c.pl.data(), c.pl.size(), 3); }
    b.int1(prm.bcf_dict.dp); b.vint(c.dp.data(), c.dp.size(), 1);
    const uint32_t l_indiv = (uint32_t)out.size() - 8 - l_shared;
    memcpy(out.data(), &l_shared, 4);
    memcpy(out.data() + 4, &l_indiv, 4);
}

extern "C" int vgl_gvcf_flush(vgl_ctx* ctx, const uint8_t** rec, int64_t* n_bytes)
{
    if (!ctx || !rec || !n_bytes) return VGL_EINVAL;
    *rec = nullptr;
    *n_bytes = 0;
    if (ctx->carry.open) {
        ctx->flush_rec = ctx->carry.rec;
        ctx->carry.open = false;
        *rec = ctx->flush_rec.data();
        *n_bytes = (int64_t)ctx->flush_rec.size();
    }
    return VGL_OK;
}

// Copy of n elements of plane i to the host, narrowed when VGL_HOST_NARROW narrows it (nothing when the host has no copy of it)
static cudaError_t d2h_plane(const vgl_ctx* ctx, const Slot& s, int i, size_t n)
{
    const PlaneBufs& b = s.plane[i];
    if (b.hn) return cudaMemcpyAsync(b.hn, b.dn, n * narrow_bytes(ctx, i), cudaMemcpyDeviceToHost, s.stream);
    return b.h ? cudaMemcpyAsync(b.h, b.d, n * 4, cudaMemcpyDeviceToHost, s.stream) : cudaSuccess;
}

// The copies of every plane but DP (it goes with the site records): g / r elements of the G- / R-shaped planes
static cudaError_t d2h_planes(const vgl_ctx* ctx, const Slot& s, size_t g, size_t r)
{
    for (int i = P_DP + 1; i < P_COUNT; ++i) {
        const cudaError_t e = d2h_plane(ctx, s, i, plane_elems(i, 0, g, r));
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// The result copies of a batch whose extents (plane elements, record bytes, compressed bytes) are only known once its kernels
// have run: enqueued on the slot's stream as soon as some API call finds the totals on the host.
static int issue_d2h(vgl_ctx* ctx, Slot& s)
{
    const vgl_params& prm = ctx->prm;
    cudaStream_t st = s.stream;
    CK(cudaEventRecord(s.ev[EV_D2H0], st));
    if (prm.host_output == VGL_HOST_BCF || prm.host_output == VGL_HOST_BGZF) {
        const bool z = prm.host_output == VGL_HOST_BGZF;
        const int64_t nb = s.h_totals[z ? 4 : 3], cap = z ? ctx->bgzf_max_blocks * (int64_t)BGZF_STRIDE : (int64_t)ctx->bcf_cap;
        const int64_t done = s.stream_copied; // what vgl_submit copied on its prediction
        if (nb > done && nb <= cap)
            CK(cudaMemcpyAsync((z ? s.h_bgzf : s.h_bcf + ctx->bcf_headroom) + done, (z ? s.d_bgzf : s.d_bcf) + done, (size_t)(nb - done), cudaMemcpyDeviceToHost, st));
        if (prm.do_gvcf && !z) { // the merger's record list and the per-sample minima of the first and the last record (the seam)
            const int32_t n_recs = s.hg_counts[0];
            if (n_recs > 0) {
                CK(cudaMemcpyAsync(s.hg_recs, s.g_recs, (size_t)n_recs * sizeof(vgl_gvcf_rec), cudaMemcpyDeviceToHost, st));
                CK(cudaStreamSynchronize(st)); // the planes to fetch depend on the records
                const size_t S = (size_t)prm.n_samples;
                for (int k : {0, n_recs - 1}) {
                    const vgl_gvcf_rec& r = s.hg_recs[k];
                    if (r.n_members == 0) continue;
                    CK(cudaMemcpyAsync(s.hg_dp + (size_t)r.plane * S, s.g_dp + (size_t)r.plane * S, S * 4, cudaMemcpyDeviceToHost, st));
                    if (s.g_pl) CK(cudaMemcpyAsync(s.hg_pl + (size_t)r.plane * S * 3, s.g_pl + (size_t)r.plane * S * 3, S * 12, cudaMemcpyDeviceToHost, st));
                }
            }
        }
        if (nb > 0 && s.n_sites > 0) ctx->stream_bytes_per_site = (double)nb / s.n_sites;
    } else
        CK(d2h_planes(ctx, s, (size_t)s.h_totals[0], (size_t)s.h_totals[1]));
    CK(cudaEventRecord(s.ev[EV_D2H1], st));
    s.early_d2h = true;
    return VGL_OK;
}

// every submit / wait looks at the other slots in flight: a batch whose kernels have finished gets its result copies enqueued
// right away, so that they run under the host's work on other slots instead of inside that slot's vgl_wait
static void progress(vgl_ctx* ctx)
{
    if (!ctx->prm.host_output) return;
    for (Slot& s : ctx->slots)
        if (s.submitted && !s.waited && !s.early_d2h && cudaEventQuery(s.ev[EV_META]) == cudaSuccess) issue_d2h(ctx, s);
}

extern "C" int vgl_submit(vgl_ctx* ctx, int slot, int64_t first_site_id, int32_t n_sites, const vgl_replay* rp, uint32_t flags)
{
    if (!ctx || slot < 0 || slot >= (int)ctx->slots.size()) return VGL_EINVAL;
    if (n_sites < 1 || n_sites > ctx->prm.max_batch_sites || first_site_id < 0) return fail(ctx, VGL_EINVAL, "n_sites / first_site_id out of range");
    Slot& s = ctx->slots[slot];
    if (s.submitted && !s.waited) return fail(ctx, VGL_ESTATE, "slot still in flight: call vgl_wait first");
    const vgl_params& prm = ctx->prm;
    if (prm.host_output == VGL_HOST_BCF || prm.host_output == VGL_HOST_BGZF) { // the input records, before anything is copied or launched
        const int64_t S = prm.n_samples;
        for (int32_t i = 0; i < n_sites; ++i) { // byte ranges must lie inside the blob
            const vgl_bcf_site_in& b = s.h_bcf_in[i];
            if ((size_t)b.id_off + b.id_len > ctx->blob_cap || (size_t)b.flt_info_off + b.flt_info_len > ctx->blob_cap ||
                (size_t)b.fmt_off + b.fmt_len > ctx->blob_cap)
                return fail(ctx, VGL_EINVAL, "vgl_bcf_site_in: byte range outside the pass-through blob");
            if (b.n_fmt > 8 || (b.n_fmt == 0) != (b.fmt_len == 0)) return fail(ctx, VGL_EINVAL, "vgl_bcf_site_in: at most 8 input FORMAT blocks, n_fmt and fmt_len both zero or both set");
            if (b.n_fmt && !bcf_fmt_blocks_tile(s.h_blob + b.fmt_off, b.fmt_len, b.n_fmt, S))
                return fail(ctx, VGL_EINVAL, "vgl_bcf_site_in: the input FORMAT blocks do not tile fmt_len bytes");
        }
    }
    CK(cudaSetDevice(prm.device_id));
    progress(ctx);
    cudaStream_t st = s.stream;
    const int64_t S = prm.n_samples, cells = (int64_t)n_sites * S;

    DevParams p;
    fill_params(ctx, s, first_site_id, n_sites, p);
    CK(cudaEventRecord(s.ev[EV_START], st));
    if (!(flags & VGL_SUBMIT_GT_ON_DEVICE)) CK(cudaMemcpyAsync(s.d_gt, s.h_gt, (size_t)cells, cudaMemcpyHostToDevice, st));
    // a replayed batch runs the general kernels (--depth inf has no draws to replay)
    const KernelSet ks = rp && ctx->plan.set != KS_TRUTH ? KS_PER_READ : ctx->plan.set;
    const bool tile_launch = ks == KS_TILE_M1F || ks == KS_TILE_M2; // the tile kernel rearms its own ticket and writes the totals itself
    if (!tile_launch) CK(cudaMemsetAsync(s.d_totals, 0, 8 * sizeof(int64_t), st));
    if (rp) {
        if (!rp->depths || !rp->read_offsets || (rp->n_reads > 0 && !rp->bases)) return fail(ctx, VGL_EINVAL, "replay: depths/read_offsets/bases required");
        if (prm.error_qs == 2 && rp->n_reads > 0 && !rp->qs) return fail(ctx, VGL_EINVAL, "replay: per-read qs required with --error-qs 2");
        if (prm.error_qs == 2 && prm.adjust_qs && rp->n_reads > 0 && !rp->adj_qs) return fail(ctx, VGL_EINVAL, "replay: adjusted qs required with --adjust-qs");
        if (ctx->plan.gl_mode == GL_M2_PRECISE && rp->n_reads > 0 && !rp->error_probs) return fail(ctx, VGL_EINVAL, "replay: error_probs required with --precise-gl 1");
        if (ctx->plan.need_tail && rp->n_reads > 0 && !rp->tail_dists) return fail(ctx, VGL_EINVAL, "replay: tail_dists required with -addI16");
        if (ctx->plan.sample_strand && rp->n_reads > 0 && !rp->strands) return fail(ctx, VGL_EINVAL, "replay: strands required when the strand is sampled");
        p.replay = 1;
        int rc;
        const size_t nr = (size_t)rp->n_reads;
        if ((rc = stage_replay(ctx, s.r_depths, rp->depths, (size_t)cells, st, &p.rp_depths))) return rc;
        if ((rc = stage_replay(ctx, s.r_off, rp->read_offsets, (size_t)cells + 1, st, &p.rp_off))) return rc;
        if ((rc = stage_replay(ctx, s.r_bases, rp->bases, nr, st, &p.rp_bases))) return rc;
        if ((rc = stage_replay(ctx, s.r_strands, rp->strands, nr, st, &p.rp_strands))) return rc;
        if ((rc = stage_replay(ctx, s.r_qs, rp->qs, nr, st, &p.rp_qs))) return rc;
        if ((rc = stage_replay(ctx, s.r_adjqs, rp->adj_qs, nr, st, &p.rp_adjqs))) return rc;
        if ((rc = stage_replay(ctx, s.r_eprob, rp->error_probs, nr, st, &p.rp_eprob))) return rc;
        if ((rc = stage_replay(ctx, s.r_tails, rp->tail_dists, nr, st, &p.rp_tails))) return rc;
        // cells deeper than 255 reads under GL model 1: their ids, in cell order (input packing, not simulation)
        if (prm.gl_model == 1 && rp->n_deep_cells > 0) {
            std::vector<int64_t> deep;
            for (int64_t c = 0; c < cells; ++c) {
                const uint8_t g = s.h_gt[c];
                if ((g & 0xF) != VGL_GT_MISSING && (g >> 4) != VGL_GT_MISSING && rp->depths[c] > 255) deep.push_back(c);
            }
            if ((int64_t)deep.size() != rp->n_deep_cells) return fail(ctx, VGL_EINVAL, "replay: n_deep_cells does not match the depths");
            if ((rc = stage_replay(ctx, s.r_deep_cells, deep.data(), deep.size(), st, &p.rp_deep_cells))) return rc;
            CK(cudaStreamSynchronize(st)); // `deep` is a temporary
            if ((rc = stage_replay(ctx, s.r_deep_codes, rp->deep_codes, deep.size() * 255, st, &p.rp_deep_codes))) return rc;
            p.rp_n_deep = (int64_t)deep.size();
        }
    }
    // status word: only the model-2 tile kernel in per-read-qs mode can raise a device-side error (a quality score outside
    // the --qs-bins ranges); it goes through the device word, cleared and copied back in stream order
    const bool narrow = prm.host_output == VGL_HOST_NARROW; // the narrowing pass can raise VGL_EOVERFLOW
    const bool bgzf = prm.host_output == VGL_HOST_BGZF;
    const bool bcf = prm.host_output == VGL_HOST_BCF || bgzf; // the serialiser posts its byte total (and VGL_EOVERFLOW) in the device words
    const bool tile_status = tile_launch && ((ks == KS_TILE_M2 && prm.error_qs == 2) || narrow || bcf);
    if (bcf) {
        CK(cudaMemcpyAsync(s.d_bcf_in, s.h_bcf_in, (size_t)n_sites * sizeof(vgl_bcf_site_in), cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(s.d_blob, s.h_blob, ctx->blob_cap, cudaMemcpyHostToDevice, st));
    }
    if (tile_status) CK(cudaMemsetAsync(s.d_totals + 2, 0, sizeof(int64_t), st));
    const bool fused = one_kernel(ks);
    if (fused && !tile_launch) CK(cudaMemsetAsync(s.d_tile_state, 0, ((size_t)p.n_tiles + 1) * sizeof(unsigned long long), st));
    CK(cudaEventRecord(s.ev[EV_H2D], st));
    // Batches run their kernels strictly one after the other, also across slots with streams of their own: left to itself the
    // GPU interleaves the kernels of all batches in flight, they all finish together, and the result copies then run while
    // the SMs idle.  In order, batch k's copies overlap batch k+1's kernels.
    // The chain also holds under VGL_HOST_NONE: the tile kernels' per-CTA scratch rows (d_m2_park, d_cnt_scratch) belong to
    // the context, so two batches' kernels must never run at the same time.
    if (ctx->chain_ev) CK(cudaStreamWaitEvent(st, ctx->chain_ev, 0));
    if (fused) {
        // one kernel does everything; its time is reported as VGL_T_EMIT (SIM / SITE / SCAN = 0)
        CK(cudaEventRecord(s.ev[EV_SIM], st));
        CK(cudaEventRecord(s.ev[EV_SITE], st));
        CK(cudaEventRecord(s.ev[EV_SCAN], st));
        if (ks == KS_TILE_M1F) launch_tile_m1f(p, st, ctx->n_sms, ctx->plan.aux);
        else if (ks == KS_TILE_M2) launch_tile_m2(p, st, ctx->n_sms, prm.error_qs);
        else launch_fused_m1f(p, st, ctx->n_sms);
        CK(cudaEventRecord(s.ev[EV_EMIT], st));
        ctx->launches += 1;
    } else if (ks == KS_TRUTH) { // truth.cu: no reads, the tags state the true genotypes
        if (rp) return fail(ctx, VGL_EINVAL, "--depth inf has no draws to replay");
        CK(cudaEventRecord(s.ev[EV_SIM], st));
        launch_truth_site(p, st, ctx->n_sms);
        CK(cudaEventRecord(s.ev[EV_SITE], st));
        launch_scan(p, st);
        CK(cudaEventRecord(s.ev[EV_SCAN], st));
        launch_truth_emit(p, st, ctx->n_sms);
        CK(cudaEventRecord(s.ev[EV_EMIT], st));
        ctx->launches += 3;
    } else {
        launch_sim(p, st);
        CK(cudaEventRecord(s.ev[EV_SIM], st));
        launch_site(p, st);
        CK(cudaEventRecord(s.ev[EV_SITE], st));
        launch_scan(p, st);
        CK(cudaEventRecord(s.ev[EV_SCAN], st));
        launch_emit(p, st);
        CK(cudaEventRecord(s.ev[EV_EMIT], st));
        ctx->launches += 4;
    }
    if (narrow) { // integer planes -> narrow planes: DP over the batch's cells, the others over the used extents in d_totals
        for (int i = 0; i < P_COUNT; ++i) {
            if (!s.plane[i].dn) continue;
            const bool per_cell = kPlanes[i].shape == PER_CELL;
            const int64_t* n_dev = per_cell ? nullptr : s.d_totals + (kPlanes[i].shape == PER_ALLELE);
            launch_narrow(s.dev(i), s.plane[i].dn, (int)narrow_bytes(ctx, i) * 8, kPlanes[i].narrow == NARROW_PL, n_dev, per_cell ? cells : 0,
                          (int64_t)plane_elems(i, (size_t)cells, ctx->g_cap, ctx->r_cap), reinterpret_cast<int32_t*>(s.d_totals + 2), st, ctx->n_sms);
            ctx->launches += 1;
        }
    }
    if (bcf) { // planes -> BCF records (bcf.cu)
        BcfArgs b;
        memset(&b, 0, sizeof b);
        b.S = (int32_t)S; b.n_sites = n_sites; b.tag_mask = prm.tag_mask;
        b.do_unobserved = prm.do_unobserved; b.do_gvcf = prm.do_gvcf; b.dict = prm.bcf_dict;
        b.sites = s.d_sites; b.site_in = s.d_bcf_in; b.blob = s.d_blob;
        b.dp = s.dev(P_DP); b.gl = s.dev<float>(P_GL); b.gp = s.dev<float>(P_GP); b.pl = s.dev(P_PL);
        b.ad = s.dev(P_AD); b.adf = s.dev(P_ADF); b.adr = s.dev(P_ADR);
        b.minmax = s.d_minmax; b.rec_len = s.d_rec_len; b.rec_off = s.d_rec_off;
        b.out = s.d_bcf; b.out_cap = (long long)ctx->bcf_cap;
        b.totals = s.d_totals; b.status = reinterpret_cast<int32_t*>(s.d_totals + 2);
        b.planes = s.d_planes;
        if (prm.do_gvcf) { // the block merger first (gvcf.cu): the records to serialise are its output, blocks included
            if (ctx->gvcf_dps.empty()) return fail(ctx, VGL_ESTATE, "VGL_HOST_BCF with -doGVCF: call vgl_set_gvcf_dps before the first submit");
            if (n_sites >= (1 << 21)) return fail(ctx, VGL_EINVAL, "-doGVCF: at most 2^21 - 1 sites per batch");
            { const int rc2 = ensure_gvcf_buffers(ctx, s); if (rc2 != VGL_OK) return rc2; }
            launch_gvcf_sin_from_bcf(s.d_bcf_in, s.g_sin, n_sites, st);
            launch_gvcf(gvcf_args(ctx, s, n_sites, ctx->gvcf_dps.data(), (int32_t)ctx->gvcf_dps.size()), st, ctx->n_sms);
            ctx->launches += 6;
            b.recs = s.g_recs; b.rec_counts = s.g_counts; b.blk_dp = s.g_dp; b.blk_pl = s.g_pl;
            CK(cudaMemcpyAsync(s.hg_counts, s.g_counts, 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        }
        launch_bcf(b, st);
        ctx->launches += 3;
        CK(cudaEventRecord(s.ev[EV_BCF], st));
        if (bgzf) {
            BgzfArgs z;
            memset(&z, 0, sizeof z);
            z.S = (int32_t)S; z.n_sites = n_sites; z.in = s.d_bcf; z.in_cap = (long long)ctx->bcf_cap;
            z.rec_off = s.d_rec_off; z.planes = s.d_planes; z.crc_pow = ctx->d_crc_pow;
            z.stage = s.d_stage; z.blk_size = s.d_blk_size; z.blk_off = s.d_blk_off; z.blk_first = s.d_blk_first; z.rng_g = s.d_blk_rng; z.out = s.d_bgzf; z.totals = s.d_totals;
            // blocks this batch can make at most (its worst-case record bytes), not the slot's capacity
            const int64_t nb_max = std::min<int64_t>(ctx->bgzf_max_blocks, bgzf_blocks_for((int64_t)((double)ctx->bcf_cap * n_sites / prm.max_batch_sites) + 65536));
            z.code = ctx->d_bgzf_code;
            if (!ctx->bgzf_code_ready) {
                // once per context: the symbol statistics of this batch's parse -> a dynamic Huffman code (RFC 1951 3.2.7)
                // every later block starts with; the simulated tags have the same statistics from batch to batch
                CK(cudaMemsetAsync(ctx->d_bgzf_hist, 0, BGZF_HIST * sizeof(uint32_t), st));
                z.hist = ctx->d_bgzf_hist;
                launch_bgzf(z, nb_max, st, ctx->n_sms);
                ctx->launches += 3;
                z.hist = nullptr;
                uint32_t hist[BGZF_HIST];
                CK(cudaMemcpyAsync(hist, ctx->d_bgzf_hist, sizeof hist, cudaMemcpyDeviceToHost, st));
                CK(cudaStreamSynchronize(st));
                uint64_t seen = 0;
                for (int i = 0; i < BGZF_HIST; ++i) seen += hist[i];
                if (seen > 1000) { // else: an (almost) empty batch, try again on the next
                    BgzfCode code;
                    bgzf_build_code(hist, false, &code);
                    CK(cudaMemcpyAsync(ctx->d_bgzf_code, &code, sizeof code, cudaMemcpyHostToDevice, st));
                    CK(cudaStreamSynchronize(st));
                    ctx->bgzf_code_ready = true;
                }
            }
            launch_bgzf(z, nb_max, st, ctx->n_sms);
            ctx->launches += 5;
        }
        CK(cudaEventRecord(s.ev[EV_KDONE], st)); // the batch's last kernel: the next batch's kernels may start (its copies follow)
        ctx->chain_ev = s.ev[EV_KDONE];
        CK(cudaMemcpyAsync(s.h_rec_off, s.d_rec_off, ((size_t)n_sites + 1) * sizeof(long long), cudaMemcpyDeviceToHost, st));
        // The stream's size is only known on the device, but the previous batch predicts it well: that many bytes (+ 3 %) follow
        // the kernels right away; vgl_wait copies what is left once it knows the size (a few per cent, or nothing).
        s.stream_copied = 0;
        if (ctx->stream_bytes_per_site > 0.0) {
            const size_t cap = bgzf ? (size_t)ctx->bgzf_max_blocks * BGZF_STRIDE : ctx->bcf_cap;
            size_t pred = (size_t)(ctx->stream_bytes_per_site * n_sites * 1.03) + 65536;
            pred = std::min(pred, cap) & ~(size_t)15;
            CK(cudaEventRecord(s.ev[EV_D2H0], st));
            CK(cudaMemcpyAsync(bgzf ? s.h_bgzf : s.h_bcf + ctx->bcf_headroom, bgzf ? s.d_bgzf : s.d_bcf, pred, cudaMemcpyDeviceToHost, st));
            CK(cudaEventRecord(s.ev[EV_D2H1], st));
            s.stream_copied = (int64_t)pred;
        }
    }
    CK(cudaGetLastError());
    if (!bcf) {
        CK(cudaEventRecord(s.ev[EV_KDONE], st));
        ctx->chain_ev = s.ev[EV_KDONE];
    }
    if (prm.host_output) CK(cudaMemcpyAsync(s.h_sites, s.d_sites, (size_t)n_sites * sizeof(vgl_site_out), cudaMemcpyDeviceToHost, st));
    if (tile_launch && !tile_status) s.h_totals[2] = 0; // the kernel posts the totals into the pinned words itself and raises no errors
    else CK(cudaMemcpyAsync(s.h_totals, s.d_totals, 8 * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CK(d2h_plane(ctx, s, P_DP, (size_t)cells));
    CK(cudaEventRecord(s.ev[EV_META], st));
    s.early_d2h = false;
    if (tile_launch && (prm.host_output == VGL_HOST_I32 || narrow)) {
        // tile kernels lay tiles out at a fixed stride: the spans are n_sites x (padded 15-genotype / 5-allele block) whatever the
        // sites turn out to be (holes are zeroed, tile_zero_holes), so the plane copies queue up behind the kernels right away
        // instead of waiting for the host to come back for the totals
        const size_t g_up = (size_t)n_sites * (((size_t)S * 15 + 3) & ~(size_t)3), r_up = (size_t)n_sites * (((size_t)S * 5 + 3) & ~(size_t)3);
        CK(cudaEventRecord(s.ev[EV_D2H0], st));
        CK(d2h_planes(ctx, s, g_up, r_up));
        CK(cudaEventRecord(s.ev[EV_D2H1], st));
        s.early_d2h = true;
    }
    s.submitted = true;
    s.waited = false;
    s.n_sites = n_sites;
    s.seq = ++ctx->submit_seq;
    s.had_d2h = false;
    return VGL_OK;
}

// -doGVCF with VGL_HOST_BCF: the device serialised every record of the batch, closing every block at the batch's ends.  A block
// may run across the seam between two batches (bcf_utils.cpp:711, 719, 790: same contig, pos <= end + 1, same dp range), so the
// last record of a batch is held back when it is a block, and merged with the next batch's first record when that joins it --
// the merged record is the one piece encoded on the host (encode_gvcf_block), written into the headroom in front of the stream.
// Batches must be waited in submission order (vgl_wait rejects any other).
static void gvcf_seam(vgl_ctx* ctx, Slot& s, vgl_batch_out* out)
{
    const size_t S = (size_t)ctx->prm.n_samples;
    vgl_ctx::Carry& c = ctx->carry;
    const int32_t n_recs = s.hg_counts[0];
    uint8_t* base = s.h_bcf + ctx->bcf_headroom;
    const long long* off = s.h_rec_off;
    int64_t lo = 0, hi = n_recs > 0 ? (int64_t)off[n_recs] : 0; // bytes of the device stream that go out
    int32_t n_out = n_recs;
    std::vector<uint8_t> front; // what precedes them
    auto load = [&](const vgl_gvcf_rec& r, vgl_ctx::Carry& d) {
        const vgl_bcf_site_in &f = s.h_bcf_in[r.first_site], &l = s.h_bcf_in[r.last_site];
        const vgl_site_out& so = s.h_sites[r.first_site];
        d.open = true;
        d.rid = f.rid, d.start = f.pos, d.end = l.pos, d.range = r.dp_range, d.min_dp = r.min_dp, d.n_alleles = so.n_alleles;
        memcpy(d.a2b, so.alleles2acgt, 8);
        memcpy(d.qs, so.qs, sizeof d.qs);
        d.dp.assign(s.hg_dp + (size_t)r.plane * S, s.hg_dp + (size_t)r.plane * S + S);
        if (s.hg_pl) d.pl.assign(s.hg_pl + (size_t)r.plane * S * 3, s.hg_pl + (size_t)r.plane * S * 3 + 3 * S);
        else d.pl.clear();
    };
    bool merged_is_last = false;
    if (n_recs > 0 && c.open) {
        const vgl_gvcf_rec& r0 = s.hg_recs[0];
        const vgl_bcf_site_in& f = s.h_bcf_in[r0.first_site];
        if (r0.n_members > 0 && c.rid == f.rid && f.pos <= c.end + 1 && c.range == r0.dp_range) { // the batch's first block continues the carried one
            vgl_ctx::Carry m;
            load(r0, m);
            c.end = m.end;
            c.min_dp = std::min(c.min_dp, m.min_dp);
            for (size_t k = 0; k < S; ++k) {
                c.dp[k] = std::min(c.dp[k], m.dp[k]);
                if (!c.pl.empty() && !m.pl.empty()) {
                    int32_t* g = &c.pl[3 * k];
                    const int32_t* q = &m.pl[3 * k];
                    if (q[1] < g[1] || (q[1] == g[1] && q[2] < g[2])) g[1] = q[1], g[2] = q[2];
                }
            }
            encode_gvcf_block(ctx, c, c.rec);
            lo = (int64_t)off[1]; // the device's version of that record is dropped
            --n_out;
            if (n_recs == 1) merged_is_last = true; // still the open block
            else { front = c.rec; c.open = false; ++n_out; }
        } else {
            front = c.rec; // the carried block ended with its batch
            c.open = false;
            ++n_out;
        }
    }
    if (n_recs > 0 && !merged_is_last) {
        const vgl_gvcf_rec& rl = s.hg_recs[n_recs - 1];
        if (rl.n_members > 0 && !(n_recs == 1 && lo > 0)) { // hold the trailing block back
            load(rl, c);
            c.rec.assign(base + off[n_recs - 1], base + off[n_recs]);
            hi = (int64_t)off[n_recs - 1];
            --n_out;
        }
    }
    if (hi < lo) hi = lo;
    uint8_t* start = base + lo - (int64_t)front.size();
    if (!front.empty()) memcpy(start, front.data(), front.size()); // headroom (lo = 0) or the dropped first record's place
    s.seam_ptr = start;
    s.seam_bytes = (int64_t)front.size() + (hi - lo);
    s.seam_recs = n_out;
    out->bcf = s.seam_ptr;
    out->bcf_bytes = s.seam_bytes;
    out->bcf_off = nullptr;
    out->n_recs = s.seam_recs;
}

extern "C" int vgl_wait(vgl_ctx* ctx, int slot, vgl_batch_out* out)
{
    if (!ctx || !out || slot < 0 || slot >= (int)ctx->slots.size()) return VGL_EINVAL;
    Slot& s = ctx->slots[slot];
    if (!s.submitted) return fail(ctx, VGL_ESTATE, "slot was not submitted");
    const vgl_params& prm = ctx->prm;
    if (prm.do_gvcf && prm.host_output == VGL_HOST_BCF && !s.waited) // the seam carries a block from one batch into the next
        for (const Slot& o : ctx->slots)
            if (o.submitted && !o.waited && o.seq < s.seq) return fail(ctx, VGL_ESTATE, "-doGVCF: wait for the batches in the order they were submitted");
    CK(cudaSetDevice(prm.device_id));
    // waiting polls, so that the other slots' result copies get enqueued the moment their kernels finish (progress())
    auto wait_event = [&](cudaEvent_t ev) -> cudaError_t {
        if (!prm.host_output || ctx->slots.size() == 1) return cudaEventSynchronize(ev);
        for (;;) {
            const cudaError_t e = cudaEventQuery(ev);
            if (e != cudaErrorNotReady) return e;
            progress(ctx);
            std::this_thread::sleep_for(std::chrono::microseconds(20));
        }
    };
    progress(ctx);
    CK(wait_event(s.ev[EV_META]));
    progress(ctx);
    const int64_t g_elems = s.h_totals[0], r_elems = s.h_totals[1];
    const int32_t status = *reinterpret_cast<int32_t*>(s.h_totals + 2);
    if (prm.host_output && !s.waited) {
        if (!s.early_d2h) { // the copies wait for the totals: enqueue them now unless an earlier call already did (progress())
            const int rc = issue_d2h(ctx, s);
            if (rc != VGL_OK) return rc;
        }
        CK(wait_event(s.ev[EV_D2H1]));
        s.had_d2h = true;
    }
    const bool first_wait = !s.waited;
    if (!s.waited) {
        float* ms = s.ms;
        CK(cudaEventElapsedTime(&ms[VGL_T_H2D], s.ev[EV_START], s.ev[EV_H2D]));
        CK(cudaEventElapsedTime(&ms[VGL_T_SIM], s.ev[EV_H2D], s.ev[EV_SIM]));
        CK(cudaEventElapsedTime(&ms[VGL_T_SITE], s.ev[EV_SIM], s.ev[EV_SITE]));
        CK(cudaEventElapsedTime(&ms[VGL_T_SCAN], s.ev[EV_SITE], s.ev[EV_SCAN]));
        CK(cudaEventElapsedTime(&ms[VGL_T_EMIT], s.ev[EV_SCAN], s.ev[EV_EMIT]));
        float meta = 0.f, d2h = 0.f;
        CK(cudaEventElapsedTime(&meta, s.ev[EV_EMIT], s.ev[EV_META]));
        if (s.had_d2h) CK(cudaEventElapsedTime(&d2h, s.ev[EV_D2H0], s.ev[EV_D2H1]));
        ms[VGL_T_D2H] = meta + d2h;
        CK(cudaEventElapsedTime(&ms[VGL_T_TOTAL], s.ev[EV_START], s.had_d2h ? s.ev[EV_D2H1] : s.ev[EV_META]));
    }
    s.waited = true;
    memset(out, 0, sizeof *out);
    out->n_sites = s.n_sites;
    out->n_samples = prm.n_samples;
    // VGL_HOST_NONE: the device planes.  Else the host copies: none under VGL_HOST_BCF / BGZF (the host gets the serialised
    // records), the narrowed ones where VGL_HOST_NARROW narrows a plane
    const bool h = prm.host_output != 0;
    auto view = [&](int i) { return h ? s.plane[i].h : s.plane[i].d; };
    out->sites = h ? s.h_sites : s.d_sites;
    out->dp = (const int32_t*)view(P_DP);
    out->gl = (const float*)view(P_GL);
    out->pl = (const int32_t*)view(P_PL);
    out->gp = (const float*)view(P_GP);
    out->ad = (const int32_t*)view(P_AD);
    out->adf = (const int32_t*)view(P_ADF);
    out->adr = (const int32_t*)view(P_ADR);
    out->narrow_bits = ctx->narrow_bits;
    out->pl_u8 = (const uint8_t*)s.plane[P_PL].hn;
    out->dp_n = s.plane[P_DP].hn;
    out->ad_n = s.plane[P_AD].hn;
    out->adf_n = s.plane[P_ADF].hn;
    out->adr_n = s.plane[P_ADR].hn;
    if (prm.host_output == VGL_HOST_BCF || prm.host_output == VGL_HOST_BGZF) {
        if (prm.host_output == VGL_HOST_BGZF) {
            out->bgzf = s.h_bgzf;
            out->bgzf_bytes = s.h_totals[4];
            out->bgzf_blocks = (int32_t)s.h_totals[5];
        }
        out->bcf = s.h_bcf ? s.h_bcf + ctx->bcf_headroom : nullptr;
        out->bcf_off = reinterpret_cast<const int64_t*>(s.h_rec_off);
        out->bcf_bytes = s.h_totals[3];
        if (prm.do_gvcf && prm.host_output == VGL_HOST_BCF && first_wait) gvcf_seam(ctx, s, out);
        else if (prm.do_gvcf && prm.host_output == VGL_HOST_BCF) { out->bcf = s.seam_ptr; out->bcf_bytes = s.seam_bytes; out->bcf_off = nullptr; out->n_recs = s.seam_recs; }
    }
    out->g_elems = g_elems;
    out->r_elems = r_elems;
    out->status = status;
    return VGL_OK;
}

extern "C" int vgl_native_draws(vgl_ctx* ctx, int slot, int64_t first_site_id, int32_t n_sites, vgl_draws* out)
{
    if (!ctx || !out || slot < 0 || slot >= (int)ctx->slots.size()) return VGL_EINVAL;
    if (n_sites < 1 || n_sites > ctx->prm.max_batch_sites || first_site_id < 0) return fail(ctx, VGL_EINVAL, "n_sites / first_site_id out of range");
    Slot& s = ctx->slots[slot];
    if (s.submitted && !s.waited) return fail(ctx, VGL_ESTATE, "slot still in flight");
    if (ctx->plan.set == KS_FUSED_M1F) return fail(ctx, VGL_ESTATE, "per-read draws do not exist under the count-level sampler (create the context with VGL_SAMPLER_PER_READ)");
    const vgl_params& prm = ctx->prm;
    CK(cudaSetDevice(prm.device_id));
    cudaStream_t st = s.stream;
    const int64_t cells = (int64_t)n_sites * prm.n_samples;
    DevParams p;
    fill_params(ctx, s, first_site_id, n_sites, p);
    CK(cudaMemcpyAsync(s.d_gt, s.h_gt, (size_t)cells, cudaMemcpyHostToDevice, st));
    const bool m2 = ctx->plan.set == KS_TILE_M2;  // the model-2 tile kernel's own sampler (read order matters there)
    const bool m1t = ctx->plan.set == KS_TILE_M1F; // the model-1 tile kernel's count-level sampler, listed read by read
    if (m2) launch_tile_m2_draws(p, st, prm.error_qs, 0, s.dev(P_DP), nullptr, nullptr, nullptr, nullptr);
    else if (m1t) launch_tile_m1f_draws(p, st, 0, s.dev(P_DP), nullptr, nullptr, nullptr, nullptr);
    else launch_sim(p, st); // depths (and counts, unused here)
    ctx->launches += 1;
    s.dr_depths.resize((size_t)cells);
    CK(cudaMemcpyAsync(s.dr_depths.data(), s.dev(P_DP), (size_t)cells * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    s.dr_off.resize((size_t)cells + 1);
    s.dr_off[0] = 0;
    for (int64_t c = 0; c < cells; ++c) s.dr_off[c + 1] = s.dr_off[c] + s.dr_depths[c]; // output layout only
    const size_t nr = (size_t)s.dr_off[cells];
    int64_t* d_off = nullptr;
    uint8_t* d_u8 = nullptr;
    double* d_e = nullptr;
    CK(cudaMalloc((void**)&d_off, ((size_t)cells + 1) * 8));
    CK(cudaMalloc((void**)&d_u8, 5 * nr + 16));
    CK(cudaMalloc((void**)&d_e, nr * 8 + 16));
    CK(cudaMemsetAsync(d_u8, 0, 5 * nr + 16, st));
    CK(cudaMemsetAsync(d_e, 0, nr * 8 + 16, st));
    CK(cudaMemcpyAsync(d_off, s.dr_off.data(), ((size_t)cells + 1) * 8, cudaMemcpyHostToDevice, st));
    if (m2) {
        launch_tile_m2_draws(p, st, prm.error_qs, 1, nullptr, d_off, d_u8, d_u8 + 2 * nr, d_e);
        // the class table holds the score the GL uses: export it as both the raw and the adjusted score
        if (nr) CK(cudaMemcpyAsync(d_u8 + 3 * nr, d_u8 + 2 * nr, nr, cudaMemcpyDeviceToDevice, st));
    } else if (m1t) {
        launch_tile_m1f_draws(p, st, 1, s.dev(P_DP), d_off, d_u8, d_u8 + nr, d_u8 + 4 * nr);
    } else {
        launch_draws(p, st, d_off, d_u8, d_u8 + nr, d_u8 + 2 * nr, d_u8 + 3 * nr, d_u8 + 4 * nr, d_e);
    }
    ctx->launches += 1;
    CK(cudaGetLastError());
    s.dr_bases.resize(nr); s.dr_strands.resize(nr); s.dr_qs.resize(nr); s.dr_adjqs.resize(nr); s.dr_tails.resize(nr);
    s.dr_eprob.resize(nr);
    if (nr) {
        CK(cudaMemcpyAsync(s.dr_bases.data(), d_u8, nr, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(s.dr_strands.data(), d_u8 + nr, nr, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(s.dr_qs.data(), d_u8 + 2 * nr, nr, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(s.dr_adjqs.data(), d_u8 + 3 * nr, nr, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(s.dr_tails.data(), d_u8 + 4 * nr, nr, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(s.dr_eprob.data(), d_e, nr * 8, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    cudaFree(d_off); cudaFree(d_u8); cudaFree(d_e);
    out->n_cells = cells;
    out->n_reads = (int64_t)nr;
    out->depths = s.dr_depths.data();
    out->read_offsets = s.dr_off.data();
    out->bases = s.dr_bases.data();
    out->strands = s.dr_strands.data();
    out->qs = prm.error_qs == 2 ? s.dr_qs.data() : nullptr;
    out->adj_qs = prm.error_qs == 2 && prm.adjust_qs ? s.dr_adjqs.data() : nullptr;
    out->tail_dists = s.dr_tails.data();
    out->error_probs = prm.error_qs != 0 ? s.dr_eprob.data() : nullptr; // --error-qs 1: each read carries its site's rate
    return VGL_OK;
}

extern "C" int vgl_selftest(int device_id, int64_t* n_mismatch, uint32_t* first_mismatch_bits)
{
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) return VGL_ENODEV;
    if (device_id < 0 || device_id >= n_dev || !n_mismatch) return VGL_EINVAL;
    if (cudaSetDevice(device_id) != cudaSuccess) return VGL_ECUDA;
    unsigned long long bad = 0;
    unsigned int first = 0;
    if (run_selftest(&bad, &first) != 0) return VGL_ECUDA;
    *n_mismatch = (int64_t)bad;
    if (first_mismatch_bits) *first_mismatch_bits = first;
    return VGL_OK;
}

extern "C" int vgl_copy_sites(vgl_ctx* ctx, int slot, vgl_site_out* host_dst)
{
    if (!ctx || !host_dst || slot < 0 || slot >= (int)ctx->slots.size()) return VGL_EINVAL;
    Slot& s = ctx->slots[slot];
    if (!s.waited) return fail(ctx, VGL_ESTATE, "vgl_copy_sites: call vgl_wait first");
    CK(cudaSetDevice(ctx->prm.device_id));
    CK(cudaMemcpyAsync(host_dst, s.d_sites, (size_t)s.n_sites * sizeof(vgl_site_out), cudaMemcpyDeviceToHost, s.stream));
    CK(cudaStreamSynchronize(s.stream));
    return VGL_OK;
}

extern "C" int vgl_slot_timing(vgl_ctx* ctx, int slot, float ms[VGL_T_COUNT])
{
    if (!ctx || !ms || slot < 0 || slot >= (int)ctx->slots.size()) return VGL_EINVAL;
    Slot& s = ctx->slots[slot];
    if (!s.waited) return VGL_ESTATE;
    memcpy(ms, s.ms, sizeof s.ms);
    return VGL_OK;
}
