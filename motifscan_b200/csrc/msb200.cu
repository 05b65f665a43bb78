// msb200.cu -- host side of libmsb200.so: the C ABI declared in include/msb200.h.
//
// Replaces the reference's native extension motifscan/motif/cscore.c for the scan path:
//   convert_args/convert_pwm/convert_seq (cscore.c:50-151)  -> msb_motifs_create, msb_seqs_from_ascii
//   scan_motif_thread/scan_motif         (cscore.c:317-476) -> msb_scan
//   motif_score_thread/motif_score       (cscore.c:174-302) -> msb_score, msb_score_select
// There is no CPU implementation in this library: without a CUDA device every entry point that
// computes returns MSB_ECUDA.
#include <cub/cub.cuh>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <limits>
#include <mutex>
#include <new>
#include <numeric>
#include <charconv>
#include <thread>

#include "kernels.cuh"
#include "prefilter_tc.cuh"

namespace msb {

static constexpr int kSelSmemKeys = 24576;   // select_ranks_kernel: 192 KB of staged keys per block

static thread_local std::string g_err;
void set_error(const std::string &msg) { g_err = msg; }
int cuda_fail(cudaError_t e, const char *what, const char *file, int line) {
    g_err = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what + " (" + file + ":" +
            std::to_string(line) + ")";
    cudaGetLastError();  // clear the sticky-less error state
    return e == cudaErrorMemoryAllocation ? MSB_ENOMEM : MSB_ECUDA;
}

int DevBuf::ensure(size_t bytes) {
    if (bytes <= cap) return MSB_OK;
    size_t want = std::max(bytes, cap + cap / 2);
    void *np = nullptr;
    if (p) { cudaFree(p); p = nullptr; cap = 0; }
    cudaError_t e = cudaMalloc(&np, want);
    if (e != cudaSuccess && want > bytes) e = cudaMalloc(&np, want = bytes);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc", __FILE__, __LINE__);
    p = np;
    cap = want;
    return MSB_OK;
}
void DevBuf::release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
}

struct PinnedBlock {
    void *p = nullptr;
    size_t cap = 0;
};

}  // namespace msb

using namespace msb;

// ------------------------------------------------------------------------------------------------
struct msb_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 0;
    cudaEvent_t ev[8] = {};
    cudaStream_t copy_stream = nullptr;   // msb_scan_ascii: host-to-device slices overlap the scan (created on first use)
    cudaEvent_t slice_ev[8] = {};
    double t[MSB_T_COUNT] = {};
    int64_t c[MSB_C_COUNT] = {};
    // scratch (grow-only, reused across calls)
    DevBuf ascii, seq_off, cand, dirty, hit_key, hit_score, key_alt, score_alt, sort_tmp, counters;
    DevBuf out_seq, out_start, out_strand, scores, scores_sorted, seg_off, ranks, sel;
    DevBuf keep, keep_pos, motif_counts, sel_aux, limit1;
    DevBuf lane_count;   // tensor-core prefilter: records per epilogue lane
    // boundary chains of the last de-duplicated range scan (msb_scan_device_boundary_sites)
    DevBuf bnd_range, bnd_cnt, bnd_dst, bnd_motif, bnd_seq, bnd_start, bnd_score, bnd_strand, bnd_flags;
    int64_t last_boundary = -1;            // sites in the bnd_* arrays; -1: the last scan collected none
    // rows of the last variant / haplotype scan (msb_scan_device_variant_rows): unsorted, sort keys, then in row
    // order; vr_core holds the edit tables (ref at | alt at | ref len | alt len), vr_eoff the edit offsets
    DevBuf vr_key, vr_idx, vr_ref, vr_alt, vr_eff, vr_other, vr_key_sorted, vr_idx_sorted, vr_core, vr_eoff;
    DevBuf vo_allele, vo_motif, vo_start, vo_strand, vo_ref, vo_alt, vo_eff, vo_other;
    int64_t last_variant_rows = -1;        // -1: the last scan was not a variant scan
    bool last_rows_other = false;          // the last variant scan recorded other-side starts (msb_scan_haplotypes)
    // Final site arrays of a scan.  Two sets, used alternately: the device-to-host copy of scan k's
    // sites (on d2h_stream, MSB_SCAN_ASYNC) reads one set while scan k + 1 fills the other.
    struct FinSet {
        DevBuf key, score, seq, start, strand, offsets;   // offsets: CSR over motifs, n_motifs + 1 entries
        cudaEvent_t read_done = nullptr;                  // recorded on d2h_stream behind the copies that read this set
        bool pending = false;
    } fin[2];
    int fin_cur = 0;
    bool fin_hold = false;                 // msb_scan_variants: the other set holds the ref scan's sites, which the alt scan
                                           // must neither reuse nor release
    bool last_counts_only = false;
    bool last_compact = false;             // MSB_SCAN_COMPACT: fin[].start holds (packed position << 1 | strand) as uint32
    const msb_seqs *last_seqs = nullptr;   // the sequence set of the last scan (its layout decodes compact sites)
    cudaStream_t d2h_stream = nullptr;
    cudaStream_t aux_stream = nullptr;     // exact_dirty_kernel beside exact_records_kernel
    cudaEvent_t aux_fork = nullptr, aux_join = nullptr;
    // final site arrays of the last scan (point into fin[fin_cur])
    uint64_t *fin_key = nullptr;
    double *fin_score = nullptr;
    int32_t *fin_seq = nullptr, *fin_start = nullptr;
    int8_t *fin_strand = nullptr;
    unsigned long long *h_counters = nullptr;  // pinned, 4 entries
    std::vector<PinnedBlock> pinned_free;
    std::mutex pinned_mu;
    std::vector<DevBuf> dev_free;     // device buffers of destroyed sequence sets, reused by the next one
    std::mutex dev_mu;
    // results of the last msb_scan_device, still on the device
    int64_t last_sites = 0;
    int32_t last_n_motifs = 0;
    int64_t last_n_seqs = 0;
    int last_key_shift = 0;
    // tuning / test knobs (msb_ctx_set_option): per context, so that contexts driven from different host
    // threads never see each other's settings
    int opt_tc_prof = 0;             // 1: print per-role cycle counters of the tensor-core prefilter to stderr
    int opt_ascii_slices = 4;        // msb_scan_ascii: upload slices (1..7)
    int opt_tc_first_lane_cap = 0;   // tests: records per lane buffer on the first attempt (0 = sized from the input)
    int opt_poison_pool = 0;         // tests: fill device buffers with 0xFF when they go back to the pool
    int opt_tc_interleave = 1;       // tensor-core prefilter: short and long motif tiles alternate (0: ascending by length)
    int opt_select_pilot = 1;        // msb_score_select: 0 = always score every sample for every motif (the plain form)
};

// Tensor-core prefilter tables (prefilter_tc.cuh).
struct TcTableSet {
    bool valid = false;
    uint64_t cutoff_version = 0;
    std::vector<int32_t> order;       // sorted index -> motif id (fast motifs only, by K steps)
    std::vector<int32_t> slow;
    std::vector<TcBatch> batches;
    int32_t lmax_fast = 0;
    int any_zero_hit = 0;
    DevBuf d_btab, d_col_info, d_len, d_order, d_slow;
};

struct msb_motifs {
    msb_ctx *ctx = nullptr;
    int32_t n = 0;
    std::vector<int32_t> lens, col_off;
    std::vector<int64_t> mat_off;
    std::vector<double> mats;     // row-major 4 x L per motif, as given
    std::vector<double> cutoffs, max_raw;
    uint64_t cutoff_version = 1;
    int32_t lmax = 0;
    DevBuf d_pwm, d_col_off, d_len, d_cutoff, d_max_raw, d_pwm32, d_floor32;
    TcTableSet tc_tables[4];
    MotifView view() const {
        MotifView v;
        v.pwm = d_pwm.as<double>();
        v.col_off = d_col_off.as<int32_t>();
        v.len = d_len.as<int32_t>();
        v.cutoff = d_cutoff.as<double>();
        v.max_raw = d_max_raw.as<double>();
        v.pwm32 = d_pwm32.as<float>();
        v.floor32 = d_floor32.as<float>();
        v.n_motifs = n;
        return v;
    }
};

struct msb_seqs {
    msb_ctx *ctx = nullptr;
    int64_t n = 0, total_bp = 0, total_packed = 0;
    int32_t min_len = 0;
    std::vector<int64_t> seq_off, poff;
    DevBuf d_codes, d_nmask, d_poff, d_len, d_seq_off, d_blk_seq, d_limit;
    bool has_limit = false;
    std::vector<int32_t> lens32;          // host copy of d_len (source of an asynchronous upload)
    PinnedBlock tables;                   // asynchronous upload: poff | seq_off | len staged in pinned memory, so that the
                                          // copies neither block the host nor wait for the copy stream to drain
    // MSB_SEQS_ASYNC: the upload runs on the context's copy stream; the first call that reads the set makes
    // the main stream wait for `ready`
    mutable cudaEvent_t ready = nullptr;
    mutable bool ready_pending = false;
    SeqView view() const {
        SeqView v;
        v.codes = d_codes.as<uint32_t>();
        v.nmask = d_nmask.as<uint32_t>();
        v.poff = d_poff.as<int64_t>();
        v.len = d_len.as<int32_t>();
        v.blk_seq = d_blk_seq.as<int32_t>();
        v.limit = has_limit ? d_limit.as<int32_t>() : nullptr;
        v.n_seqs = n;
        v.total_packed = total_packed;
        return v;
    }
};

struct msb_result {
    msb_ctx *ctx = nullptr;
    int device = 0;
    int64_t n_sites = 0;
    int32_t n_motifs = 0;
    PinnedBlock block;       // score (8n) | seq_idx (4n) | start (4n) | strand (n) | pad | motif offsets (8 (n_motifs + 1))
    int32_t *seq_idx = nullptr;
    int32_t *start = nullptr;
    double *score = nullptr;
    int8_t *strand = nullptr;
    int64_t *offsets = nullptr;
    uint32_t *compact = nullptr;            // MSB_SCAN_COMPACT: packed position << 1 | strand bit, instead of the three arrays
    std::vector<int64_t> poff;              // compact: packed start of every sequence of the scanned set (+ end)
    std::vector<char> decoded;              // compact: seq_idx | start | strand, filled by the first msb_result_arrays
    std::vector<int64_t> counts;
    cudaEvent_t t0 = nullptr, done = nullptr;   // on the context's d2h stream around the copies
    bool pending = false;                       // MSB_SCAN_ASYNC: the copies may still be in flight
};

// ------------------------------------------------------------------------------------------------
static int pinned_get(msb_ctx *ctx, size_t bytes, PinnedBlock *out) {
    {
        std::lock_guard<std::mutex> g(ctx->pinned_mu);
        int best = -1;
        for (size_t i = 0; i < ctx->pinned_free.size(); i++)
            if (ctx->pinned_free[i].cap >= bytes && ctx->pinned_free[i].cap <= 4 * bytes + (64 << 10) &&   // a table does not take a result's block
                (best < 0 || ctx->pinned_free[i].cap < ctx->pinned_free[best].cap))
                best = (int) i;
        if (best >= 0) {
            *out = ctx->pinned_free[best];
            ctx->pinned_free.erase(ctx->pinned_free.begin() + best);
            return MSB_OK;
        }
    }
    // some headroom, whole MiB: the next scan's result of about the same size finds this block in the pool
    size_t cap = bytes < (1 << 20) ? std::max<size_t>(bytes, 4096) : (((bytes + bytes / 8) >> 20) + 1) << 20;
    void *p = nullptr;
    MSB_CUDA(cudaHostAlloc(&p, cap, cudaHostAllocDefault));
    out->p = p;
    out->cap = cap;
    return MSB_OK;
}
static void pinned_put(msb_ctx *ctx, PinnedBlock b) {
    if (!b.p) return;
    std::lock_guard<std::mutex> g(ctx->pinned_mu);
    // a genome-wide scan holds one block per unit (~50 for hg19) until its sites are gathered, step after step:
    // page-locking is slow (~0.3 ms/MB), so the pool keeps them all
    if (ctx->pinned_free.size() < 512) ctx->pinned_free.push_back(b);
    else cudaFreeHost(b.p);
}

// Device buffers of sequence sets come from / go back to a small per-context pool: a scan service
// creates and destroys one msb_seqs per request, and cudaMalloc / cudaFree would otherwise
// synchronise the device twice per request.
static int dev_take(msb_ctx *ctx, DevBuf &b, size_t bytes) {
    {
        std::lock_guard<std::mutex> g(ctx->dev_mu);
        int best = -1;
        for (size_t i = 0; i < ctx->dev_free.size(); i++)
            // best fit, whatever the excess: a unit of a quarter of the usual size takes a full-size buffer rather
            // than a cudaMalloc (which synchronises the device in the middle of a pipelined scan)
            if (ctx->dev_free[i].cap >= bytes &&
                (best < 0 || ctx->dev_free[i].cap < ctx->dev_free[best].cap))
                best = (int) i;
        if (best >= 0) {
            b = ctx->dev_free[best];
            ctx->dev_free.erase(ctx->dev_free.begin() + best);
            return MSB_OK;
        }
    }
    return b.ensure(bytes);
}
static void dev_give(msb_ctx *ctx, DevBuf &b) {
    if (!b.p) return;
    if (ctx->opt_poison_pool) cudaMemsetAsync(b.p, 0xFF, b.cap, ctx->stream);
    std::lock_guard<std::mutex> g(ctx->dev_mu);
    if (ctx->dev_free.size() < 96) {
        ctx->dev_free.push_back(b);
        b.p = nullptr;
        b.cap = 0;
    } else {
        b.release();
    }
}

static int ensure_copy_stream(msb_ctx *ctx) {
    if (!ctx->copy_stream) MSB_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    return MSB_OK;
}

// An asynchronously uploaded sequence set becomes readable on the main stream behind its `ready` event.
static int seqs_ready(const msb_seqs *S) {
    if (S && S->ready_pending) {
        MSB_CUDA(cudaStreamWaitEvent(S->ctx->stream, S->ready, 0));
        S->ready_pending = false;
    }
    return MSB_OK;
}

static inline float ev_ms(cudaEvent_t a, cudaEvent_t b) {
    float ms = 0;
    cudaEventElapsedTime(&ms, a, b);
    return ms;
}

// ------------------------------------------------------------------------------------------------
extern "C" {

const char *msb_last_error(void) { return g_err.c_str(); }
int msb_version(void) { return 100; }

int msb_device_count(int *count) {
    if (!count) { set_error("msb_device_count: null"); return MSB_EINVAL; }
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { cudaGetLastError(); n = 0; }
    *count = n;
    return MSB_OK;
}

int msb_device_pci_bus_id(int device, char *out, int len) {
    if (!out || len < 16) { set_error("msb_device_pci_bus_id: buffer too small"); return MSB_EINVAL; }
    MSB_CUDA(cudaDeviceGetPCIBusId(out, len, device));
    return MSB_OK;
}

int msb_pinned_alloc(int64_t bytes, void **ptr) {
    if (!ptr || bytes < 0) { set_error("msb_pinned_alloc: bad argument"); return MSB_EINVAL; }
    MSB_CUDA(cudaHostAlloc(ptr, (size_t) std::max<int64_t>(bytes, 1), cudaHostAllocDefault));
    return MSB_OK;
}
int msb_pinned_free(void *ptr) {
    if (ptr) MSB_CUDA(cudaFreeHost(ptr));
    return MSB_OK;
}

int msb_ctx_create(int device, void *stream, msb_ctx **out) {
    if (!out) { set_error("msb_ctx_create: null out"); return MSB_EINVAL; }
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        set_error("no CUDA device available: libmsb200 has no CPU path");
        return MSB_ECUDA;
    }
    if (device < 0 || device >= n) { set_error("msb_ctx_create: device out of range"); return MSB_EINVAL; }
    MSB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    MSB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("libmsb200 is built for sm_100a (B200) only; device is sm_" + std::to_string(prop.major) +
                  std::to_string(prop.minor));
        return MSB_ECUDA;
    }
    msb_ctx *ctx = new (std::nothrow) msb_ctx();
    if (!ctx) { set_error("out of host memory"); return MSB_ENOMEM; }
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    if (stream) {
        ctx->stream = (cudaStream_t) stream;
    } else {
        cudaError_t se = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
        if (se != cudaSuccess) { delete ctx; return cuda_fail(se, "cudaStreamCreate", __FILE__, __LINE__); }
        ctx->own_stream = true;
    }
    for (auto &evt : ctx->ev) cudaEventCreate(&evt);
    cudaHostAlloc((void **) &ctx->h_counters, 4 * sizeof(unsigned long long), cudaHostAllocDefault);
    if (ctx->counters.ensure(4 * sizeof(unsigned long long)) != MSB_OK || !ctx->h_counters) {
        msb_ctx_destroy(ctx);
        return MSB_ENOMEM;
    }
    ctx->opt_tc_prof = std::getenv("MSB_TC_PROF") ? 1 : 0;
    if (cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->aux_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->aux_join, cudaEventDisableTiming) != cudaSuccess) {
        cudaGetLastError();
        if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
        ctx->aux_stream = nullptr;   // everything stays on the main stream
    }
    cudaFuncSetAttribute(prefilter_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemBytes);
    cudaFuncSetAttribute(prefilter_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemBytes);
    cudaFuncSetAttribute(select_ranks_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSelSmemKeys * 8);
    cudaFuncSetAttribute(select_ranks_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSelSmemKeys * 8);
    *out = ctx;
    return MSB_OK;
}

int msb_ctx_destroy(msb_ctx *ctx) {
    if (!ctx) return MSB_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (DevBuf *b : {&ctx->ascii, &ctx->seq_off, &ctx->cand, &ctx->dirty, &ctx->hit_key, &ctx->hit_score,
                      &ctx->key_alt, &ctx->score_alt, &ctx->sort_tmp, &ctx->counters, &ctx->out_seq,
                      &ctx->out_start, &ctx->out_strand, &ctx->scores,
                      &ctx->scores_sorted, &ctx->seg_off, &ctx->ranks, &ctx->sel, &ctx->keep, &ctx->keep_pos,
                      &ctx->motif_counts, &ctx->sel_aux, &ctx->limit1, &ctx->lane_count, &ctx->bnd_range,
                      &ctx->bnd_cnt, &ctx->bnd_dst, &ctx->bnd_motif, &ctx->bnd_seq, &ctx->bnd_start, &ctx->bnd_score,
                      &ctx->bnd_strand, &ctx->bnd_flags, &ctx->vr_key, &ctx->vr_idx, &ctx->vr_ref, &ctx->vr_alt,
                      &ctx->vr_eff, &ctx->vr_other, &ctx->vr_key_sorted, &ctx->vr_idx_sorted, &ctx->vr_core,
                      &ctx->vr_eoff, &ctx->vo_allele, &ctx->vo_motif, &ctx->vo_start, &ctx->vo_strand, &ctx->vo_ref,
                      &ctx->vo_alt, &ctx->vo_eff, &ctx->vo_other})
        b->release();
    if (ctx->d2h_stream) cudaStreamSynchronize(ctx->d2h_stream);
    for (auto &f : ctx->fin) {
        for (DevBuf *b : {&f.key, &f.score, &f.seq, &f.start, &f.strand, &f.offsets}) b->release();
        if (f.read_done) cudaEventDestroy(f.read_done);
    }
    if (ctx->d2h_stream) cudaStreamDestroy(ctx->d2h_stream);
    if (ctx->aux_stream) { cudaStreamSynchronize(ctx->aux_stream); cudaStreamDestroy(ctx->aux_stream); }
    if (ctx->aux_fork) cudaEventDestroy(ctx->aux_fork);
    if (ctx->aux_join) cudaEventDestroy(ctx->aux_join);
    for (auto &b : ctx->pinned_free) cudaFreeHost(b.p);
    for (auto &b : ctx->dev_free) b.release();
    if (ctx->h_counters) cudaFreeHost(ctx->h_counters);
    for (auto &evt : ctx->ev) if (evt) cudaEventDestroy(evt);
    for (auto &evt : ctx->slice_ev) if (evt) cudaEventDestroy(evt);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return MSB_OK;
}

int msb_ctx_sync(msb_ctx *ctx) {
    if (!ctx) { set_error("null ctx"); return MSB_EINVAL; }
    MSB_CUDA(cudaStreamSynchronize(ctx->stream));
    return MSB_OK;
}

int msb_ctx_timings(const msb_ctx *ctx, double *ms, int n) {
    if (!ctx || !ms) { set_error("msb_ctx_timings: null"); return MSB_EINVAL; }
    for (int i = 0; i < n && i < MSB_T_COUNT; i++) ms[i] = ctx->t[i];
    return MSB_OK;
}
int msb_ctx_counters(const msb_ctx *ctx, int64_t *v, int n) {
    if (!ctx || !v) { set_error("msb_ctx_counters: null"); return MSB_EINVAL; }
    for (int i = 0; i < n && i < MSB_C_COUNT; i++) v[i] = ctx->c[i];
    return MSB_OK;
}

// ---- motifs ------------------------------------------------------------------------------------
// fp32 screening threshold of every motif for the exact stage's dirty-window kernel: a window whose
// raw score accumulated in fp32 from the fp32-rounded matrix is below floor32[m] cannot satisfy the
// reference's predicate.  T is the conservative bound on the exact raw score that the prefilter
// tables use (see "Prefilter tables" below); the fp32 path is off by at most
// sum_c |v_c| 2^-24 (rounding the entries) + (L - 1) 2^-24 max|partial sum| <= L 2^-23 abs_sum
// (= 2^-18 abs_sum for L = 32), and the margin taken here is 2^-17 (abs_sum + |T| + 1): at least twice the
// worst case, about four times the typical one.
static int upload_floors(msb_motifs *M) {
    std::vector<float> floors((size_t) std::max<int32_t>(M->n, 1), std::numeric_limits<float>::infinity());
    for (int32_t m = 0; m < M->n; m++) {
        const int L = M->lens[m];
        const double max_raw = M->max_raw[m], cutoff = M->cutoffs[m];
        if (L < 1 || !(max_raw > 0) || std::isnan(cutoff) || (std::isinf(cutoff) && cutoff > 0)) continue;   // never a site
        if (std::isinf(cutoff)) { floors[m] = -std::numeric_limits<float>::infinity(); continue; }
        const double *mat = M->mats.data() + M->mat_off[m];
        double abs_sum = 0;
        bool finite = true;
        for (int c = 0; c < L; c++) {
            double a = 0;
            for (int r = 0; r < 4; r++) { a = std::max(a, std::fabs(mat[(size_t) r * L + c])); finite = finite && std::isfinite(mat[(size_t) r * L + c]); }
            abs_sum += a;
        }
        if (!finite || abs_sum > 1e30) { floors[m] = -std::numeric_limits<float>::infinity(); continue; }   // no screening (fp32 would overflow; a NaN sum also passes the screen)
        const double T = max_raw * (cutoff - 1e-10) - 1e-12 * (max_raw * (std::fabs(cutoff) + 1.0) + abs_sum);
        const double f = T - std::ldexp(abs_sum + std::fabs(T) + 1.0, -17);
        float ff = (float) f;
        if ((double) ff > f) ff = std::nextafterf(ff, -std::numeric_limits<float>::infinity());
        floors[m] = ff;
    }
    MSB_TRY(M->d_floor32.ensure(floors.size() * sizeof(float)));
    MSB_CUDA(cudaMemcpyAsync(M->d_floor32.p, floors.data(), floors.size() * sizeof(float), cudaMemcpyHostToDevice, M->ctx->stream));
    MSB_CUDA(cudaStreamSynchronize(M->ctx->stream));
    return MSB_OK;
}

int msb_motifs_create(msb_ctx *ctx, int32_t n, const int32_t *lens, const double *mats,
                      const int64_t *mat_off, const double *cutoffs, msb_motifs **out) {
    if (!ctx || !out || n < 0 || (n > 0 && (!lens || !mats || !mat_off))) {
        set_error("msb_motifs_create: bad argument");
        return MSB_EINVAL;
    }
    *out = nullptr;
    if ((uint64_t) n >= (1ull << (64 - kMotifShift))) { set_error("too many motifs"); return MSB_EINVAL; }
    for (int32_t m = 0; m < n; m++)
        if (lens[m] < 0 || mat_off[m] < 0) { set_error("msb_motifs_create: negative length/offset"); return MSB_EINVAL; }
    MSB_CUDA(cudaSetDevice(ctx->device));
    msb_motifs *M = new (std::nothrow) msb_motifs();
    if (!M) { set_error("out of host memory"); return MSB_ENOMEM; }
    M->ctx = ctx;
    M->n = n;
    M->lens.assign(lens, lens + n);
    M->col_off.resize(n + 1);
    M->mat_off.resize(n);
    M->cutoffs.resize(n);
    M->max_raw.resize(n);
    int64_t total_cols = 0;
    for (int32_t m = 0; m < n; m++) {
        M->col_off[m] = (int32_t) total_cols;
        total_cols += lens[m];
        M->lmax = std::max(M->lmax, lens[m]);
    }
    M->col_off[n] = (int32_t) total_cols;
    M->mats.resize((size_t) total_cols * 4);
    std::vector<double> dev_pwm((size_t) total_cols * 4);  // [motif][col][row]
    for (int32_t m = 0; m < n; m++) {
        const int L = lens[m];
        const double *src = mats + mat_off[m];
        double *dst = M->mats.data() + 4 * (size_t) M->col_off[m];
        M->mat_off[m] = 4 * (int64_t) M->col_off[m];
        std::memcpy(dst, src, sizeof(double) * 4 * (size_t) L);
        // get_max_raw_score, cscore.c:36-48: column maximum floored at 0, summed ascending.
        double max_raw = 0;
        for (int j = 0; j < L; j++) {
            double col_max = 0;
            for (int r = 0; r < 4; r++) {
                const double v = src[(size_t) r * L + j];
                if (v > col_max) col_max = v;
                dev_pwm[4 * ((size_t) M->col_off[m] + j) + r] = v;
            }
            max_raw += col_max;
        }
        M->max_raw[m] = max_raw;
        M->cutoffs[m] = cutoffs ? cutoffs[m] : 1.0;  // cscore.c:71-75
    }
    int rc = MSB_OK;
    auto up = [&](DevBuf &b, const void *src, size_t bytes) {
        if (rc != MSB_OK) return;
        rc = b.ensure(std::max<size_t>(bytes, 16));
        if (rc == MSB_OK && bytes) {
            cudaError_t e = cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, ctx->stream);
            if (e != cudaSuccess) rc = cuda_fail(e, "cudaMemcpyAsync", __FILE__, __LINE__);
        }
    };
    up(M->d_pwm, dev_pwm.data(), dev_pwm.size() * sizeof(double));
    std::vector<float> dev_pwm32(dev_pwm.size());
    for (size_t i = 0; i < dev_pwm.size(); i++) dev_pwm32[i] = (float) dev_pwm[i];
    up(M->d_pwm32, dev_pwm32.data(), dev_pwm32.size() * sizeof(float));
    up(M->d_col_off, M->col_off.data(), M->col_off.size() * sizeof(int32_t));
    up(M->d_len, M->lens.data(), (size_t) n * sizeof(int32_t));
    up(M->d_cutoff, M->cutoffs.data(), (size_t) n * sizeof(double));
    up(M->d_max_raw, M->max_raw.data(), (size_t) n * sizeof(double));
    if (rc == MSB_OK) {
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = cuda_fail(e, "cudaStreamSynchronize", __FILE__, __LINE__);
    }
    if (rc == MSB_OK) rc = upload_floors(M);
    if (rc != MSB_OK) { msb_motifs_destroy(M); return rc; }
    *out = M;
    return MSB_OK;
}

int msb_motifs_set_cutoffs(msb_motifs *M, const double *cutoffs) {
    if (!M) { set_error("null motifs"); return MSB_EINVAL; }
    MSB_CUDA(cudaSetDevice(M->ctx->device));
    for (int32_t m = 0; m < M->n; m++) M->cutoffs[m] = cutoffs ? cutoffs[m] : 1.0;
    M->cutoff_version++;
    if (M->n)
        MSB_CUDA(cudaMemcpyAsync(M->d_cutoff.p, M->cutoffs.data(), (size_t) M->n * sizeof(double),
                                 cudaMemcpyHostToDevice, M->ctx->stream));
    MSB_CUDA(cudaStreamSynchronize(M->ctx->stream));
    return upload_floors(M);
}

int msb_motifs_count(const msb_motifs *M, int32_t *n) {
    if (!M || !n) { set_error("null"); return MSB_EINVAL; }
    *n = M->n;
    return MSB_OK;
}
int msb_motifs_max_raw(const msb_motifs *M, double *out) {
    if (!M || !out) { set_error("null"); return MSB_EINVAL; }
    std::copy(M->max_raw.begin(), M->max_raw.end(), out);
    return MSB_OK;
}
int msb_motifs_destroy(msb_motifs *M) {
    if (!M) return MSB_OK;
    cudaSetDevice(M->ctx->device);
    cudaStreamSynchronize(M->ctx->stream);
    for (DevBuf *b : {&M->d_pwm, &M->d_col_off, &M->d_len, &M->d_cutoff, &M->d_max_raw, &M->d_pwm32, &M->d_floor32}) b->release();
    for (auto &t : M->tc_tables) {
        t.d_btab.release(); t.d_col_info.release(); t.d_len.release(); t.d_order.release(); t.d_slow.release();
    }
    delete M;
    return MSB_OK;
}

// ---- sequences ---------------------------------------------------------------------------------
// Shared by msb_seqs_from_ascii and msb_seqs_extract: lay the sequences out in the packed space
// (every sequence starts at a multiple of 32 bases), take the device buffers from the pool, upload
// the per-sequence tables and clear the code / mask planes (the kernels that read windows rely on
// zero padding behind the last block).  `seq_off` holds the n_seqs + 1 cumulative lengths.
static int seqs_prepare(msb_ctx *ctx, int64_t n_seqs, const int64_t *seq_off, msb_seqs **out,
                        std::vector<int32_t> &lens, cudaStream_t on_stream = nullptr) {
    msb_seqs *S = new (std::nothrow) msb_seqs();
    if (!S) { set_error("out of host memory"); return MSB_ENOMEM; }
    S->ctx = ctx;
    S->n = n_seqs;
    S->total_bp = seq_off[n_seqs];
    S->seq_off.assign(seq_off, seq_off + n_seqs + 1);
    S->poff.resize(n_seqs + 1);
    lens.assign((size_t) std::max<int64_t>(n_seqs, 1), 0);
    int64_t at = 0;
    int32_t min_len = n_seqs ? std::numeric_limits<int32_t>::max() : 0;
    for (int64_t i = 0; i < n_seqs; i++) {
        const int64_t len = seq_off[i + 1] - seq_off[i];
        S->poff[i] = at;
        lens[i] = (int32_t) len;
        min_len = std::min<int32_t>(min_len, (int32_t) len);
        at += (len + kPadBases - 1) / kPadBases * kPadBases;
    }
    S->poff[n_seqs] = at;
    S->total_packed = at;
    S->min_len = min_len;
    if ((uint64_t) at >= (1ull << kPosBits)) { delete S; set_error("sequence set too large"); return MSB_EINVAL; }

    int rc = MSB_OK;
    const int64_t n_blocks = at / kPadBases;
    // +8 / +4 words of zero padding: the prefilter reads up to 3 code words / 2 mask words
    // starting at the word of a thread's first window.
    if ((rc = dev_take(ctx, S->d_codes, (size_t) (2 * n_blocks + 8) * 4)) != MSB_OK ||
        (rc = dev_take(ctx, S->d_nmask, (size_t) (n_blocks + 4) * 4)) != MSB_OK ||
        (rc = dev_take(ctx, S->d_blk_seq, (size_t) std::max<int64_t>(n_blocks, 1) * 4)) != MSB_OK ||
        (rc = dev_take(ctx, S->d_poff, (size_t) (n_seqs + 1) * 8)) != MSB_OK ||
        (rc = dev_take(ctx, S->d_len, (size_t) std::max<int64_t>(n_seqs, 1) * 4)) != MSB_OK ||
        (rc = dev_take(ctx, S->d_seq_off, (size_t) (n_seqs + 1) * 8)) != MSB_OK) {
        msb_seqs_destroy(S);
        return rc;
    }
    cudaStream_t st = on_stream ? on_stream : ctx->stream;
    cudaError_t e = cudaSuccess;
    auto step = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    step(cudaMemsetAsync(S->d_codes.p, 0, (size_t) (2 * n_blocks + 8) * 4, st));
    step(cudaMemsetAsync(S->d_nmask.p, 0, (size_t) (n_blocks + 4) * 4, st));
    // the owner table comes out of the recycled pool too: msb_scan_ascii scans slice k before slice k + 1 is
    // encoded, and a position tile may reach into the next slice's blocks
    step(cudaMemsetAsync(S->d_blk_seq.p, 0, (size_t) std::max<int64_t>(n_blocks, 1) * 4, st));
    const void *h_poff = S->poff.data(), *h_seq_off = S->seq_off.data(), *h_len = lens.data();
    if (on_stream) {
        const size_t a = (size_t) (n_seqs + 1) * 8, c = (size_t) std::max<int64_t>(n_seqs, 1) * 4;
        if (pinned_get(ctx, 2 * a + c, &S->tables) == MSB_OK) {
            char *t = (char *) S->tables.p;
            std::memcpy(t, S->poff.data(), a);
            std::memcpy(t + a, S->seq_off.data(), a);
            if (n_seqs) std::memcpy(t + 2 * a, lens.data(), (size_t) n_seqs * 4);
            h_poff = t; h_seq_off = t + a; h_len = t + 2 * a;
        }
    }
    step(cudaMemcpyAsync(S->d_poff.p, h_poff, (size_t) (n_seqs + 1) * 8, cudaMemcpyHostToDevice, st));
    step(cudaMemcpyAsync(S->d_seq_off.p, h_seq_off, (size_t) (n_seqs + 1) * 8, cudaMemcpyHostToDevice, st));
    if (n_seqs) step(cudaMemcpyAsync(S->d_len.p, h_len, (size_t) n_seqs * 4, cudaMemcpyHostToDevice, st));
    if (e != cudaSuccess) {
        msb_seqs_destroy(S);
        return cuda_fail(e, "seqs_prepare", __FILE__, __LINE__);
    }
    *out = S;
    return MSB_OK;
}

int msb_seqs_from_ascii(msb_ctx *ctx, int64_t n_seqs, const char *bytes, const int64_t *seq_off,
                        msb_seqs **out) {
    if (!ctx || !out || n_seqs < 0 || !seq_off || (seq_off[n_seqs] > 0 && !bytes)) {
        set_error("msb_seqs_from_ascii: bad argument");
        return MSB_EINVAL;
    }
    *out = nullptr;
    if (seq_off[0] != 0) { set_error("seq_off[0] must be 0"); return MSB_EINVAL; }
    for (int64_t i = 0; i < n_seqs; i++) {
        const int64_t len = seq_off[i + 1] - seq_off[i];
        if (len < 0 || len > (int64_t) 0x7fffffff - 64) {
            set_error("msb_seqs_from_ascii: sequence offsets not ascending or sequence >= 2^31 bases");
            return MSB_EINVAL;
        }
    }
    MSB_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    MSB_CUDA(cudaEventRecord(ctx->ev[0], st));
    msb_seqs *S = nullptr;
    std::vector<int32_t> lens;
    MSB_TRY(seqs_prepare(ctx, n_seqs, seq_off, &S, lens));
    int rc = ctx->ascii.ensure((size_t) std::max<int64_t>(S->total_bp, 16));
    if (rc != MSB_OK) { msb_seqs_destroy(S); return rc; }
    const int64_t n_blocks = S->total_packed / kPadBases;
    cudaError_t e = cudaSuccess;
    auto step = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    if (S->total_bp) step(cudaMemcpyAsync(ctx->ascii.p, bytes, (size_t) S->total_bp, cudaMemcpyHostToDevice, st));
    step(cudaEventRecord(ctx->ev[1], st));
    if (e == cudaSuccess && n_blocks > 0) {
        const int64_t grid = (n_blocks + 255) / 256;
        encode_pack_kernel<<<(unsigned) grid, 256, 0, st>>>(
            ctx->ascii.as<uint8_t>(), S->d_seq_off.as<int64_t>(), S->d_poff.as<int64_t>(), S->d_len.as<int32_t>(),
            n_seqs, 0, n_blocks, S->d_codes.as<uint32_t>(), S->d_nmask.as<uint32_t>(), S->d_blk_seq.as<int32_t>());
        step(cudaGetLastError());
    }
    step(cudaEventRecord(ctx->ev[2], st));
    step(cudaStreamSynchronize(st));  // `bytes` and `lens` may go away after return
    if (e != cudaSuccess) {
        msb_seqs_destroy(S);
        return cuda_fail(e, "msb_seqs_from_ascii", __FILE__, __LINE__);
    }
    ctx->t[MSB_T_H2D] = ev_ms(ctx->ev[0], ctx->ev[1]);
    ctx->t[MSB_T_ENCODE] = ev_ms(ctx->ev[1], ctx->ev[2]);
    *out = S;
    return MSB_OK;
}

int msb_seqs_from_packed(msb_ctx *ctx, int64_t n_seqs, const int64_t *lens, const uint32_t *codes,
                         const uint32_t *nmask, int flags, msb_seqs **out) {
    if (!ctx || !out || n_seqs < 0 || (n_seqs > 0 && !lens)) { set_error("msb_seqs_from_packed: bad argument"); return MSB_EINVAL; }
    *out = nullptr;
    std::vector<int64_t> seq_off((size_t) n_seqs + 1, 0);
    for (int64_t i = 0; i < n_seqs; i++) {
        if (lens[i] < 0 || lens[i] > (int64_t) 0x7fffffff - 64) { set_error("msb_seqs_from_packed: sequence length out of range"); return MSB_EINVAL; }
        seq_off[i + 1] = seq_off[i] + lens[i];
    }
    if (seq_off[n_seqs] > 0 && (!codes || !nmask)) { set_error("msb_seqs_from_packed: null planes"); return MSB_EINVAL; }
    MSB_CUDA(cudaSetDevice(ctx->device));
    const bool async = (flags & MSB_SEQS_ASYNC) != 0;
    if (async) MSB_TRY(ensure_copy_stream(ctx));
    cudaStream_t st = async ? ctx->copy_stream : ctx->stream;
    if (!async) MSB_CUDA(cudaEventRecord(ctx->ev[0], st));
    msb_seqs *S = nullptr;
    {
        std::vector<int32_t> l32;
        MSB_TRY(seqs_prepare(ctx, n_seqs, seq_off.data(), &S, l32, st));
        S->lens32.swap(l32);   // seqs_prepare's copy of the lengths reads this vector: it lives as long as the set
    }
    const int64_t n_blocks = S->total_packed / kPadBases;
    cudaError_t e = cudaSuccess;
    auto step = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    if (n_blocks) {
        step(cudaMemcpyAsync(S->d_codes.p, codes, (size_t) n_blocks * 8, cudaMemcpyHostToDevice, st));
        step(cudaMemcpyAsync(S->d_nmask.p, nmask, (size_t) n_blocks * 4, cudaMemcpyHostToDevice, st));
    }
    if (!async) step(cudaEventRecord(ctx->ev[1], st));
    if (e == cudaSuccess && n_blocks > 0) {
        packed_fixup_kernel<<<(unsigned) ((n_blocks + 255) / 256), 256, 0, st>>>(
            S->d_poff.as<int64_t>(), S->d_len.as<int32_t>(), n_seqs, n_blocks, S->d_codes.as<uint32_t>(),
            S->d_nmask.as<uint32_t>(), S->d_blk_seq.as<int32_t>());
        step(cudaGetLastError());
    }
    if (async) {
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&S->ready, cudaEventDisableTiming);
        step(cudaEventRecord(S->ready, st));
        if (e == cudaSuccess) S->ready_pending = true;
    } else {
        step(cudaEventRecord(ctx->ev[2], st));
        step(cudaStreamSynchronize(st));   // the caller's planes may go away after return
    }
    if (e != cudaSuccess) { msb_seqs_destroy(S); return cuda_fail(e, "msb_seqs_from_packed", __FILE__, __LINE__); }
    if (!async) {
        ctx->t[MSB_T_H2D] = ev_ms(ctx->ev[0], ctx->ev[1]);
        ctx->t[MSB_T_ENCODE] = ev_ms(ctx->ev[1], ctx->ev[2]);
    }
    *out = S;
    return MSB_OK;
}

int msb_seqs_wait(const msb_seqs *S) {
    if (!S) { set_error("null seqs"); return MSB_EINVAL; }
    if (S->ready) { MSB_CUDA(cudaSetDevice(S->ctx->device)); MSB_CUDA(cudaEventSynchronize(S->ready)); }
    return MSB_OK;
}

int msb_seqs_to_packed(msb_ctx *ctx, const msb_seqs *S, uint32_t *codes, uint32_t *nmask) {
    if (!ctx || !S) { set_error("msb_seqs_to_packed: null"); return MSB_EINVAL; }
    const int64_t n_blocks = S->total_packed / kPadBases;
    if (n_blocks == 0) return MSB_OK;
    if (!codes || !nmask) { set_error("msb_seqs_to_packed: null planes"); return MSB_EINVAL; }
    MSB_CUDA(cudaSetDevice(ctx->device));
    MSB_TRY(seqs_ready(S));
    MSB_CUDA(cudaMemcpyAsync(codes, S->d_codes.p, (size_t) n_blocks * 8, cudaMemcpyDeviceToHost, ctx->stream));
    MSB_CUDA(cudaMemcpyAsync(nmask, S->d_nmask.p, (size_t) n_blocks * 4, cudaMemcpyDeviceToHost, ctx->stream));
    MSB_CUDA(cudaStreamSynchronize(ctx->stream));
    return MSB_OK;
}

}  // extern "C"

// msb_seqs_extract; with a substitution table (sub_off != nullptr) msb_seqs_extract_subst; with an edit table
// (ins_off != nullptr) msb_seqs_extract_edits, or with edit_off == nullptr (one edit per sequence)
// msb_seqs_extract_splice.
static int seqs_extract(msb_ctx *ctx, const msb_seqs *src, int64_t n, const int32_t *src_idx, const int64_t *start,
                        const int64_t *end, const int64_t *sub_off, const int32_t *sub_pos, const uint8_t *sub_code,
                        const int64_t *edit_off, const int32_t *edit_at, const int32_t *edit_del, const int64_t *ins_off,
                        const uint8_t *ins_code, msb_seqs **out, const char *what) {
    if (!ctx || !src || !out || n < 0 || (n > 0 && (!src_idx || !start || !end))) {
        set_error(std::string(what) + ": bad argument");
        return MSB_EINVAL;
    }
    *out = nullptr;
    if (src->ctx != ctx) { set_error(std::string(what) + ": source belongs to another context"); return MSB_EINVAL; }
    MSB_TRY(seqs_ready(src));
    // pysam's fetch (genome/__init__.py:135) clips `end` at the sequence length; an interval that
    // starts behind it, or is reversed, is empty.
    std::vector<int64_t> seq_off((size_t) n + 1, 0), clipped_start((size_t) std::max<int64_t>(n, 1), 0);
    const bool edits = ins_off != nullptr, one_each = edits && !edit_off;
    const int64_t n_edits = !edits ? 0 : one_each ? n : edit_off[n], n_ins = edits ? ins_off[n_edits] : 0;
    if (edits && ((edit_off && edit_off[0] != 0) || ins_off[0] != 0 || (n_edits > 0 && (!edit_at || !edit_del)) ||
                  (n_ins > 0 && !ins_code))) {
        set_error(std::string(what) + ": bad edit table");
        return MSB_EINVAL;
    }
    // where each edit's bases land (one edit per sequence: at its own start, edit_at)
    std::vector<int32_t> edit_dst((size_t) (one_each ? 0 : std::max<int64_t>(n_edits, 1)));
    for (int64_t i = 0; i < n; i++) {
        if (src_idx[i] < 0 || src_idx[i] >= src->n) { set_error(std::string(what) + ": source index out of range"); return MSB_EINVAL; }
        if (start[i] < 0) { set_error(std::string(what) + ": negative start"); return MSB_EINVAL; }
        const int64_t slen = src->seq_off[src_idx[i] + 1] - src->seq_off[src_idx[i]];
        const int64_t a = std::min(start[i], slen), b = std::min(end[i], slen);
        int64_t len = std::max<int64_t>(b - a, 0);
        if (edits) {
            // the cut interval loses each edit's [at, at + del) and gains its inserted bases there
            const int64_t e0 = one_each ? i : edit_off[i], e1 = one_each ? i + 1 : edit_off[i + 1];
            if (e1 < e0) { set_error(std::string(what) + ": edit offsets not ascending"); return MSB_EINVAL; }
            const int64_t ilen = len;
            for (int64_t k = e0; k < e1; k++) {
                if (ins_off[k + 1] < ins_off[k]) { set_error(std::string(what) + ": insertion offsets not ascending"); return MSB_EINVAL; }
                if (edit_at[k] < 0 || edit_del[k] < 0 || (int64_t) edit_at[k] + edit_del[k] > ilen) {
                    set_error(std::string(what) + ": edit outside its interval");
                    return MSB_EINVAL;
                }
                if (k > e0) {
                    // an insertion occupies its junction: the next edit starts behind at + max(del, 1)
                    if (edit_at[k] < edit_at[k - 1]) { set_error(std::string(what) + ": edits out of order"); return MSB_EINVAL; }
                    if (edit_at[k] < edit_at[k - 1] + std::max(edit_del[k - 1], 1)) {
                        set_error(std::string(what) + ": edits overlap");
                        return MSB_EINVAL;
                    }
                }
                if (!one_each) edit_dst[(size_t) k] = (int32_t) (edit_at[k] + (len - ilen));
                len += ins_off[k + 1] - ins_off[k] - edit_del[k];
                if (len > (int64_t) 0x7fffffff - 64) { set_error(std::string(what) + ": edited sequence >= 2^31 bases"); return MSB_EINVAL; }
            }
        }
        clipped_start[i] = a;
        seq_off[i + 1] = seq_off[i] + len;
    }
    for (int64_t k = 0; k < n_ins; k++)
        if (ins_code[k] > 3) { set_error(std::string(what) + ": inserted base not an A/C/G/T code"); return MSB_EINVAL; }
    const int64_t n_sub = sub_off ? sub_off[n] : 0;
    if (sub_off) {
        if (sub_off[0] != 0 || (n_sub > 0 && (!sub_pos || !sub_code))) { set_error(std::string(what) + ": bad substitution table"); return MSB_EINVAL; }
        for (int64_t i = 0; i < n; i++) {
            if (sub_off[i + 1] < sub_off[i]) { set_error(std::string(what) + ": substitution offsets not ascending"); return MSB_EINVAL; }
            for (int64_t k = sub_off[i]; k < sub_off[i + 1]; k++)
                if (sub_pos[k] < 0 || sub_pos[k] >= seq_off[i + 1] - seq_off[i] || sub_code[k] > 3) {
                    set_error(std::string(what) + ": substitution outside its sequence or not an A/C/G/T code");
                    return MSB_EINVAL;
                }
        }
    }
    MSB_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    MSB_CUDA(cudaEventRecord(ctx->ev[0], st));
    msb_seqs *S = nullptr;
    std::vector<int32_t> lens;
    MSB_TRY(seqs_prepare(ctx, n, seq_off.data(), &S, lens));
    // the tables ride in the (otherwise unused here) ASCII scratch:
    // src_idx (4n) | start (8n) [| sub_off (8 (n + 1)) | sub_pos (4 n_sub) | sub_code (n_sub)]
    //                           [| edit_off (8 (n + 1)) | edit_at, edit_del, edit_dst (4 n_edits each)
    //                            | ins_off (8 (n_edits + 1)) | ins_code (n_ins)]; one edit per sequence: no
    //                            edit_off, and edit_dst is edit_at
    auto al = [](size_t x) { return (x + 15) & ~(size_t) 15; };
    const size_t o_start = al((size_t) n * 4), o_soff = o_start + al((size_t) n * 8);
    const size_t o_spos = o_soff + al((size_t) (n + 1) * 8), o_scode = o_spos + al((size_t) n_sub * 4);
    const size_t o_eoff = o_soff, o_at = o_eoff + al((size_t) (n + 1) * 8), o_del = o_at + al((size_t) n_edits * 4);
    const size_t o_dst = o_del + al((size_t) n_edits * 4), o_ioff = o_dst + al((size_t) n_edits * 4);
    const size_t o_icode = o_ioff + al((size_t) (n_edits + 1) * 8);
    const size_t bytes = sub_off ? o_scode + (size_t) n_sub : edits ? o_icode + (size_t) n_ins : o_start + (size_t) n * 8;
    int rc = ctx->ascii.ensure(std::max<size_t>(bytes, 16));
    if (rc != MSB_OK) { msb_seqs_destroy(S); return rc; }
    char *base = (char *) ctx->ascii.p;
    const int64_t n_blocks = S->total_packed / kPadBases;
    cudaError_t e = cudaSuccess;
    auto step = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    if (n) {
        step(cudaMemcpyAsync(base, src_idx, (size_t) n * 4, cudaMemcpyHostToDevice, st));
        step(cudaMemcpyAsync(base + o_start, clipped_start.data(), (size_t) n * 8, cudaMemcpyHostToDevice, st));
    }
    if (sub_off) {
        step(cudaMemcpyAsync(base + o_soff, sub_off, (size_t) (n + 1) * 8, cudaMemcpyHostToDevice, st));
        if (n_sub) {
            step(cudaMemcpyAsync(base + o_spos, sub_pos, (size_t) n_sub * 4, cudaMemcpyHostToDevice, st));
            step(cudaMemcpyAsync(base + o_scode, sub_code, (size_t) n_sub, cudaMemcpyHostToDevice, st));
        }
    }
    if (edits) {
        if (!one_each) step(cudaMemcpyAsync(base + o_eoff, edit_off, (size_t) (n + 1) * 8, cudaMemcpyHostToDevice, st));
        if (n_edits) {
            step(cudaMemcpyAsync(base + o_at, edit_at, (size_t) n_edits * 4, cudaMemcpyHostToDevice, st));
            step(cudaMemcpyAsync(base + o_del, edit_del, (size_t) n_edits * 4, cudaMemcpyHostToDevice, st));
            if (!one_each)
                step(cudaMemcpyAsync(base + o_dst, edit_dst.data(), (size_t) n_edits * 4, cudaMemcpyHostToDevice, st));
        }
        step(cudaMemcpyAsync(base + o_ioff, ins_off, (size_t) (n_edits + 1) * 8, cudaMemcpyHostToDevice, st));
        if (n_ins) step(cudaMemcpyAsync(base + o_icode, ins_code, (size_t) n_ins, cudaMemcpyHostToDevice, st));
    }
    step(cudaEventRecord(ctx->ev[1], st));
    if (e == cudaSuccess && n_blocks > 0) {
        const int64_t grid = (n_blocks + 255) / 256;
        if (sub_off)
            extract_subst_kernel<<<(unsigned) grid, 256, 0, st>>>(
                src->view(), (const int32_t *) base, (const int64_t *) (base + o_start), (const int64_t *) (base + o_soff),
                (const int32_t *) (base + o_spos), (const uint8_t *) (base + o_scode), S->d_poff.as<int64_t>(),
                S->d_len.as<int32_t>(), n, n_blocks, S->d_codes.as<uint32_t>(), S->d_nmask.as<uint32_t>(),
                S->d_blk_seq.as<int32_t>());
        else if (edits)
            extract_edits_kernel<<<(unsigned) grid, 256, 0, st>>>(
                src->view(), (const int32_t *) base, (const int64_t *) (base + o_start),
                one_each ? nullptr : (const int64_t *) (base + o_eoff), (const int32_t *) (base + o_at),
                (const int32_t *) (base + o_del), (const int32_t *) (base + (one_each ? o_at : o_dst)),
                (const int64_t *) (base + o_ioff), (const uint8_t *) (base + o_icode), S->d_poff.as<int64_t>(),
                S->d_len.as<int32_t>(), n, n_blocks, S->d_codes.as<uint32_t>(), S->d_nmask.as<uint32_t>(),
                S->d_blk_seq.as<int32_t>());
        else
            extract_pack_kernel<<<(unsigned) grid, 256, 0, st>>>(
                src->view(), (const int32_t *) base, (const int64_t *) (base + o_start), S->d_poff.as<int64_t>(),
                S->d_len.as<int32_t>(), n, n_blocks, S->d_codes.as<uint32_t>(), S->d_nmask.as<uint32_t>(),
                S->d_blk_seq.as<int32_t>());
        step(cudaGetLastError());
    }
    step(cudaEventRecord(ctx->ev[2], st));
    step(cudaStreamSynchronize(st));  // host tables go out of scope
    if (e != cudaSuccess) {
        msb_seqs_destroy(S);
        return cuda_fail(e, what, __FILE__, __LINE__);
    }
    ctx->t[MSB_T_H2D] = ev_ms(ctx->ev[0], ctx->ev[1]);
    ctx->t[MSB_T_ENCODE] = ev_ms(ctx->ev[1], ctx->ev[2]);
    *out = S;
    return MSB_OK;
}

extern "C" {

int msb_seqs_extract(msb_ctx *ctx, const msb_seqs *src, int64_t n, const int32_t *src_idx,
                     const int64_t *start, const int64_t *end, msb_seqs **out) {
    return seqs_extract(ctx, src, n, src_idx, start, end, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                        nullptr, out, "msb_seqs_extract");
}

int msb_seqs_extract_subst(msb_ctx *ctx, const msb_seqs *src, int64_t n, const int32_t *src_idx, const int64_t *start,
                           const int64_t *end, const int64_t *sub_off, const int32_t *sub_pos, const uint8_t *sub_code,
                           msb_seqs **out) {
    if (!sub_off) { set_error("msb_seqs_extract_subst: null substitution offsets"); return MSB_EINVAL; }
    return seqs_extract(ctx, src, n, src_idx, start, end, sub_off, sub_pos, sub_code, nullptr, nullptr, nullptr, nullptr,
                        nullptr, out, "msb_seqs_extract_subst");
}

int msb_seqs_extract_splice(msb_ctx *ctx, const msb_seqs *src, int64_t n, const int32_t *src_idx, const int64_t *start,
                            const int64_t *end, const int32_t *splice_at, const int32_t *del_len, const int64_t *ins_off,
                            const uint8_t *ins_code, msb_seqs **out) {
    if (!ins_off) { set_error("msb_seqs_extract_splice: null insertion offsets"); return MSB_EINVAL; }
    // one edit per sequence (edit_off == nullptr)
    return seqs_extract(ctx, src, n, src_idx, start, end, nullptr, nullptr, nullptr, nullptr, splice_at, del_len,
                        ins_off, ins_code, out, "msb_seqs_extract_splice");
}

int msb_seqs_extract_edits(msb_ctx *ctx, const msb_seqs *src, int64_t n, const int32_t *src_idx, const int64_t *start,
                           const int64_t *end, const int64_t *edit_off, const int32_t *edit_at, const int32_t *edit_del,
                           const int64_t *ins_off, const uint8_t *ins_code, msb_seqs **out) {
    if (!edit_off || !ins_off) { set_error("msb_seqs_extract_edits: null edit offsets"); return MSB_EINVAL; }
    return seqs_extract(ctx, src, n, src_idx, start, end, nullptr, nullptr, nullptr, edit_off, edit_at, edit_del, ins_off,
                        ins_code, out, "msb_seqs_extract_edits");
}

int msb_seqs_window_ncount(msb_ctx *ctx, const msb_seqs *src, int64_t n, const int32_t *src_idx, const int64_t *start,
                           int32_t length, int32_t *counts) {
    if (!ctx || !src || n < 0 || length < 0 || (n > 0 && (!src_idx || !start || !counts))) {
        set_error("msb_seqs_window_ncount: bad argument");
        return MSB_EINVAL;
    }
    if (src->ctx != ctx) { set_error("msb_seqs_window_ncount: source belongs to another context"); return MSB_EINVAL; }
    MSB_TRY(seqs_ready(src));
    for (int64_t i = 0; i < n; i++)
        if (src_idx[i] < 0 || src_idx[i] >= src->n || start[i] < 0) { set_error("msb_seqs_window_ncount: window out of range"); return MSB_EINVAL; }
    if (n == 0) return MSB_OK;
    MSB_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    // tables ride in the ASCII scratch: src_idx (4n) | start (8n) | counts (4n)
    const size_t a_off = ((size_t) n * 4 + 15) & ~(size_t) 15, c_off = a_off + (((size_t) n * 8 + 15) & ~(size_t) 15);
    MSB_TRY(ctx->ascii.ensure(c_off + (size_t) n * 4));
    char *base = (char *) ctx->ascii.p;
    MSB_CUDA(cudaMemcpyAsync(base, src_idx, (size_t) n * 4, cudaMemcpyHostToDevice, st));
    MSB_CUDA(cudaMemcpyAsync(base + a_off, start, (size_t) n * 8, cudaMemcpyHostToDevice, st));
    window_ncount_kernel<<<(unsigned) ((n + 255) / 256), 256, 0, st>>>(src->view(), (const int32_t *) base, (const int64_t *) (base + a_off),
                                                                      length, n, (int32_t *) (base + c_off));
    MSB_CUDA(cudaGetLastError());
    MSB_CUDA(cudaMemcpyAsync(counts, base + c_off, (size_t) n * 4, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaStreamSynchronize(st));
    return MSB_OK;
}

int msb_seqs_lengths(const msb_seqs *S, int64_t *lens) {
    if (!S || (!lens && S->n)) { set_error("msb_seqs_lengths: null"); return MSB_EINVAL; }
    for (int64_t i = 0; i < S->n; i++) lens[i] = S->seq_off[i + 1] - S->seq_off[i];
    return MSB_OK;
}

int msb_seqs_set_start_limit(msb_seqs *S, const int32_t *limit) {
    if (!S) { set_error("null seqs"); return MSB_EINVAL; }
    if (!limit || S->n == 0) { S->has_limit = false; return MSB_OK; }
    for (int64_t i = 0; i < S->n; i++)
        if (limit[i] < 0) { set_error("msb_seqs_set_start_limit: negative limit"); return MSB_EINVAL; }
    MSB_CUDA(cudaSetDevice(S->ctx->device));
    MSB_TRY(S->d_limit.ensure((size_t) S->n * 4));
    MSB_CUDA(cudaMemcpyAsync(S->d_limit.p, limit, (size_t) S->n * 4, cudaMemcpyHostToDevice, S->ctx->stream));
    MSB_CUDA(cudaStreamSynchronize(S->ctx->stream));
    S->has_limit = true;
    return MSB_OK;
}

int msb_seqs_count(const msb_seqs *S, int64_t *n_seqs, int64_t *total_bp) {
    if (!S) { set_error("null seqs"); return MSB_EINVAL; }
    if (n_seqs) *n_seqs = S->n;
    if (total_bp) *total_bp = S->total_bp;
    return MSB_OK;
}

int msb_seqs_codes(msb_ctx *ctx, const msb_seqs *S, int8_t *codes) {
    if (!ctx || !S || (!codes && S->total_bp)) { set_error("msb_seqs_codes: null"); return MSB_EINVAL; }
    if (S->total_bp == 0) return MSB_OK;
    MSB_CUDA(cudaSetDevice(ctx->device));
    MSB_TRY(seqs_ready(S));
    DevBuf tmp;
    MSB_TRY(tmp.ensure((size_t) S->total_bp));
    const int64_t grid = (S->total_packed + 255) / 256;
    unpack_codes_kernel<<<(unsigned) grid, 256, 0, ctx->stream>>>(S->view(), S->d_seq_off.as<int64_t>(), tmp.as<int8_t>());
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(codes, tmp.p, (size_t) S->total_bp, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    tmp.release();
    if (e != cudaSuccess) return cuda_fail(e, "msb_seqs_codes", __FILE__, __LINE__);
    return MSB_OK;
}

int msb_seqs_destroy(msb_seqs *S) {
    if (!S) return MSB_OK;
    cudaSetDevice(S->ctx->device);
    if (S->ready) { cudaEventSynchronize(S->ready); cudaEventDestroy(S->ready); }
    cudaStreamSynchronize(S->ctx->stream);
    for (DevBuf *b : {&S->d_codes, &S->d_nmask, &S->d_poff, &S->d_len, &S->d_seq_off, &S->d_blk_seq, &S->d_limit}) dev_give(S->ctx, *b);
    pinned_put(S->ctx, S->tables);
    delete S;
    return MSB_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// Prefilter tables (prefilter_tc.cuh).
//
// For one strand of motif m let V[b][c] be its PWM (forward: M[b][c], cscore.c:348; reverse:
// M[3-b][L-1-c], cscore.c:351), colmax_c = max_b V[b][c] and d[b][c] = colmax_c - V[b][c] >= 0 the
// "deficit" of base b at column c, so that  raw = sum_c colmax_c - sum_c d[b_c][c].  The raw threshold
// T is a strict under-estimate of the smallest exact raw score the reference could accept:
//     score/max_raw - cutoff >= -1e-10  (evaluated in double, cscore.c:357-358)
//     =>  raw >= T = max_raw * (cutoff - 1e-10) - 1e-12 * (max_raw * (|cutoff| + 1) + sum_c max_b |M[b][c]|)
// (the 1e-12 term is > 1000x the worst-case rounding of the L-term double sum, the division
// and the subtraction).  A window the reference can accept therefore has
//     sum_c d[b_c][c]  <=  D = sum_c colmax_c - T (+ slack for the rounding of these host sums).
// (For a motif longer than kMaxFastLen, colmax_c of a column behind the first kMaxFastLen is replaced by
// max(colmax_c, 0): an N there adds 0; see tc_fill_column.)
// The stored e4m3 entries are  e[b][c] = RU( beta - s * d[b][c] )  (rounded towards +inf, floored
// at -448), with beta an e4m3 value, C = L * beta and s = (C - C/64) / D.  Then for every window
// with sum d <= D:   sum_c e >= C - s * sum d >= C/64 > 5,  more than the tensor core's f16
// accumulation can lose (prefilter_tc.cuh), so the accumulator's sign bit is clear: the candidates
// are a superset of the reference's hits.
// ------------------------------------------------------------------------------------------------
namespace msb {

// Motifs the prefilter can take: up to kMaxTcLen columns.  It looks at the first kMaxFastLen columns of a
// strand only (tc_fill_column), the exact stage scores the whole window, and the producer's all-N test spans
// kMaxTcLen bases.
static bool motif_is_fast(const msb_motifs *M, int32_t m) {
    const int L = M->lens[m];
    if (L < 1 || L > kMaxTcLen) return false;
    const double *mat = M->mats.data() + M->mat_off[m];
    for (int k = 0; k < 4 * L; k++)
        if (!std::isfinite(mat[k])) return false;
    return true;
}

static float e4m3_value(int v) {
    const int e = (v >> 3) & 15, m = v & 7;
    const float mag = e == 0 ? std::ldexp((float) m / 8.f, -6) : std::ldexp(1.f + (float) m / 8.f, e - 7);
    return (v & 0x80) ? -mag : mag;
}
// smallest e4m3 value >= x, saturating at +-448; never the byte 0x80 (-0)
static uint8_t e4m3_round_up(double x) {
    static const std::vector<double> mag = [] {     // the 127 non-negative magnitudes, ascending
        std::vector<double> v(0x7F);
        for (int i = 0; i < 0x7F; i++) v[i] = (double) e4m3_value(i);
        return v;
    }();
    if (!(x > -448.0)) return 0xFE;  // -448 (also NaN -> most negative: cannot create candidates)
    if (x > 448.0) return 0x7E;
    if (x <= 0) {
        // largest magnitude <= |x| among the negatives, i.e. round towards zero
        const int best = (int) (std::upper_bound(mag.begin(), mag.end(), -x) - mag.begin()) - 1;
        return best <= 0 ? 0x00 : (uint8_t) (0x80 | best);
    }
    const int v = (int) (std::lower_bound(mag.begin(), mag.end(), x) - mag.begin());
    return v >= 0x7F ? 0x7E : (uint8_t) v;
}

static inline size_t tc_byte(int ks_idx, int col, int k_in_step) {
    return (size_t) ks_idx * kTcUnitBytes + (size_t) (k_in_step >> 4) * 4096 + (size_t) col * 16 + (size_t) (k_in_step & 15);
}

static void tc_fill_never(uint8_t *tile, int col) {
    for (int b = 0; b < 4; b++) tile[tc_byte(0, col, b)] = 0xFE;  // any ACGT base at offset 0: -448
}

static void tc_fill_column(const msb_motifs *M, int32_t m, int rev, uint8_t *tile, int col) {
    const int L = M->lens[m];
    const double *mat = M->mats.data() + M->mat_off[m];
    auto V = [&](int b, int c) { return rev ? mat[(size_t) (3 - b) * L + (L - 1 - c)] : mat[(size_t) b * L + c]; };
    const double max_raw = M->max_raw[m];
    const double cutoff = M->cutoffs[m];
    if (!(max_raw > 0) || std::isnan(cutoff) || (std::isinf(cutoff) && cutoff > 0)) { tc_fill_never(tile, col); return; }
    // A motif longer than kMaxFastLen columns is prefiltered on its first kMaxFastLen columns (of this strand)
    // alone.  An N anywhere in those columns makes the window dirty (the producer's horizon), so on this path
    // they hold A/C/G/T.  A column behind them may hold an N, which adds 0 (cscore.c:346): such a column
    // contributes at most max(colmax_c, 0), more than colmax_c when all four entries are negative.  So the
    // budget below takes colmax_c for the kept columns and max(colmax_c, 0) for the others; then the sum over
    // the kept columns of d <= D for every window the reference accepts, whatever sits behind them.
    const int kept = std::min(L, kMaxFastLen);
    double cms = 0, abs_sum = 0;
    std::vector<double> colmax((size_t) L);
    for (int c = 0; c < L; c++) {
        double mx = -INFINITY, a = 0;
        for (int b = 0; b < 4; b++) { mx = std::max(mx, V(b, c)); a = std::max(a, std::fabs(V(b, c))); }
        colmax[c] = mx;
        cms += c < kept ? mx : std::max(mx, 0.0);
        abs_sum += a;
    }
    double D;
    if (std::isinf(cutoff)) {
        D = INFINITY;  // -inf: every window with a finite score is a site
    } else {
        const double T = max_raw * (cutoff - 1e-10) - 1e-12 * (max_raw * (std::fabs(cutoff) + 1.0) + abs_sum);
        D = cms - T;
        D += 1e-12 * (std::fabs(cms) + std::fabs(T) + abs_sum);
        if (D < 0) { tc_fill_never(tile, col); return; }  // even the best window is below the cutoff
    }
    // beta: an e4m3 value near 384 / kept (exactly representable, so the all-best window sums to C)
    const double beta = (double) e4m3_value(e4m3_round_up(384.0 / kept));
    const double C = beta * kept;
    double s = std::isinf(D) ? 0.0 : (C - C / 64.0) / std::max(D, 1e-300);
    if (!(s < 1e30)) s = 1e30;
    for (int c = 0; c < kept; c++)
        for (int b = 0; b < 4; b++) {
            const double d = colmax[c] - V(b, c);
            const double x = d > 0 ? beta - s * d : beta;
            const int k = 4 * c + b;
            tile[tc_byte(k >> 5, col, k & 31)] = e4m3_round_up(x);
        }
}

static int ensure_tc_tables(msb_ctx *ctx, msb_motifs *M, int strand, TcTableSet **out) {
    TcTableSet &T = M->tc_tables[strand];
    if (T.valid && T.cutoff_version == M->cutoff_version) { *out = &T; return MSB_OK; }
    T.valid = false;
    T.order.clear();
    T.slow.clear();
    T.batches.clear();
    T.lmax_fast = 0;
    T.any_zero_hit = 0;
    std::vector<int32_t> fast;
    for (int32_t m = 0; m < M->n; m++) {
        if (motif_is_fast(M, m)) fast.push_back(m);
        else if (M->lens[m] >= 1) T.slow.push_back(m);
    }
    auto ksteps = [&](int32_t m) { return (std::min(M->lens[m], kMaxFastLen) + 7) / 8; };
    std::stable_sort(fast.begin(), fast.end(), [&](int32_t a, int32_t b) { return M->lens[a] < M->lens[b]; });
    const int cols_per_motif = strand == 3 ? 2 : 1;
    const int motifs_per_tile = kTcCols / cols_per_motif;
    const size_t n_tiles = (fast.size() + motifs_per_tile - 1) / motifs_per_tile;
    if (ctx->opt_tc_interleave && n_tiles > 2) {
        // Tile order.  Sorted by length the tiles' K steps ascend (750 motifs: 2 2 3 3 4 4).  An epilogue warp set
        // has the duration of its unit's MMAs plus the next unit's to get through a unit (the two TMEM buffers
        // alternate), and its work per unit does not depend on K: next to each other the two short tiles leave it
        // 4 K steps of time, the long ones 8.  Short and long tiles alternate instead (2 4 2 3 3 4: never fewer than 5);
        // the last, possibly partial, tile stays last.
        const size_t n_full = fast.size() / motifs_per_tile;
        std::vector<int32_t> mixed;
        mixed.reserve(fast.size());
        size_t lo = 0, hi = n_full;
        for (size_t i = 0; lo < hi; i++) {
            const size_t g = (i & 1) ? --hi : lo++;
            mixed.insert(mixed.end(), fast.begin() + g * motifs_per_tile, fast.begin() + (g + 1) * motifs_per_tile);
        }
        mixed.insert(mixed.end(), fast.begin() + n_full * motifs_per_tile, fast.end());
        fast.swap(mixed);
    }
    T.order = fast;
    std::vector<uint32_t> col_info(std::max<size_t>(n_tiles, 1) * kTcCols, 0xffffffffu);
    std::vector<int32_t> tc_len(std::max<size_t>(fast.size(), 1), 0);
    std::vector<uint8_t> btab;
    const uint32_t max_units = kTcMaxUnits;
    TcBatch cur;
    std::memset(&cur, 0, sizeof(cur));
    uint32_t cur_units = 0;
    for (size_t t = 0; t < n_tiles; t++) {
        const size_t k0 = t * motifs_per_tile, k1 = std::min(fast.size(), k0 + motifs_per_tile);
        int ks = 1;
        for (size_t k = k0; k < k1; k++) ks = std::max(ks, ksteps(fast[k]));
        if (cur.n_tiles == kTcMaxTiles || cur_units + ks > max_units) {
            T.batches.push_back(cur);
            std::memset(&cur, 0, sizeof(cur));
            cur_units = 0;
        }
        if (cur.n_tiles == 0) { cur.b_off = (uint32_t) btab.size(); cur.first_tile = (uint32_t) t; }
        cur.ks[cur.n_tiles] = (uint8_t) ks;
        cur.unit_off[cur.n_tiles] = (uint8_t) cur_units;
        cur.n_tiles++;
        cur_units += ks;
        cur.b_bytes = cur_units * kTcUnitBytes;
        const size_t base = btab.size();
        btab.resize(base + (size_t) ks * kTcUnitBytes, 0);
        uint8_t *tile = btab.data() + base;
        for (int col = 0; col < kTcCols; col++) {
            const size_t k = k0 + (size_t) (col / cols_per_motif);
            if (k >= k1) { tc_fill_never(tile, col); continue; }
            const int32_t m = fast[k];
            const int rev = strand == 3 ? (col & 1) : (strand == 2 ? 1 : 0);
            tc_fill_column(M, m, rev, tile, col);
            col_info[t * kTcCols + col] = ((uint32_t) k << 1) | (uint32_t) rev;
        }
        for (size_t k = k0; k < k1; k++) {
            const int32_t m = fast[k];
            tc_len[k] = M->lens[m];
            T.lmax_fast = std::max(T.lmax_fast, M->lens[m]);
            // all-N window: score = 0 / max_raw (cscore.c:342-357 with every base skipped)
            const double z = 0.0 / M->max_raw[m];
            if (z - M->cutoffs[m] >= -1e-10) T.any_zero_hit = 1;
        }
    }
    if (cur.n_tiles) T.batches.push_back(cur);
    if (btab.empty()) btab.resize(16, 0);
    MSB_TRY(T.d_btab.ensure(btab.size()));
    MSB_TRY(T.d_col_info.ensure(col_info.size() * 4));
    MSB_TRY(T.d_len.ensure(tc_len.size() * 4));
    MSB_TRY(T.d_order.ensure(std::max<size_t>(fast.size() * 4, 16)));
    MSB_TRY(T.d_slow.ensure(std::max<size_t>(T.slow.size() * 4, 16)));
    cudaStream_t st = ctx->stream;
    MSB_CUDA(cudaMemcpyAsync(T.d_btab.p, btab.data(), btab.size(), cudaMemcpyHostToDevice, st));
    MSB_CUDA(cudaMemcpyAsync(T.d_col_info.p, col_info.data(), col_info.size() * 4, cudaMemcpyHostToDevice, st));
    MSB_CUDA(cudaMemcpyAsync(T.d_len.p, tc_len.data(), tc_len.size() * 4, cudaMemcpyHostToDevice, st));
    if (!fast.empty()) MSB_CUDA(cudaMemcpyAsync(T.d_order.p, fast.data(), fast.size() * 4, cudaMemcpyHostToDevice, st));
    if (!T.slow.empty()) MSB_CUDA(cudaMemcpyAsync(T.d_slow.p, T.slow.data(), T.slow.size() * 4, cudaMemcpyHostToDevice, st));
    MSB_CUDA(cudaStreamSynchronize(st));
    T.cutoff_version = M->cutoff_version;
    T.valid = true;
    *out = &T;
    return MSB_OK;
}

static int read_counters(msb_ctx *ctx) {
    MSB_CUDA(cudaMemcpyAsync(ctx->h_counters, ctx->counters.p, 4 * sizeof(unsigned long long),
                             cudaMemcpyDeviceToHost, ctx->stream));
    MSB_CUDA(cudaStreamSynchronize(ctx->stream));
    return MSB_OK;
}

static int launch_positions(msb_ctx *ctx, const ExactParams &E, const int64_t *pos, int64_t n_pos, int64_t pos_base,
                            const int32_t *ids, int32_t n_ids) {
    // one thread per (position, motif); split so that a launch stays below 2^31 blocks
    if (n_pos <= 0 || n_ids <= 0) return MSB_OK;
    const int64_t max_threads = (int64_t) 1 << 38;
    const int64_t pos_per_launch = std::max<int64_t>(1, max_threads / n_ids);
    for (int64_t at = 0; at < n_pos; at += pos_per_launch) {
        const int64_t cnt = std::min(pos_per_launch, n_pos - at);
        const int64_t threads = cnt * n_ids;
        ExactParams e2 = E;
        if (pos) {
            exact_positions_kernel<<<(unsigned) ((threads + 255) / 256), 256, 0, ctx->stream>>>(e2, pos + at, cnt, 0, ids, n_ids);
        } else {
            // pos == nullptr: the packed position is pos_base + the thread's position index
            exact_positions_kernel<<<(unsigned) ((threads + 255) / 256), 256, 0, ctx->stream>>>(e2, nullptr, cnt, pos_base + at, ids, n_ids);
        }
        MSB_CUDA(cudaGetLastError());
        ctx->c[MSB_C_LAUNCHES]++;
    }
    return MSB_OK;
}

// Packed-position ranges [lo, hi) of a range scan; nullptr = the whole sequence set.
typedef std::vector<std::pair<int64_t, int64_t>> RangeList;

static int make_ranges(const msb_seqs *S, int64_t n_ranges, const int64_t *r_seq, const int64_t *r_start,
                       const int64_t *r_end, RangeList *out) {
    if (n_ranges < 0 || (n_ranges > 0 && (!r_seq || !r_start || !r_end))) { set_error("msb_scan_ranges: bad ranges"); return MSB_EINVAL; }
    out->clear();
    for (int64_t i = 0; i < n_ranges; i++) {
        if (r_seq[i] < 0 || r_seq[i] >= S->n) { set_error("msb_scan_ranges: sequence index out of range"); return MSB_EINVAL; }
        if (r_start[i] < 0) { set_error("msb_scan_ranges: negative start"); return MSB_EINVAL; }
        const int64_t slen = S->seq_off[r_seq[i] + 1] - S->seq_off[r_seq[i]];
        const int64_t a = std::min(r_start[i], slen), b = std::min(r_end[i], slen);
        if (b > a) out->push_back({S->poff[r_seq[i]] + a, S->poff[r_seq[i]] + b});
    }
    std::sort(out->begin(), out->end());
    for (size_t i = 1; i < out->size(); i++)
        if ((*out)[i].first < (*out)[i - 1].second) { set_error("msb_scan_ranges: ranges overlap"); return MSB_EINVAL; }
    return MSB_OK;
}

// `before_range(k)`: called on the host right before the prefilter launches of range k are enqueued
// (msb_scan_ascii makes the stream wait for that slice's bytes and encodes them there).
typedef std::function<int(size_t)> RangeHook;

// `limit_override`: a device array of per-sequence start limits used instead of the set's own
// (msb_score_select scans only the offset-0 window of every sample); `cand_scale`: the candidate buffers
// are sized for that many times the usual candidate density.
// `boundary`: with MSB_SCAN_DEDUP, also collect the boundary chains of every range (boundary_chains_kernel).
static int scan_device(msb_ctx *ctx, msb_motifs *M, const msb_seqs *S, int strand, int flags,
                       const RangeList *ranges = nullptr, const RangeHook *before_range = nullptr,
                       const int32_t *limit_override = nullptr, int cand_scale = 1, bool boundary = false) {
    if (!ctx || !M || !S) { set_error("msb_scan: null argument"); return MSB_EINVAL; }
    if (strand < 1 || strand > 3) { set_error("msb_scan: strand must be 1, 2 or 3"); return MSB_EINVAL; }
    if (M->ctx != ctx || S->ctx != ctx) { set_error("msb_scan: motifs/seqs belong to another context"); return MSB_EINVAL; }
    MSB_CUDA(cudaSetDevice(ctx->device));
    MSB_TRY(seqs_ready(S));
    RangeList whole;
    if (!ranges) {
        if (S->total_packed) whole.push_back({0, S->total_packed});
        ranges = &whole;
    }
    int64_t span = 0;
    for (auto &r : *ranges) span += r.second - r.first;
    TcTableSet *TT = nullptr;
    MSB_TRY(ensure_tc_tables(ctx, M, strand, &TT));
    const int32_t n_fast = (int32_t) TT->order.size();
    const int32_t n_slow = (int32_t) TT->slow.size();
    const int32_t *d_order = TT->d_order.as<int32_t>();
    const int32_t *d_slow = TT->d_slow.as<int32_t>();
    cudaStream_t st = ctx->stream;
    std::fill(ctx->c, ctx->c + MSB_C_COUNT, 0);
    ctx->last_sites = 0;
    ctx->last_n_motifs = M->n;
    ctx->last_n_seqs = S->n;
    boundary = boundary && (flags & MSB_SCAN_DEDUP);
    ctx->last_boundary = boundary ? 0 : -1;
    ctx->last_variant_rows = -1;
    // this scan's final arrays go to the set the previous scan did not use; a copy that still reads it
    // (an asynchronous result two scans back) is waited for on the device, not on the host
    const int fin_set = ctx->fin_cur ^ 1;
    msb_ctx::FinSet &F = ctx->fin[fin_set];
    if (F.pending) { MSB_CUDA(cudaStreamWaitEvent(st, F.read_done, 0)); F.pending = false; }
    const bool counts_only = (flags & MSB_SCAN_COUNTS) && !(flags & MSB_SCAN_DEDUP);
    ctx->last_compact = false;
    ctx->last_seqs = S;
    MSB_TRY(F.offsets.ensure((size_t) (M->n + 1) * 8));  // CSR offsets over motifs
    MSB_CUDA(cudaMemsetAsync(F.offsets.p, 0, (size_t) (M->n + 1) * 8, st));
    ctx->fin_key = nullptr;
    if (M->n == 0 || span == 0) {
        MSB_CUDA(cudaStreamSynchronize(st));
        ctx->fin_cur = fin_set;
        ctx->last_counts_only = counts_only;
        return MSB_OK;
    }
    SeqView sv = S->view();
    if (limit_override) sv.limit = limit_override;
    const MotifView mv = M->view();
    // site key = motif << key_shift | packed position << 1 | strand (make_site_key)
    int pos_bits = 1, motif_bits = 1;
    while ((1ll << pos_bits) < S->total_packed) pos_bits++;
    while ((1ll << motif_bits) < (int64_t) M->n) motif_bits++;
    const int key_shift = pos_bits + 1;
    ctx->last_key_shift = key_shift;

    // ---- stage 1: prefilter ------------------------------------------------------------------
    const double cells = (double) span * (double) std::max<int32_t>(n_fast, 1);
    int64_t cand_cap = (int64_t) std::min<double>(std::max<double>(cells / 512.0 * cand_scale, 1 << 22), (double) (1ll << 30));   // in 8-byte units
    int64_t dirty_cap = std::max<int64_t>(1 << 16, span / 64);
    if (ctx->cand.cap / 8 > (size_t) cand_cap) cand_cap = (int64_t) (ctx->cand.cap / 8);
    if (ctx->dirty.cap / 8 > (size_t) dirty_cap) dirty_cap = (int64_t) (ctx->dirty.cap / 8);
    // tensor-core prefilter: one record buffer per epilogue lane of the largest grid launched
    int64_t tc_grid = 1;
    for (auto &r : *ranges)
        tc_grid = std::max<int64_t>(tc_grid, std::min<int64_t>(ctx->sm_count, (r.second + kTcTileBases - 1) / kTcTileBases - r.first / kTcTileBases));
    const int32_t n_lanes = (int32_t) (tc_grid * kTcLanesPerCta);
    int64_t lane_cap = 0;
    int64_t n_dirty = 0, n_rec = 0;
    MSB_CUDA(cudaEventRecord(ctx->ev[0], st));
    for (int attempt = 0;; attempt++) {
        MSB_TRY(ctx->cand.ensure((size_t) cand_cap * 8));
        MSB_TRY(ctx->dirty.ensure((size_t) dirty_cap * 8));
        MSB_CUDA(cudaMemsetAsync(ctx->counters.p, 0, 4 * sizeof(unsigned long long), st));
        TcParams P;
        P.seq = sv;
        P.btab = TT->d_btab.as<uint8_t>();
        P.lmax_all = std::max(TT->lmax_fast, 1);
        P.any_zero_hit = TT->any_zero_hit;
        lane_cap = std::max<int64_t>(cand_cap / 2 / n_lanes, 1);   // 16-byte records per lane buffer
        if (attempt == 0 && ctx->opt_tc_first_lane_cap > 0) lane_cap = std::min<int64_t>(lane_cap, ctx->opt_tc_first_lane_cap);
        MSB_TRY(ctx->lane_count.ensure((size_t) n_lanes * 4));
        MSB_CUDA(cudaMemsetAsync(ctx->lane_count.p, 0, (size_t) n_lanes * 4, st));
        P.cand = ctx->cand.as<uint4>();
        P.cand_cap = lane_cap;
        P.lane_count = ctx->lane_count.as<uint32_t>();
        P.dirty = ctx->dirty.as<int64_t>();
        P.dirty_cap = dirty_cap;
        P.counters = ctx->counters.as<unsigned long long>();
        P.prof = nullptr;
        DevBuf prof;
        if (ctx->opt_tc_prof) {
            MSB_TRY(prof.ensure((size_t) (ctx->sm_count + 16) * 16 * 8));
            MSB_CUDA(cudaMemsetAsync(prof.p, 0, (size_t) (ctx->sm_count + 16) * 16 * 8, st));
            P.prof = prof.as<long long>();
        }
        const size_t smem = kTcSmemBytes;  // > half an SM's shared memory: one CTA per SM, which owns the TMEM
        unsigned grid = 1;
        for (size_t ri = 0; ri < ranges->size(); ri++) {
            const auto &r = (*ranges)[ri];
            if (before_range) MSB_TRY((*before_range)(ri));
            P.pos_lo = r.first;
            P.pos_hi = r.second;
            const int64_t n_ptiles = (r.second + kTcTileBases - 1) / kTcTileBases - r.first / kTcTileBases;
            grid = (unsigned) std::min<int64_t>(ctx->sm_count, n_ptiles);
            for (size_t b = 0; b < TT->batches.size(); b++) {
                P.batch = TT->batches[b];
                P.emit_dirty = (b == 0);
                if (ctx->opt_tc_prof) prefilter_tc_kernel<true><<<grid, kTcThreads, smem, st>>>(P);
                else prefilter_tc_kernel<false><<<grid, kTcThreads, smem, st>>>(P);
                MSB_CUDA(cudaGetLastError());
                ctx->c[MSB_C_LAUNCHES]++;
                ctx->c[MSB_C_PREFILTER_LAUNCHES]++;
            }
        }
        lane_totals_kernel<<<(unsigned) std::min<int64_t>((n_lanes + 1023) / 1024, 128), 1024, 0, st>>>(ctx->lane_count.as<uint32_t>(), n_lanes, lane_cap,
                                               ctx->counters.as<unsigned long long>());
        MSB_CUDA(cudaGetLastError());
        ctx->c[MSB_C_LAUNCHES]++;
        if (ctx->opt_tc_prof) {
            std::vector<long long> h((size_t) (ctx->sm_count + 16) * 16);
            MSB_CUDA(cudaMemcpyAsync(h.data(), prof.p, h.size() * 8, cudaMemcpyDeviceToHost, st));
            MSB_CUDA(cudaStreamSynchronize(st));
            const long long *o = h.data();   // CTA 0 of the last batch
            const double un = (double) std::max<long long>(o[4], 1);
            fprintf(stderr, "[tc_prof] cta0: %lld units, %.0f clk/unit | issuer: wait stream %.0f, wait tmem_empty %.0f, issue %.0f | "
                    "epilogue warp 4: wait stream %.0f, wait tmem_full %.0f, ld %.0f, process %.0f (clk/unit); "
                    "units with a candidate %.3f, process there %.0f clk, elsewhere %.0f clk\n",
                    o[4], o[0] / un, o[1] / un, o[2] / un, o[3] / un, o[11] / un, o[8] / un, o[9] / un, o[10] / un,
                    o[14] / un, (double) o[13] / std::max<long long>(o[14], 1),
                    (double) (o[10] - o[13]) / std::max<long long>(o[12] - o[14], 1));
            const long long *tl = h.data() + (size_t) grid * 16;
            for (int i = 0; i < 12; i++)
                fprintf(stderr, "[tc_prof] unit %d: issuer woke %6lld issued %6lld | warp %lld wait_start %6lld woke %6lld ld_done %6lld proc_done %6lld\n",
                        2000 + i, tl[i * 8 + 0] - tl[0], tl[i * 8 + 1] - tl[0], tl[i * 8 + 6], tl[i * 8 + 2] - tl[0], tl[i * 8 + 3] - tl[0],
                        tl[i * 8 + 4] - tl[0], tl[i * 8 + 5] - tl[0]);
            prof.release();
        }
        MSB_CUDA(cudaEventRecord(ctx->ev[1], st));
        MSB_TRY(read_counters(ctx));
        n_rec = (int64_t) ctx->h_counters[0];   // records: (window, 64-column chunk) pairs with at least one flagged accumulator
        n_dirty = (int64_t) ctx->h_counters[1];
        // a lane that ran out of room only counted: grow every lane buffer to the largest count seen
        const int64_t worst = (int64_t) ctx->h_counters[3];
        const bool overflow = worst > lane_cap;
        if (!overflow && n_dirty <= dirty_cap) break;
        if (attempt >= 2) { set_error("msb_scan: candidate buffers kept overflowing"); return MSB_ENOMEM; }
        ctx->c[MSB_C_RETRIES]++;
        if (overflow) cand_cap = std::max(cand_cap, (worst + worst / 8 + 16) * 2 * n_lanes);
        dirty_cap = std::max(dirty_cap, n_dirty + n_dirty / 16 + 1024);
        MSB_CUDA(cudaEventRecord(ctx->ev[0], st));
    }
    ctx->c[MSB_C_CANDIDATES] = n_rec;
    ctx->c[MSB_C_DIRTY] = n_dirty;

    // ---- stage 2: exact fp64 re-score ----------------------------------------------------------
    int64_t hit_cap = std::max<int64_t>(n_rec + n_rec / 4 + 1024, 1 << 16);   // a record can flag several columns
    if (n_dirty) hit_cap += std::min<int64_t>(n_dirty * 2 * std::max(n_fast, 1), 1 << 24);
    if (n_slow) hit_cap += 1 << 20;
    if (ctx->hit_key.cap / 8 > (size_t) hit_cap) hit_cap = (int64_t) (ctx->hit_key.cap / 8);
    int64_t n_hits = 0;
    for (int attempt = 0;; attempt++) {
        MSB_TRY(ctx->hit_key.ensure((size_t) hit_cap * 8));
        MSB_TRY(ctx->hit_score.ensure((size_t) hit_cap * 8));
        MSB_CUDA(cudaMemsetAsync(ctx->counters.as<unsigned long long>() + 2, 0, sizeof(unsigned long long), st));
        const bool forked = ctx->aux_stream && cudaEventRecord(ctx->aux_fork, st) == cudaSuccess;
        bool join_aux = false;
        ExactParams E;
        E.seq = sv;
        E.mot = mv;
        E.strand = strand;
        E.key_shift = key_shift;
        E.hit_key = ctx->hit_key.as<uint64_t>();
        E.hit_score = ctx->hit_score.as<double>();
        E.hit_cap = hit_cap;
        E.counters = ctx->counters.as<unsigned long long>();
        if (n_dirty && n_fast) {
            // one block = 8 warps x 32 positions x one chunk of kDirtyMotifs motifs.  The dirty windows of a scan are
            // few (N-run edges) and this kernel is latency-bound at low occupancy: it runs beside exact_records on a
            // second stream (both only append to the hit buffers), forked behind the counter reset and joined below.
            // It is launched FIRST so that its ~100 blocks hold their slots before exact_records' thousands arrive.
            const int64_t blocks = ((n_dirty + 255) / 256) * ((n_fast + kDirtyMotifs - 1) / kDirtyMotifs);
            if (blocks > 0x7fffffffll) { set_error("msb_scan: too many dirty windows for one launch"); return MSB_EINVAL; }
            cudaStream_t ds = st;
            if (ctx->aux_stream && forked) {
                MSB_CUDA(cudaStreamWaitEvent(ctx->aux_stream, ctx->aux_fork, 0));
                ds = ctx->aux_stream;
            }
            exact_dirty_kernel<<<(unsigned) blocks, 256, 0, ds>>>(E, ctx->dirty.as<int64_t>(), n_dirty, d_order, n_fast);
            MSB_CUDA(cudaGetLastError());
            if (ds != st) {
                MSB_CUDA(cudaEventRecord(ctx->aux_join, ds));
                join_aux = true;
            }
            ctx->c[MSB_C_LAUNCHES]++;
        }
        if (n_rec) {
            exact_records_kernel<<<(unsigned) (((int64_t) n_lanes * 32 + 255) / 256), 256, 0, st>>>(
                E, ctx->cand.as<uint4>(), lane_cap, ctx->lane_count.as<uint32_t>(), n_lanes, d_order,
                TT->d_col_info.as<uint32_t>());
            MSB_CUDA(cudaGetLastError());
            ctx->c[MSB_C_LAUNCHES]++;
        }
        if (join_aux) MSB_CUDA(cudaStreamWaitEvent(st, ctx->aux_join, 0));   // behind exact_records' launch: the two overlap
        if (n_slow)
            for (auto &r : *ranges)
                MSB_TRY(launch_positions(ctx, E, nullptr, r.second - r.first, r.first, d_slow, n_slow));
        MSB_CUDA(cudaEventRecord(ctx->ev[2], st));
        MSB_TRY(read_counters(ctx));
        n_hits = (int64_t) ctx->h_counters[2];
        if (n_hits <= hit_cap) break;
        if (attempt >= 2) { set_error("msb_scan: hit buffers kept overflowing"); return MSB_ENOMEM; }
        ctx->c[MSB_C_RETRIES]++;
        hit_cap = n_hits + 1024;
    }
    ctx->c[MSB_C_HITS] = n_hits;

    // ---- stage 3: order (motif, sequence, start, fwd < rev), decode, optional de-duplication ----
    int64_t n_final = n_hits;
    if (counts_only) {
        // MSB_SCAN_COUNTS: nobody will look at the sites -- a histogram of the keys' motif field replaces
        // the sort, the decode and the site arrays
        MSB_TRY(ctx->motif_counts.ensure((size_t) (M->n + 1) * 8));
        MSB_CUDA(cudaMemsetAsync(ctx->motif_counts.p, 0, (size_t) (M->n + 1) * 8, st));
        if (n_hits) {
            const bool in_smem = (size_t) M->n * 4 <= 40 * 1024;
            const unsigned grid = (unsigned) std::min<int64_t>((n_hits + 2047) / 2048, (int64_t) ctx->sm_count * 8);
            count_hits_kernel<<<grid, 256, in_smem ? (size_t) M->n * 4 : 0, st>>>(
                ctx->hit_key.as<uint64_t>(), n_hits, key_shift, M->n, in_smem ? 1 : 0, ctx->motif_counts.as<unsigned long long>());
            MSB_CUDA(cudaGetLastError());
            ctx->c[MSB_C_LAUNCHES]++;
        }
        size_t scan_bytes = 0;
        MSB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, ctx->motif_counts.as<int64_t>(), F.offsets.as<int64_t>(), M->n + 1, st));
        MSB_TRY(ctx->sort_tmp.ensure(std::max<size_t>(scan_bytes, 16)));
        MSB_CUDA(cub::DeviceScan::ExclusiveSum(ctx->sort_tmp.p, scan_bytes, ctx->motif_counts.as<int64_t>(), F.offsets.as<int64_t>(), M->n + 1, st));
    } else if (n_hits) {
        const bool dedup = (flags & MSB_SCAN_DEDUP) != 0;
        if ((size_t) n_hits * 25 > ((size_t) 4 << 30) && !ctx->fin_hold) {
            // a very large result (billions of sites): the other set of final arrays, which only exists so that a
            // copy can overlap the next scan, gives its memory back first
            msb_ctx::FinSet &O = ctx->fin[fin_set ^ 1];
            if (O.pending) { MSB_CUDA(cudaEventSynchronize(O.read_done)); O.pending = false; }
            for (DevBuf *b : {&O.key, &O.score, &O.seq, &O.start, &O.strand}) b->release();
        }
        // without de-duplication the sorted arrays ARE the final ones; with it they are scratch and the
        // survivors are scattered into the final set
        DevBuf &s_key = dedup ? ctx->key_alt : F.key, &s_score = dedup ? ctx->score_alt : F.score;
        DevBuf &s_seq = dedup ? ctx->out_seq : F.seq, &s_start = dedup ? ctx->out_start : F.start;
        DevBuf &s_strand = dedup ? ctx->out_strand : F.strand;
        MSB_TRY(s_key.ensure((size_t) n_hits * 8));
        MSB_TRY(s_score.ensure((size_t) n_hits * 8));
        MSB_TRY(s_seq.ensure((size_t) n_hits * 4));
        MSB_TRY(s_start.ensure((size_t) n_hits * 4));
        MSB_TRY(s_strand.ensure((size_t) n_hits));
        const int end_bit = key_shift + motif_bits;
        size_t tmp_bytes = 0;
        MSB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, ctx->hit_key.as<uint64_t>(), s_key.as<uint64_t>(),
                                                 ctx->hit_score.as<double>(), s_score.as<double>(), n_hits, 0, end_bit, st));
        MSB_TRY(ctx->sort_tmp.ensure(std::max<size_t>(tmp_bytes, 16)));
        MSB_CUDA(cub::DeviceRadixSort::SortPairs(ctx->sort_tmp.p, tmp_bytes, ctx->hit_key.as<uint64_t>(), s_key.as<uint64_t>(),
                                                 ctx->hit_score.as<double>(), s_score.as<double>(), n_hits, 0, end_bit, st));
        const unsigned grid = (unsigned) ((n_hits + 255) / 256);
        const bool compact = (flags & MSB_SCAN_COMPACT) && !dedup && key_shift <= 32;
        if (compact) {
            compact_sites_kernel<<<grid, 256, 0, st>>>(s_key.as<uint64_t>(), n_hits, key_shift, s_start.as<uint32_t>());
            ctx->last_compact = true;
        } else {
            decode_sites_kernel<<<grid, 256, 0, st>>>(sv, s_key.as<uint64_t>(), n_hits, key_shift, s_seq.as<int32_t>(),
                                                      s_start.as<int32_t>(), s_strand.as<int8_t>());
        }
        MSB_CUDA(cudaGetLastError());
        ctx->c[MSB_C_LAUNCHES] += 2;  // sort (several CUB kernels, counted once) + decode
        if (dedup) {
            // scanner.py:171-193 on the device: keep flags, exclusive scan, scatter.
            MSB_TRY(ctx->keep.ensure((size_t) n_hits * 4));
            MSB_TRY(ctx->keep_pos.ensure((size_t) n_hits * 8));
            MSB_TRY(F.key.ensure((size_t) n_hits * 8));
            MSB_TRY(F.score.ensure((size_t) n_hits * 8));
            MSB_TRY(F.seq.ensure((size_t) n_hits * 4));
            MSB_TRY(F.start.ensure((size_t) n_hits * 4));
            MSB_TRY(F.strand.ensure((size_t) n_hits));
            dedup_flags_kernel<<<grid, 256, 0, st>>>(s_key.as<uint64_t>(), s_seq.as<int32_t>(), s_start.as<int32_t>(),
                                                     s_strand.as<int8_t>(), s_score.as<double>(),
                                                     n_hits, mv.len, key_shift, ctx->keep.as<int32_t>());
            MSB_CUDA(cudaGetLastError());
            size_t scan_bytes = 0;
            MSB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, ctx->keep.as<int32_t>(), ctx->keep_pos.as<int64_t>(), n_hits, st));
            MSB_TRY(ctx->sort_tmp.ensure(std::max<size_t>(scan_bytes, 16)));
            MSB_CUDA(cub::DeviceScan::ExclusiveSum(ctx->sort_tmp.p, scan_bytes, ctx->keep.as<int32_t>(), ctx->keep_pos.as<int64_t>(), n_hits, st));
            scatter_kept_kernel<<<grid, 256, 0, st>>>(ctx->keep.as<int32_t>(), ctx->keep_pos.as<int64_t>(), n_hits, s_key.as<uint64_t>(),
                                                      s_score.as<double>(), s_seq.as<int32_t>(), s_start.as<int32_t>(),
                                                      s_strand.as<int8_t>(), F.key.as<uint64_t>(), F.score.as<double>(),
                                                      F.seq.as<int32_t>(), F.start.as<int32_t>(), F.strand.as<int8_t>());
            MSB_CUDA(cudaGetLastError());
            ctx->c[MSB_C_LAUNCHES] += 3;
            // boundary chains, read from the raw sorted sites and their keep flags before anything reuses them
            const int64_t n_ranges = (int64_t) ranges->size(), cells = (int64_t) M->n * n_ranges;
            std::vector<int64_t> rr;
            if (boundary && cells) {
                rr.resize((size_t) 2 * n_ranges);
                for (int64_t k = 0; k < n_ranges; k++) { rr[k] = (*ranges)[k].first; rr[n_ranges + k] = (*ranges)[k].second; }
                MSB_TRY(ctx->bnd_range.ensure(rr.size() * 8));
                MSB_TRY(ctx->bnd_cnt.ensure((size_t) (cells + 1) * 8));
                MSB_TRY(ctx->bnd_dst.ensure((size_t) (cells + 1) * 8));
                MSB_CUDA(cudaMemcpyAsync(ctx->bnd_range.p, rr.data(), rr.size() * 8, cudaMemcpyHostToDevice, st));
                MSB_CUDA(cudaMemsetAsync(ctx->bnd_cnt.p, 0, (size_t) (cells + 1) * 8, st));
            }
            auto chains = [&](int mode) {
                boundary_chains_kernel<<<(unsigned) ((cells + 255) / 256), 256, 0, st>>>(
                    s_key.as<uint64_t>(), s_seq.as<int32_t>(), s_start.as<int32_t>(), s_strand.as<int8_t>(), s_score.as<double>(),
                    ctx->keep.as<int32_t>(), n_hits, ctx->bnd_range.as<int64_t>(), ctx->bnd_range.as<int64_t>() + n_ranges, n_ranges,
                    M->n, mv.len, key_shift, mode, ctx->bnd_cnt.as<int64_t>(), ctx->bnd_dst.as<int64_t>(), ctx->bnd_motif.as<int32_t>(),
                    ctx->bnd_seq.as<int32_t>(), ctx->bnd_start.as<int32_t>(), ctx->bnd_score.as<double>(), ctx->bnd_strand.as<int8_t>(),
                    ctx->bnd_flags.as<int8_t>());
                ctx->c[MSB_C_LAUNCHES]++;
                return cudaGetLastError();
            };
            int64_t n_boundary = 0;
            if (boundary && cells) {
                MSB_CUDA(chains(0));
                size_t bs = 0;
                MSB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bs, ctx->bnd_cnt.as<int64_t>(), ctx->bnd_dst.as<int64_t>(), cells + 1, st));
                MSB_TRY(ctx->sort_tmp.ensure(std::max<size_t>(bs, 16)));
                MSB_CUDA(cub::DeviceScan::ExclusiveSum(ctx->sort_tmp.p, bs, ctx->bnd_cnt.as<int64_t>(), ctx->bnd_dst.as<int64_t>(), cells + 1, st));
                MSB_CUDA(cudaMemcpyAsync(&n_boundary, ctx->bnd_dst.as<int64_t>() + cells, 8, cudaMemcpyDeviceToHost, st));
            }
            int32_t last_keep = 0;
            int64_t last_pos = 0;
            MSB_CUDA(cudaMemcpyAsync(&last_keep, ctx->keep.as<int32_t>() + (n_hits - 1), 4, cudaMemcpyDeviceToHost, st));
            MSB_CUDA(cudaMemcpyAsync(&last_pos, ctx->keep_pos.as<int64_t>() + (n_hits - 1), 8, cudaMemcpyDeviceToHost, st));
            MSB_CUDA(cudaStreamSynchronize(st));
            n_final = last_pos + last_keep;
            if (n_boundary) {
                MSB_TRY(ctx->bnd_motif.ensure((size_t) n_boundary * 4));
                MSB_TRY(ctx->bnd_seq.ensure((size_t) n_boundary * 4));
                MSB_TRY(ctx->bnd_start.ensure((size_t) n_boundary * 4));
                MSB_TRY(ctx->bnd_score.ensure((size_t) n_boundary * 8));
                MSB_TRY(ctx->bnd_strand.ensure((size_t) n_boundary));
                MSB_TRY(ctx->bnd_flags.ensure((size_t) n_boundary));
                MSB_CUDA(chains(1));
                ctx->last_boundary = n_boundary;
            }
        }
        ctx->fin_key = F.key.as<uint64_t>();
        ctx->fin_score = F.score.as<double>();
        ctx->fin_seq = F.seq.as<int32_t>();
        ctx->fin_start = F.start.as<int32_t>();
        ctx->fin_strand = F.strand.as<int8_t>();
        motif_offsets_kernel<<<(unsigned) ((M->n + 1 + 255) / 256), 256, 0, st>>>(ctx->fin_key, n_final, M->n, key_shift,
                                                                                  F.offsets.as<int64_t>());
        MSB_CUDA(cudaGetLastError());
        ctx->c[MSB_C_LAUNCHES] += 1;
    }
    MSB_CUDA(cudaEventRecord(ctx->ev[3], st));
    MSB_CUDA(cudaStreamSynchronize(st));
    ctx->t[MSB_T_PREFILTER] = ev_ms(ctx->ev[0], ctx->ev[1]);
    ctx->t[MSB_T_EXACT] = ev_ms(ctx->ev[1], ctx->ev[2]);
    ctx->t[MSB_T_ORDER] = ev_ms(ctx->ev[2], ctx->ev[3]);
    ctx->t[MSB_T_D2H] = 0;
    ctx->last_sites = n_final;
    ctx->fin_cur = fin_set;
    ctx->last_counts_only = counts_only;
    return MSB_OK;
}

}  // namespace msb

extern "C" {

int msb_ctx_set_option(msb_ctx *ctx, const char *name, int value) {
    if (!ctx) { set_error("msb_ctx_set_option: null ctx"); return MSB_EINVAL; }
    if (name && !std::strcmp(name, "tc_prof") && (value == 0 || value == 1)) { ctx->opt_tc_prof = value; return MSB_OK; }
    if (name && !std::strcmp(name, "tc_first_lane_cap") && value >= 0) { ctx->opt_tc_first_lane_cap = value; return MSB_OK; }
    if (name && !std::strcmp(name, "ascii_slices") && value >= 1 && value <= 7) { ctx->opt_ascii_slices = value; return MSB_OK; }
    if (name && !std::strcmp(name, "poison_pool") && (value == 0 || value == 1)) { ctx->opt_poison_pool = value; return MSB_OK; }
    if (name && !std::strcmp(name, "tc_interleave") && (value == 0 || value == 1)) { ctx->opt_tc_interleave = value; return MSB_OK; }
    if (name && !std::strcmp(name, "select_pilot") && (value == 0 || value == 1)) { ctx->opt_select_pilot = value; return MSB_OK; }
    set_error("msb_ctx_set_option: unknown option or value");
    return MSB_EINVAL;
}

int msb_scan_device(msb_ctx *ctx, const msb_motifs *M, const msb_seqs *S, int strand, int flags, int64_t *n_sites) {
    MSB_TRY(scan_device(ctx, const_cast<msb_motifs *>(M), S, strand, flags));
    if (n_sites) *n_sites = ctx->last_sites;
    return MSB_OK;
}

int msb_scan_device_counts(msb_ctx *ctx, int64_t *counts, int32_t n_motifs) {
    if (!ctx || (!counts && n_motifs)) { set_error("msb_scan_device_counts: null"); return MSB_EINVAL; }
    if (n_motifs != ctx->last_n_motifs) { set_error("msb_scan_device_counts: no scan with that many motifs"); return MSB_EINVAL; }
    if (n_motifs == 0) return MSB_OK;
    MSB_CUDA(cudaSetDevice(ctx->device));
    std::vector<int64_t> offsets((size_t) n_motifs + 1, 0);
    if (ctx->last_sites)
        MSB_CUDA(cudaMemcpyAsync(offsets.data(), ctx->fin[ctx->fin_cur].offsets.p, offsets.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    MSB_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int32_t m = 0; m < n_motifs; m++) counts[m] = offsets[m + 1] - offsets[m];
    return MSB_OK;
}

int msb_scan_device_region_counts(msb_ctx *ctx, int64_t *counts, int32_t n_motifs) {
    if (!ctx || (!counts && n_motifs)) { set_error("msb_scan_device_region_counts: null"); return MSB_EINVAL; }
    if (n_motifs != ctx->last_n_motifs) { set_error("msb_scan_device_region_counts: no scan with that many motifs"); return MSB_EINVAL; }
    if (n_motifs == 0) return MSB_OK;
    MSB_CUDA(cudaSetDevice(ctx->device));
    std::fill(counts, counts + n_motifs, (int64_t) 0);
    if (ctx->last_counts_only) { set_error("msb_scan_device_region_counts: the last scan kept per-motif counts only (MSB_SCAN_COUNTS)"); return MSB_EINVAL; }
    if (ctx->last_compact) { set_error("msb_scan_device_region_counts: the last scan kept compact sites (MSB_SCAN_COMPACT)"); return MSB_EINVAL; }
    if (ctx->last_sites == 0) return MSB_OK;
    cudaStream_t st = ctx->stream;
    MSB_TRY(ctx->sel.ensure((size_t) n_motifs * 8));
    MSB_CUDA(cudaMemsetAsync(ctx->sel.p, 0, (size_t) n_motifs * 8, st));
    region_counts_kernel<<<(unsigned) ((ctx->last_sites + 255) / 256), 256, 0, st>>>(
        ctx->fin_key, ctx->fin_seq, ctx->last_sites, ctx->last_key_shift, ctx->sel.as<unsigned long long>());
    MSB_CUDA(cudaGetLastError());
    MSB_CUDA(cudaMemcpyAsync(counts, ctx->sel.p, (size_t) n_motifs * 8, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaStreamSynchronize(st));
    return MSB_OK;
}

int msb_scan_device_boundary_sites(msb_ctx *ctx, int64_t cap, int64_t *n, int32_t *motif, int32_t *seq_idx, int32_t *start,
                                   double *score, int8_t *strand, int8_t *flags) {
    if (!ctx || !n) { set_error("msb_scan_device_boundary_sites: null"); return MSB_EINVAL; }
    if (ctx->last_boundary < 0) {
        set_error("msb_scan_device_boundary_sites: the last scan was not a de-duplicated range scan (MSB_SCAN_DEDUP)");
        return MSB_EINVAL;
    }
    const int64_t nb = ctx->last_boundary;
    *n = nb;
    if (nb == 0 || cap < nb) return MSB_OK;
    if (!motif || !seq_idx || !start || !score || !strand || !flags) { set_error("msb_scan_device_boundary_sites: null array"); return MSB_EINVAL; }
    MSB_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    MSB_CUDA(cudaMemcpyAsync(motif, ctx->bnd_motif.p, (size_t) nb * 4, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaMemcpyAsync(seq_idx, ctx->bnd_seq.p, (size_t) nb * 4, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaMemcpyAsync(start, ctx->bnd_start.p, (size_t) nb * 4, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaMemcpyAsync(score, ctx->bnd_score.p, (size_t) nb * 8, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaMemcpyAsync(strand, ctx->bnd_strand.p, (size_t) nb, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaMemcpyAsync(flags, ctx->bnd_flags.p, (size_t) nb, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaStreamSynchronize(st));
    return MSB_OK;
}

int msb_scan_device_cell_stats(msb_ctx *ctx, int32_t n_motifs, int64_t n_seqs, int64_t *counts, double *best) {
    if (!ctx || n_seqs < 0 || ((!counts || !best) && n_motifs && n_seqs)) { set_error("msb_scan_device_cell_stats: null"); return MSB_EINVAL; }
    if (n_motifs != ctx->last_n_motifs) { set_error("msb_scan_device_cell_stats: no scan with that many motifs"); return MSB_EINVAL; }
    if (n_seqs != ctx->last_n_seqs) { set_error("msb_scan_device_cell_stats: n_seqs differs from the scanned set"); return MSB_EINVAL; }
    const size_t cells = (size_t) n_motifs * (size_t) n_seqs;
    if (cells == 0) return MSB_OK;
    std::fill(counts, counts + cells, (int64_t) 0);
    std::fill(best, best + cells, std::numeric_limits<double>::quiet_NaN());
    if (ctx->last_counts_only) { set_error("msb_scan_device_cell_stats: the last scan kept per-motif counts only (MSB_SCAN_COUNTS)"); return MSB_EINVAL; }
    if (ctx->last_compact) { set_error("msb_scan_device_cell_stats: the last scan kept compact sites (MSB_SCAN_COMPACT)"); return MSB_EINVAL; }
    if (ctx->last_sites == 0) return MSB_OK;
    MSB_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    MSB_TRY(ctx->sel.ensure(cells * 16));
    MSB_CUDA(cudaMemsetAsync(ctx->sel.p, 0, cells * 16, st));
    unsigned long long *d_count = ctx->sel.as<unsigned long long>(), *d_best = d_count + cells;
    cell_stats_kernel<<<(unsigned) ((ctx->last_sites + 32 * 256 - 1) / (32 * 256)), 256, 0, st>>>(
        ctx->fin_key, ctx->fin_seq, ctx->fin_score, ctx->last_sites, ctx->last_key_shift, n_seqs, d_count, d_best);
    MSB_CUDA(cudaGetLastError());
    std::vector<uint64_t> keys(cells);
    MSB_CUDA(cudaMemcpyAsync(counts, d_count, cells * 8, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaMemcpyAsync(keys.data(), d_best, cells * 8, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaStreamSynchronize(st));
    for (size_t c = 0; c < cells; c++) {
        if (!counts[c]) continue;
        const uint64_t k = keys[c], b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;   // order_key_inv
        std::memcpy(best + c, &b, 8);
    }
    return MSB_OK;
}

}  // extern "C"

// msb_scan_variants_ex / msb_scan_haplotypes: context i carries the edits [edit_off[i], edit_off[i + 1]), edit k
// replacing the ref bases [at[k], at[k] + ref_len[k]) by alt_len[k] bases; edit_off == nullptr: one edit per context,
// edit i (msb_scan_variants_ex: no offset table, no alt starts and no other-side starts on the device).  Checks the tables, runs the two scans and
// the row kernel, and leaves the rows in order on the device.
static int scan_edit_rows(msb_ctx *ctx, const msb_motifs *M, const msb_seqs *ref, const msb_seqs *alt, const int64_t *edit_off,
                          const int32_t *at, const int32_t *ref_len, const int32_t *alt_len, int strand, int64_t *n_rows,
                          const char *what) {
    const int64_t n = ref->n;
    auto fail = [&](const char *msg) { set_error(std::string(what) + ": " + msg); return MSB_EINVAL; };
    const bool one_each = edit_off == nullptr;
    if (!one_each && edit_off[0] != 0) return fail("edit offsets must start at 0");
    const int64_t n_edits = one_each ? n : edit_off[n];
    std::vector<int32_t> alt_at((size_t) (one_each ? 0 : std::max<int64_t>(n_edits, 1)));
    int32_t max_len = 0;
    for (int64_t i = 0; i < n; i++) {
        const int64_t e0 = one_each ? i : edit_off[i], e1 = one_each ? i + 1 : edit_off[i + 1];
        if (e1 < e0) return fail("edit offsets not ascending");
        const int64_t len_r = ref->seq_off[i + 1] - ref->seq_off[i], len_a = alt->seq_off[i + 1] - alt->seq_off[i];
        max_len = std::max<int32_t>(max_len, (int32_t) std::max(len_r, len_a));
        int64_t shift = 0, prev_end = 0;
        for (int64_t k = e0; k < e1; k++) {
            if (at[k] < 0 || ref_len[k] < 0 || alt_len[k] < 0 || std::max(ref_len[k], alt_len[k]) < 1 ||
                (int64_t) at[k] + ref_len[k] > len_r || (int64_t) at[k] + shift + alt_len[k] > len_a)
                return fail("core outside its context");
            // an insertion occupies its junction: the next edit starts behind at + max(ref_len, 1)
            if (k > e0 && at[k] < prev_end) return fail("edits out of order or overlapping");
            if (!one_each) alt_at[(size_t) k] = (int32_t) (at[k] + shift);
            shift += alt_len[k] - ref_len[k];
            prev_end = (int64_t) at[k] + std::max(ref_len[k], 1);
        }
        if (len_a - len_r != shift) return fail("a context's length change differs from its edits'");
    }
    int seq_bits = 0, motif_bits = 0, start_bits = 0;
    const int side_bits = n_edits > n ? 1 : 0;      // several edits in a context: ref and alt rows may share a start
    while ((1ll << seq_bits) < n) seq_bits++;
    while ((1ll << motif_bits) < (int64_t) M->n) motif_bits++;
    while ((1ll << start_bits) < (int64_t) max_len) start_bits++;
    if (seq_bits + motif_bits + start_bits + 1 + side_bits > 64)
        return fail("too many contexts x motifs x context bases for a 64-bit row key");
    // the two scans: the ref sites stay in their final set while the alt scan fills the other one
    double t_pre = 0, t_exact = 0, t_order = 0;
    MSB_TRY(scan_device(ctx, const_cast<msb_motifs *>(M), ref, strand, 0));
    const msb_ctx::FinSet &FR = ctx->fin[ctx->fin_cur];
    VariantSide R;
    R.seq = ref->view();
    R.key = FR.key.as<uint64_t>(); R.seq_idx = FR.seq.as<int32_t>(); R.start = FR.start.as<int32_t>();
    R.strand = FR.strand.as<int8_t>(); R.score = FR.score.as<double>();
    R.n = ctx->last_sites;
    R.key_shift = ctx->last_key_shift;
    t_pre += ctx->t[MSB_T_PREFILTER]; t_exact += ctx->t[MSB_T_EXACT]; t_order += ctx->t[MSB_T_ORDER];
    const int64_t c_retries = ctx->c[MSB_C_RETRIES];
    ctx->fin_hold = true;
    const int rc_alt = scan_device(ctx, const_cast<msb_motifs *>(M), alt, strand, 0);
    ctx->fin_hold = false;
    MSB_TRY(rc_alt);
    ctx->c[MSB_C_RETRIES] += c_retries;
    const msb_ctx::FinSet &FA = ctx->fin[ctx->fin_cur];
    VariantSide A;
    A.seq = alt->view();
    A.key = FA.key.as<uint64_t>(); A.seq_idx = FA.seq.as<int32_t>(); A.start = FA.start.as<int32_t>();
    A.strand = FA.strand.as<int8_t>(); A.score = FA.score.as<double>();
    A.n = ctx->last_sites;
    A.key_shift = ctx->last_key_shift;
    t_pre += ctx->t[MSB_T_PREFILTER]; t_exact += ctx->t[MSB_T_EXACT]; t_order += ctx->t[MSB_T_ORDER];
    if (R.n == 0) R.key = nullptr;   // empty lists: nothing is read
    if (A.n == 0) A.key = nullptr;
    // rows: at most one per site of either list
    cudaStream_t st = ctx->stream;
    const int64_t cap = std::max<int64_t>(R.n + A.n, 1);
    MSB_TRY(ctx->vr_key.ensure((size_t) cap * 8));
    MSB_TRY(ctx->vr_idx.ensure((size_t) cap * 4));
    MSB_TRY(ctx->vr_ref.ensure((size_t) cap * 8));
    MSB_TRY(ctx->vr_alt.ensure((size_t) cap * 8));
    MSB_TRY(ctx->vr_eff.ensure((size_t) cap));
    if (!one_each) MSB_TRY(ctx->vr_other.ensure((size_t) cap * 4));
    // device edit table: at | ref len | alt len [| alt at]
    MSB_TRY(ctx->vr_core.ensure((size_t) std::max<int64_t>((one_each ? 3 : 4) * n_edits, 1) * 4));
    int32_t *d_core = ctx->vr_core.as<int32_t>();
    if (!one_each) {
        MSB_TRY(ctx->vr_eoff.ensure((size_t) (n + 1) * 8));
        MSB_CUDA(cudaMemcpyAsync(ctx->vr_eoff.p, edit_off, (size_t) (n + 1) * 8, cudaMemcpyHostToDevice, st));
    }
    if (n_edits) {
        MSB_CUDA(cudaMemcpyAsync(d_core, at, (size_t) n_edits * 4, cudaMemcpyHostToDevice, st));
        MSB_CUDA(cudaMemcpyAsync(d_core + n_edits, ref_len, (size_t) n_edits * 4, cudaMemcpyHostToDevice, st));
        MSB_CUDA(cudaMemcpyAsync(d_core + 2 * n_edits, alt_len, (size_t) n_edits * 4, cudaMemcpyHostToDevice, st));
        if (!one_each)
            MSB_CUDA(cudaMemcpyAsync(d_core + 3 * n_edits, alt_at.data(), (size_t) n_edits * 4, cudaMemcpyHostToDevice, st));
    }
    R.at = d_core; R.len = d_core + n_edits; A.len = d_core + 2 * n_edits; A.at = one_each ? d_core : d_core + 3 * n_edits;
    const int64_t *d_eoff = one_each ? nullptr : ctx->vr_eoff.as<int64_t>();
    int32_t *d_other = one_each ? nullptr : ctx->vr_other.as<int32_t>();
    MSB_CUDA(cudaMemsetAsync(ctx->counters.p, 0, sizeof(unsigned long long), st));
    MSB_CUDA(cudaEventRecord(ctx->ev[4], st));
    if (R.n + A.n) {
        variant_rows_kernel<<<(unsigned) ((R.n + A.n + 255) / 256), 256, 0, st>>>(
            R, A, M->view(), d_eoff, motif_bits, start_bits, side_bits,
            ctx->counters.as<unsigned long long>(), ctx->vr_key.as<uint64_t>(), ctx->vr_idx.as<int32_t>(),
            ctx->vr_ref.as<double>(), ctx->vr_alt.as<double>(), ctx->vr_eff.as<int8_t>(), d_other);
        MSB_CUDA(cudaGetLastError());
        ctx->c[MSB_C_LAUNCHES]++;
    }
    MSB_CUDA(cudaEventRecord(ctx->ev[5], st));
    MSB_TRY(read_counters(ctx));
    const int64_t rows = (int64_t) ctx->h_counters[0];
    if (rows) {
        // (context, motif, start, strand, side) order: one radix sort of the row keys with the row index as the value
        MSB_TRY(ctx->vr_key_sorted.ensure((size_t) rows * 8));
        MSB_TRY(ctx->vr_idx_sorted.ensure((size_t) rows * 4));
        MSB_TRY(ctx->vo_allele.ensure((size_t) rows * 4));
        MSB_TRY(ctx->vo_motif.ensure((size_t) rows * 4));
        MSB_TRY(ctx->vo_start.ensure((size_t) rows * 4));
        MSB_TRY(ctx->vo_strand.ensure((size_t) rows));
        MSB_TRY(ctx->vo_ref.ensure((size_t) rows * 8));
        MSB_TRY(ctx->vo_alt.ensure((size_t) rows * 8));
        MSB_TRY(ctx->vo_eff.ensure((size_t) rows));
        if (!one_each) MSB_TRY(ctx->vo_other.ensure((size_t) rows * 4));
        const int end_bit = seq_bits + motif_bits + start_bits + 1 + side_bits;
        size_t tmp_bytes = 0;
        MSB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, ctx->vr_key.as<uint64_t>(), ctx->vr_key_sorted.as<uint64_t>(),
                                                 ctx->vr_idx.as<int32_t>(), ctx->vr_idx_sorted.as<int32_t>(), rows, 0, end_bit, st));
        MSB_TRY(ctx->sort_tmp.ensure(std::max<size_t>(tmp_bytes, 16)));
        MSB_CUDA(cub::DeviceRadixSort::SortPairs(ctx->sort_tmp.p, tmp_bytes, ctx->vr_key.as<uint64_t>(), ctx->vr_key_sorted.as<uint64_t>(),
                                                 ctx->vr_idx.as<int32_t>(), ctx->vr_idx_sorted.as<int32_t>(), rows, 0, end_bit, st));
        variant_gather_kernel<<<(unsigned) ((rows + 255) / 256), 256, 0, st>>>(
            ctx->vr_key_sorted.as<uint64_t>(), ctx->vr_idx_sorted.as<int32_t>(), rows, motif_bits, start_bits, side_bits,
            ctx->vr_ref.as<double>(), ctx->vr_alt.as<double>(), ctx->vr_eff.as<int8_t>(), d_other,
            ctx->vo_allele.as<int32_t>(), ctx->vo_motif.as<int32_t>(), ctx->vo_start.as<int32_t>(), ctx->vo_strand.as<int8_t>(),
            ctx->vo_ref.as<double>(), ctx->vo_alt.as<double>(), ctx->vo_eff.as<int8_t>(),
            one_each ? nullptr : ctx->vo_other.as<int32_t>());
        MSB_CUDA(cudaGetLastError());
        ctx->c[MSB_C_LAUNCHES] += 2;
    }
    MSB_CUDA(cudaEventRecord(ctx->ev[6], st));
    MSB_CUDA(cudaStreamSynchronize(st));
    ctx->t[MSB_T_PREFILTER] = t_pre;
    ctx->t[MSB_T_EXACT] = t_exact;
    ctx->t[MSB_T_ORDER] = t_order;
    ctx->t[MSB_T_ROWS] = ev_ms(ctx->ev[4], ctx->ev[5]);
    ctx->t[MSB_T_ROW_SORT] = ev_ms(ctx->ev[5], ctx->ev[6]);
    ctx->t[MSB_T_D2H] = 0;
    ctx->last_variant_rows = rows;
    ctx->last_rows_other = !one_each;
    if (n_rows) *n_rows = rows;
    return MSB_OK;
}

extern "C" {

int msb_scan_variants(msb_ctx *ctx, const msb_motifs *M, const msb_seqs *ref, const msb_seqs *alt, const int32_t *core_start,
                      const int32_t *core_len, int strand, int64_t *n_rows) {
    if (!ctx || !M || !ref || !alt) { set_error("msb_scan_variants: null argument"); return MSB_EINVAL; }
    if (ref->n != alt->n || ref->seq_off != alt->seq_off) {
        set_error("msb_scan_variants: the ref and alt sets must hold sequences of the same lengths");
        return MSB_EINVAL;
    }
    const int64_t n = ref->n;
    if (n > 0 && (!core_start || !core_len)) { set_error("msb_scan_variants: null core table"); return MSB_EINVAL; }
    for (int64_t i = 0; i < n; i++)
        if (core_len[i] < 1) { set_error("msb_scan_variants: core outside its context"); return MSB_EINVAL; }
    return msb_scan_variants_ex(ctx, M, ref, alt, core_start, core_len, core_len, strand, n_rows);
}

int msb_scan_variants_ex(msb_ctx *ctx, const msb_motifs *M, const msb_seqs *ref, const msb_seqs *alt, const int32_t *core_start,
                         const int32_t *ref_core_len, const int32_t *alt_core_len, int strand, int64_t *n_rows) {
    if (!ctx || !M || !ref || !alt) { set_error("msb_scan_variants: null argument"); return MSB_EINVAL; }
    if (ref->n != alt->n) { set_error("msb_scan_variants: the ref and alt sets must hold the same number of contexts"); return MSB_EINVAL; }
    const int64_t n = ref->n;
    if (n > 0 && (!core_start || !ref_core_len || !alt_core_len)) { set_error("msb_scan_variants: null core table"); return MSB_EINVAL; }
    // one edit per context (edit_off == nullptr)
    return scan_edit_rows(ctx, M, ref, alt, nullptr, core_start, ref_core_len, alt_core_len, strand, n_rows,
                          "msb_scan_variants");
}

int msb_scan_haplotypes(msb_ctx *ctx, const msb_motifs *M, const msb_seqs *ref, const msb_seqs *alt, const int64_t *edit_off,
                        const int32_t *edit_at, const int32_t *edit_ref_len, const int32_t *edit_alt_len, int strand,
                        int64_t *n_rows) {
    if (!ctx || !M || !ref || !alt || !edit_off) { set_error("msb_scan_haplotypes: null argument"); return MSB_EINVAL; }
    if (ref->n != alt->n) { set_error("msb_scan_haplotypes: the ref and alt sets must hold the same number of contexts"); return MSB_EINVAL; }
    if (edit_off[ref->n] > 0 && (!edit_at || !edit_ref_len || !edit_alt_len)) {
        set_error("msb_scan_haplotypes: null edit table");
        return MSB_EINVAL;
    }
    return scan_edit_rows(ctx, M, ref, alt, edit_off, edit_at, edit_ref_len, edit_alt_len, strand, n_rows, "msb_scan_haplotypes");
}

static int device_rows(msb_ctx *ctx, int64_t cap, int64_t *n, int32_t *context, int32_t *motif, int32_t *start,
                       int8_t *strand, double *ref_score, double *alt_score, int8_t *effect, int32_t *other_start,
                       const char *what) {
    if (!ctx || !n) { set_error(std::string(what) + ": null"); return MSB_EINVAL; }
    if (ctx->last_variant_rows < 0) { set_error(std::string(what) + ": the last scan was not a variant scan"); return MSB_EINVAL; }
    const int64_t rows = ctx->last_variant_rows;
    *n = rows;
    if (rows == 0 || cap < rows) return MSB_OK;
    if (!context || !motif || !start || !strand || !ref_score || !alt_score || !effect) {
        set_error(std::string(what) + ": null array");
        return MSB_EINVAL;
    }
    MSB_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    MSB_CUDA(cudaEventRecord(ctx->ev[0], st));
    MSB_CUDA(cudaMemcpyAsync(context, ctx->vo_allele.p, (size_t) rows * 4, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaMemcpyAsync(motif, ctx->vo_motif.p, (size_t) rows * 4, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaMemcpyAsync(start, ctx->vo_start.p, (size_t) rows * 4, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaMemcpyAsync(strand, ctx->vo_strand.p, (size_t) rows, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaMemcpyAsync(ref_score, ctx->vo_ref.p, (size_t) rows * 8, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaMemcpyAsync(alt_score, ctx->vo_alt.p, (size_t) rows * 8, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaMemcpyAsync(effect, ctx->vo_eff.p, (size_t) rows, cudaMemcpyDeviceToHost, st));
    if (other_start) MSB_CUDA(cudaMemcpyAsync(other_start, ctx->vo_other.p, (size_t) rows * 4, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaEventRecord(ctx->ev[1], st));
    MSB_CUDA(cudaStreamSynchronize(st));
    ctx->t[MSB_T_D2H] = ev_ms(ctx->ev[0], ctx->ev[1]);
    return MSB_OK;
}

int msb_scan_device_variant_rows(msb_ctx *ctx, int64_t cap, int64_t *n, int32_t *allele, int32_t *motif, int32_t *start,
                                 int8_t *strand, double *ref_score, double *alt_score, int8_t *effect) {
    return device_rows(ctx, cap, n, allele, motif, start, strand, ref_score, alt_score, effect, nullptr,
                       "msb_scan_device_variant_rows");
}

int msb_scan_device_haplotype_rows(msb_ctx *ctx, int64_t cap, int64_t *n, int32_t *context, int32_t *motif, int32_t *start,
                                   int8_t *strand, double *ref_score, double *alt_score, int8_t *effect, int32_t *other_start) {
    if (ctx && ctx->last_variant_rows >= 0 && !ctx->last_rows_other) {
        set_error("msb_scan_device_haplotype_rows: the last scan was not msb_scan_haplotypes");
        return MSB_EINVAL;
    }
    if (ctx && ctx->last_variant_rows > 0 && cap >= ctx->last_variant_rows && !other_start) {
        set_error("msb_scan_device_haplotype_rows: null array");
        return MSB_EINVAL;
    }
    return device_rows(ctx, cap, n, context, motif, start, strand, ref_score, alt_score, effect, other_start,
                       "msb_scan_device_haplotype_rows");
}

int msb_scan_ranges_device(msb_ctx *ctx, const msb_motifs *M, const msb_seqs *S, int strand, int flags,
                           int64_t n_ranges, const int64_t *seq_idx, const int64_t *start, const int64_t *end,
                           int64_t *n_sites) {
    if (!S) { set_error("msb_scan_ranges: null seqs"); return MSB_EINVAL; }
    RangeList ranges;
    MSB_TRY(make_ranges(S, n_ranges, seq_idx, start, end, &ranges));
    if (flags & MSB_SCAN_DEDUP) {
        // the reference de-duplicates over a whole region's site list (scanner.py:171-193); two ranges of one
        // sequence would cut a chain of overlapping sites in two and the halves would be resolved independently.
        // With one range per sequence the per-sequence de-duplication is per range; the chains at the range edges
        // are kept for the caller (msb_scan_device_boundary_sites), who knows what lies beyond them.
        std::vector<int64_t> seqs(seq_idx, seq_idx + n_ranges);
        std::sort(seqs.begin(), seqs.end());
        if (std::adjacent_find(seqs.begin(), seqs.end()) != seqs.end()) {
            set_error("msb_scan_ranges: MSB_SCAN_DEDUP is not defined across range boundaries; scan whole sequences");
            return MSB_EINVAL;
        }
    }
    MSB_TRY(scan_device(ctx, const_cast<msb_motifs *>(M), S, strand, flags, &ranges, nullptr, nullptr, 1, true));
    if (n_sites) *n_sites = ctx->last_sites;
    return MSB_OK;
}

static int collect_result(msb_ctx *ctx, const msb_motifs *M, int flags, msb_result **out);

int msb_scan_ranges(msb_ctx *ctx, const msb_motifs *M, const msb_seqs *S, int strand, int flags,
                    int64_t n_ranges, const int64_t *seq_idx, const int64_t *start, const int64_t *end,
                    msb_result **out) {
    if (!out) { set_error("msb_scan_ranges: null out"); return MSB_EINVAL; }
    *out = nullptr;
    MSB_TRY(msb_scan_ranges_device(ctx, M, S, strand, flags, n_ranges, seq_idx, start, end, nullptr));
    return collect_result(ctx, M, flags, out);
}

int msb_scan_ascii(msb_ctx *ctx, const msb_motifs *M, int64_t n_seqs, const char *bytes, const int64_t *seq_off,
                   int strand, int flags, msb_seqs **seqs_out, msb_result **out) {
    if (!ctx || !M || !out || n_seqs < 0 || !seq_off || (seq_off[n_seqs] > 0 && !bytes)) {
        set_error("msb_scan_ascii: bad argument");
        return MSB_EINVAL;
    }
    *out = nullptr;
    if (seqs_out) *seqs_out = nullptr;
    if (seq_off[0] != 0) { set_error("seq_off[0] must be 0"); return MSB_EINVAL; }
    for (int64_t i = 0; i < n_seqs; i++) {
        const int64_t len = seq_off[i + 1] - seq_off[i];
        if (len < 0 || len > (int64_t) 0x7fffffff - 64) {
            set_error("msb_scan_ascii: sequence offsets not ascending or sequence >= 2^31 bases");
            return MSB_EINVAL;
        }
    }
    MSB_CUDA(cudaSetDevice(ctx->device));
    const int64_t total_bp = seq_off[n_seqs];
    // Small inputs and an unusable copy stream take the plain path.
    const int kSlices = ctx->opt_ascii_slices;
    bool sliced = total_bp >= (8 << 20) && n_seqs >= kSlices;
    if (sliced && ensure_copy_stream(ctx) != MSB_OK) sliced = false;
    if (sliced && !ctx->slice_ev[0]) {
        for (auto &evt : ctx->slice_ev)
            if (sliced && cudaEventCreateWithFlags(&evt, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); sliced = false; }
    }
    msb_seqs *S = nullptr;
    int rc = MSB_OK;
    if (!sliced) {
        MSB_TRY(msb_seqs_from_ascii(ctx, n_seqs, bytes, seq_off, &S));
        rc = msb_scan_ex(ctx, M, S, strand, flags, out);
    } else {
        cudaStream_t st = ctx->stream;
        MSB_CUDA(cudaEventRecord(ctx->ev[6], st));
        std::vector<int32_t> lens;
        MSB_TRY(seqs_prepare(ctx, n_seqs, seq_off, &S, lens));
        rc = ctx->ascii.ensure((size_t) total_bp);
        // slices of whole sequences, each about twice the bytes of the one before: the first copy, which
        // nothing can hide, is short, and every later one lands while a longer scan is running
        int64_t cut[8];
        cut[0] = 0;
        for (int k = 1; k <= kSlices; k++) {
            const int64_t want = (int64_t) ((double) total_bp * (double) ((1 << k) - 1) / (double) ((1 << kSlices) - 1));
            cut[k] = k == kSlices ? n_seqs : std::lower_bound(seq_off + cut[k - 1], seq_off + n_seqs, want) - seq_off;
        }
        RangeList ranges;
        std::vector<int> slice_of;
        cudaError_t e = cudaEventRecord(ctx->slice_ev[kSlices], st);   // the tables of seqs_prepare are on their way
        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->copy_stream, ctx->slice_ev[kSlices], 0);
        for (int k = 0; k < kSlices && e == cudaSuccess && rc == MSB_OK; k++) {
            const int64_t a = seq_off[cut[k]], b = seq_off[cut[k + 1]];
            if (b > a) e = cudaMemcpyAsync((char *) ctx->ascii.p + a, bytes + a, (size_t) (b - a), cudaMemcpyHostToDevice, ctx->copy_stream);
            if (e == cudaSuccess) e = cudaEventRecord(ctx->slice_ev[k], ctx->copy_stream);
            if (S->poff[cut[k + 1]] > S->poff[cut[k]]) {
                ranges.push_back({S->poff[cut[k]], S->poff[cut[k + 1]]});
                slice_of.push_back(k);
            }
        }
        if (rc == MSB_OK && e != cudaSuccess) rc = cuda_fail(e, "msb_scan_ascii H2D", __FILE__, __LINE__);
        std::vector<char> encoded(kSlices, 0);
        RangeHook hook = [&](size_t ri) -> int {
            const int k = slice_of[ri];
            if (encoded[k]) return MSB_OK;   // a retry after a buffer overflow: the codes are already there
            MSB_CUDA(cudaStreamWaitEvent(st, ctx->slice_ev[k], 0));
            const int64_t b0 = ranges[ri].first / kPadBases, b1 = ranges[ri].second / kPadBases;
            encode_pack_kernel<<<(unsigned) ((b1 - b0 + 255) / 256), 256, 0, st>>>(
                ctx->ascii.as<uint8_t>(), S->d_seq_off.as<int64_t>(), S->d_poff.as<int64_t>(), S->d_len.as<int32_t>(),
                n_seqs, b0, b1, S->d_codes.as<uint32_t>(), S->d_nmask.as<uint32_t>(), S->d_blk_seq.as<int32_t>());
            MSB_CUDA(cudaGetLastError());
            encoded[k] = 1;
            return MSB_OK;
        };
        if (rc == MSB_OK) rc = scan_device(ctx, const_cast<msb_motifs *>(M), S, strand, flags, &ranges, &hook);
        if (rc == MSB_OK) rc = collect_result(ctx, M, flags, out);
        cudaStreamSynchronize(ctx->copy_stream);   // `bytes` may go away after return, also on failure
        cudaStreamSynchronize(st);
        ctx->t[MSB_T_H2D] = 0;                      // hidden behind the scan; not separable
        ctx->t[MSB_T_ENCODE] = 0;
    }
    if (rc != MSB_OK) {
        if (*out) { msb_result_destroy(*out); *out = nullptr; }
        msb_seqs_destroy(S);
        return rc;
    }
    if (seqs_out) *seqs_out = S; else msb_seqs_destroy(S);
    return MSB_OK;
}

int msb_scan_ex(msb_ctx *ctx, const msb_motifs *M, const msb_seqs *S, int strand, int flags, msb_result **out) {
    if (!out) { set_error("msb_scan: null out"); return MSB_EINVAL; }
    *out = nullptr;
    MSB_TRY(scan_device(ctx, const_cast<msb_motifs *>(M), S, strand, flags));
    return collect_result(ctx, M, flags, out);
}

// Sites of the last scan_device on this context -> pinned host memory.  The copies run on the context's
// d2h stream behind an event of the main stream, so with MSB_SCAN_ASYNC the caller's next scan overlaps them
// (it fills the other FinSet); without the flag the call waits for them.
static int result_finish(msb_result *R) {
    if (!R->pending) return MSB_OK;
    cudaError_t e = cudaEventSynchronize(R->done);
    if (e != cudaSuccess) return cuda_fail(e, "msb_result_wait", __FILE__, __LINE__);
    R->pending = false;
    for (int32_t m = 0; m < R->n_motifs; m++) R->counts[m] = R->offsets[m + 1] - R->offsets[m];
    float ms = 0;
    if (cudaEventElapsedTime(&ms, R->t0, R->done) == cudaSuccess && R->ctx) R->ctx->t[MSB_T_D2H] = ms; else cudaGetLastError();
    return MSB_OK;
}

static int collect_result(msb_ctx *ctx, const msb_motifs *M, int flags, msb_result **out) {
    if (ctx->last_counts_only) { set_error("msb_scan: MSB_SCAN_COUNTS keeps no sites; use msb_scan_device / msb_scan_ranges_device + msb_scan_device_counts"); return MSB_EINVAL; }
    if (!ctx->d2h_stream) MSB_CUDA(cudaStreamCreateWithFlags(&ctx->d2h_stream, cudaStreamNonBlocking));
    msb_ctx::FinSet &F = ctx->fin[ctx->fin_cur];
    if (!F.read_done) MSB_CUDA(cudaEventCreateWithFlags(&F.read_done, cudaEventDisableTiming));
    msb_result *R = new (std::nothrow) msb_result();
    if (!R) { set_error("out of host memory"); return MSB_ENOMEM; }
    R->ctx = ctx;
    R->device = ctx->device;
    R->n_sites = ctx->last_sites;
    R->n_motifs = M->n;
    R->counts.assign((size_t) M->n, 0);
    const int64_t n = R->n_sites;
    const bool compact = ctx->last_compact && n > 0;
    const size_t off_at = ((size_t) (compact ? 12 : 17) * (size_t) n + 7) & ~(size_t) 7;
    int rc = pinned_get(ctx, off_at + (size_t) (M->n + 1) * 8, &R->block);
    if (rc != MSB_OK) { delete R; return rc; }
    char *base = (char *) R->block.p;
    R->score = (double *) base;
    if (compact) {
        R->compact = (uint32_t *) (base + 8 * n);
        R->poff = ctx->last_seqs->poff;
    } else {
        R->seq_idx = (int32_t *) (base + 8 * n);
        R->start = (int32_t *) (base + 12 * n);
        R->strand = (int8_t *) (base + 16 * n);
    }
    R->offsets = (int64_t *) (base + off_at);
    cudaStream_t st = ctx->stream, cs = ctx->d2h_stream;
    cudaError_t e = cudaEventCreate(&R->t0);
    auto step = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    step(cudaEventCreate(&R->done));
    step(cudaEventRecord(ctx->ev[4], st));                 // everything the scan enqueued
    step(cudaStreamWaitEvent(cs, ctx->ev[4], 0));
    step(cudaEventRecord(R->t0, cs));
    if (n) {
        step(cudaMemcpyAsync(R->score, ctx->fin_score, (size_t) n * 8, cudaMemcpyDeviceToHost, cs));
        if (compact) {
            step(cudaMemcpyAsync(R->compact, ctx->fin_start, (size_t) n * 4, cudaMemcpyDeviceToHost, cs));
        } else {
            step(cudaMemcpyAsync(R->seq_idx, ctx->fin_seq, (size_t) n * 4, cudaMemcpyDeviceToHost, cs));
            step(cudaMemcpyAsync(R->start, ctx->fin_start, (size_t) n * 4, cudaMemcpyDeviceToHost, cs));
            step(cudaMemcpyAsync(R->strand, ctx->fin_strand, (size_t) n, cudaMemcpyDeviceToHost, cs));
        }
    }
    step(cudaMemcpyAsync(R->offsets, F.offsets.p, (size_t) (M->n + 1) * 8, cudaMemcpyDeviceToHost, cs));
    step(cudaEventRecord(R->done, cs));
    step(cudaEventRecord(F.read_done, cs));
    if (e != cudaSuccess) { msb_result_destroy(R); return cuda_fail(e, "msb_scan D2H", __FILE__, __LINE__); }
    F.pending = true;
    R->pending = true;
    if (!(flags & MSB_SCAN_ASYNC)) {
        rc = result_finish(R);
        if (rc != MSB_OK) { msb_result_destroy(R); return rc; }
    }
    *out = R;
    return MSB_OK;
}

int msb_result_wait(msb_result *R) {
    if (!R) { set_error("null result"); return MSB_EINVAL; }
    return result_finish(R);
}

int msb_scan(msb_ctx *ctx, const msb_motifs *M, const msb_seqs *S, int strand, msb_result **out) {
    return msb_scan_ex(ctx, M, S, strand, 0, out);
}

int msb_result_total(const msb_result *R, int64_t *n) {
    if (!R || !n) { set_error("null"); return MSB_EINVAL; }
    *n = R->n_sites;   // known when the scan returns, also for an asynchronous result
    return MSB_OK;
}
int msb_result_counts(const msb_result *R, int64_t *counts) {
    if (!R || (!counts && R->n_motifs)) { set_error("null"); return MSB_EINVAL; }
    MSB_TRY(result_finish(const_cast<msb_result *>(R)));
    std::copy(R->counts.begin(), R->counts.end(), counts);
    return MSB_OK;
}
int msb_result_arrays(const msb_result *R, const int32_t **seq_idx, const int32_t **start,
                      const double **score, const int8_t **strand) {
    if (!R) { set_error("null result"); return MSB_EINVAL; }
    MSB_TRY(result_finish(const_cast<msb_result *>(R)));
    if (R->compact && !R->seq_idx) {   // first look at a compact result: find every site's sequence on the host
        msb_result *W = const_cast<msb_result *>(R);
        const int64_t n = R->n_sites;
        W->decoded.resize((size_t) 9 * n + 16);
        W->seq_idx = (int32_t *) W->decoded.data();
        W->start = W->seq_idx + n;
        W->strand = (int8_t *) (W->start + n);
        const std::vector<int64_t> &poff = R->poff;
        const int nt = n < (1 << 20) ? 1 : (int) std::min<unsigned>(std::max(1u, std::thread::hardware_concurrency()), 16u);
        auto work = [&](int t) {
            int64_t s = 0;   // sites of one motif ascend in position: the previous site's sequence is a good first guess
            for (int64_t i = n * t / nt; i < n * (t + 1) / nt; i++) {
                const int64_t p = (int64_t) (R->compact[i] >> 1);
                if (!(poff[s] <= p && p < poff[s + 1]))
                    s = (int64_t) (std::upper_bound(poff.begin(), poff.end() - 1, p) - poff.begin()) - 1;
                W->seq_idx[i] = (int32_t) s;
                W->start[i] = (int32_t) (p - poff[s]);
                W->strand[i] = (int8_t) ((R->compact[i] & 1u) + 1);
            }
        };
        std::vector<std::thread> pool;
        for (int t = 1; t < nt; t++) pool.emplace_back(work, t);
        work(0);
        for (auto &th : pool) th.join();
    }
    if (seq_idx) *seq_idx = R->seq_idx;
    if (start) *start = R->start;
    if (score) *score = R->score;
    if (strand) *strand = R->strand;
    return MSB_OK;
}
int msb_result_compact(const msb_result *R, const uint32_t **pos_strand, const double **score, const int64_t **poff,
                       int64_t *n_seqs) {
    if (!R) { set_error("null result"); return MSB_EINVAL; }
    MSB_TRY(result_finish(const_cast<msb_result *>(R)));
    if (pos_strand) *pos_strand = R->compact;           // NULL: the result is not compact
    if (score) *score = R->score;
    if (poff) *poff = R->poff.empty() ? nullptr : R->poff.data();
    if (n_seqs) *n_seqs = R->poff.empty() ? 0 : (int64_t) R->poff.size() - 1;
    return MSB_OK;
}

int msb_result_destroy(msb_result *R) {
    if (!R) return MSB_OK;
    cudaSetDevice(R->device);
    if (R->pending && R->done) cudaEventSynchronize(R->done);   // the copies write into the block
    if (R->t0) cudaEventDestroy(R->t0);
    if (R->done) cudaEventDestroy(R->done);
    if (R->ctx) pinned_put(R->ctx, R->block);
    else if (R->block.p) cudaFreeHost(R->block.p);
    delete R;
    return MSB_OK;
}

// ---- host-side gather ----------------------------------------------------------------------------
// The reference's pool hands out whole motifs and its results are per-motif lists (cscore.c:323-328,
// 425-436); here several GPUs (or several batches of one) each return a motif-major array over THEIR
// sequences, in ascending sequence order across parts, so the gathered list of motif m is part 0's slice,
// then part 1's, ...: a copy, no sort, no pickling.  Host threads split the motifs by bytes.
}  // extern "C"

// Shared skeleton of the gathers: per-motif destination offsets, motifs split over host threads by output
// size, `copy(part, src entry offset, dst entry offset, count)` moves one (motif, part) slice.
template <typename Copy>
static int merge_plan_run(int32_t n_parts, int32_t n_motifs, const int64_t *counts, int32_t n_threads, int64_t bytes_per_entry,
                          Copy copy) {
    std::vector<int64_t> src_off((size_t) n_parts * n_motifs), dst_off((size_t) n_motifs + 1, 0);
    for (int32_t p = 0; p < n_parts; p++) {
        int64_t at = 0;
        for (int32_t m = 0; m < n_motifs; m++) {
            const int64_t c = counts[(size_t) p * n_motifs + m];
            if (c < 0) { set_error("msb_merge: negative count"); return MSB_EINVAL; }
            src_off[(size_t) p * n_motifs + m] = at;
            at += c;
            dst_off[m + 1] += c;
        }
    }
    for (int32_t m = 0; m < n_motifs; m++) dst_off[m + 1] += dst_off[m];
    const int64_t total = dst_off[n_motifs];
    if (total == 0) return MSB_OK;
    int nt = std::max(1, std::min<int>(n_threads, 64));
    if (total * bytes_per_entry < (4 << 20)) nt = 1;
    auto work = [&](int t) {
        // motifs [m0, m1): boundaries at equal shares of the output
        const int64_t lo = total * t / nt, hi = total * (t + 1) / nt;
        const int32_t m0 = (int32_t) (std::lower_bound(dst_off.begin(), dst_off.end() - 1, lo) - dst_off.begin());
        const int32_t m1 = t + 1 == nt ? n_motifs : (int32_t) (std::lower_bound(dst_off.begin(), dst_off.end() - 1, hi) - dst_off.begin());
        for (int32_t m = m0; m < m1; m++) {
            int64_t at = dst_off[m];
            for (int32_t p = 0; p < n_parts; p++) {
                const int64_t c = counts[(size_t) p * n_motifs + m];
                if (!c) continue;
                copy(p, src_off[(size_t) p * n_motifs + m], at, c);
                at += c;
            }
        }
    };
    if (nt == 1) { work(0); return MSB_OK; }
    std::vector<std::thread> pool;
    for (int t = 1; t < nt; t++) pool.emplace_back(work, t);
    work(0);
    for (auto &th : pool) th.join();
    return MSB_OK;
}

extern "C" {

int msb_merge_motif_major(int32_t n_parts, int32_t n_motifs, const int64_t *counts, const void *const *src,
                          void *dst, int32_t elem_size, const int64_t *add_i32, int32_t n_threads) {
    if (n_parts < 0 || n_motifs < 0 || elem_size < 1 || (n_parts > 0 && n_motifs > 0 && (!counts || !src))) {
        set_error("msb_merge_motif_major: bad argument");
        return MSB_EINVAL;
    }
    if (add_i32 && elem_size != 4) { set_error("msb_merge_motif_major: an addend needs 4-byte elements"); return MSB_EINVAL; }
    if (n_parts == 0 || n_motifs == 0) return MSB_OK;
    int64_t total = 0;
    for (size_t i = 0; i < (size_t) n_parts * n_motifs; i++) total += counts[i];
    if (total > 0 && !dst) { set_error("msb_merge_motif_major: null destination"); return MSB_EINVAL; }
    return merge_plan_run(n_parts, n_motifs, counts, n_threads, elem_size, [&](int32_t p, int64_t from_at, int64_t to_at, int64_t c) {
        const char *from = (const char *) src[p] + from_at * elem_size;
        char *to = (char *) dst + to_at * elem_size;
        if (add_i32 && add_i32[p]) {
            const int32_t add = (int32_t) add_i32[p];
            const int32_t *f = (const int32_t *) from;
            int32_t *o = (int32_t *) to;
            for (int64_t i = 0; i < c; i++) o[i] = f[i] + add;
        } else {
            std::memcpy(to, from, (size_t) c * elem_size);
        }
    });
}

int msb_merge_sites(int32_t n_parts, int32_t n_motifs, const int64_t *counts, const int32_t *const *seq_idx,
                    const int32_t *const *start, const double *const *score, const int8_t *const *strand,
                    const int32_t *const *seq_to_group, const int32_t *const *seq_offset, int32_t *out_group,
                    int32_t *out_start, double *out_score, int8_t *out_strand, int32_t n_threads) {
    if (n_parts < 0 || n_motifs < 0 || (n_parts > 0 && n_motifs > 0 && (!counts || !seq_idx || !start || !score || !strand))) {
        set_error("msb_merge_sites: bad argument");
        return MSB_EINVAL;
    }
    if (n_parts == 0 || n_motifs == 0) return MSB_OK;
    int64_t total = 0;
    for (size_t i = 0; i < (size_t) n_parts * n_motifs; i++) total += counts[i];
    if (total > 0 && (!out_group || !out_start || !out_score || !out_strand)) { set_error("msb_merge_sites: null destination"); return MSB_EINVAL; }
    return merge_plan_run(n_parts, n_motifs, counts, n_threads, 17, [&](int32_t p, int64_t from_at, int64_t to_at, int64_t c) {
        const int32_t *sq = seq_idx[p] + from_at, *st = start[p] + from_at;
        const int32_t *grp = seq_to_group ? seq_to_group[p] : nullptr, *off = seq_offset ? seq_offset[p] : nullptr;
        int32_t *og = out_group + to_at, *os = out_start + to_at;
        for (int64_t i = 0; i < c; i++) {
            const int32_t q = sq[i];
            og[i] = grp ? grp[q] : q;
            os[i] = off ? st[i] + off[q] : st[i];
        }
        std::memcpy(out_score + to_at, score[p] + from_at, (size_t) c * 8);
        std::memcpy(out_strand + to_at, strand[p] + from_at, (size_t) c);
    });
}

int msb_merge_sites_compact(int32_t n_parts, int32_t n_motifs, const int64_t *counts, const uint32_t *const *pos_strand,
                            const double *const *score, const int64_t *const *poff, const int64_t *n_seqs,
                            const int32_t *const *seq_to_group, const int32_t *const *seq_offset, int32_t *out_group,
                            int32_t *out_start, double *out_score, int8_t *out_strand, int32_t n_threads) {
    if (n_parts < 0 || n_motifs < 0 || (n_parts > 0 && n_motifs > 0 && (!counts || !pos_strand || !score || !poff || !n_seqs))) {
        set_error("msb_merge_sites_compact: bad argument");
        return MSB_EINVAL;
    }
    if (n_parts == 0 || n_motifs == 0) return MSB_OK;
    int64_t total = 0;
    for (size_t i = 0; i < (size_t) n_parts * n_motifs; i++) total += counts[i];
    if (total > 0 && (!out_group || !out_start || !out_score || !out_strand)) { set_error("msb_merge_sites_compact: null destination"); return MSB_EINVAL; }
    return merge_plan_run(n_parts, n_motifs, counts, n_threads, 17, [&](int32_t p, int64_t from_at, int64_t to_at, int64_t c) {
        const uint32_t *ps = pos_strand[p] + from_at;
        const int64_t *po = poff[p];
        const int64_t ns = n_seqs[p];
        const int32_t *grp = seq_to_group ? seq_to_group[p] : nullptr, *off = seq_offset ? seq_offset[p] : nullptr;
        int32_t *og = out_group + to_at, *os = out_start + to_at;
        int8_t *od = out_strand + to_at;
        int64_t q = 0;   // positions ascend within a (motif, part) slice: the previous site's sequence is the first guess
        for (int64_t i = 0; i < c; i++) {
            const int64_t pos = (int64_t) (ps[i] >> 1);
            if (!(po[q] <= pos && pos < po[q + 1])) q = (int64_t) (std::upper_bound(po, po + ns, pos) - po) - 1;
            og[i] = grp ? grp[q] : (int32_t) q;
            os[i] = (int32_t) (pos - po[q]) + (off ? off[q] : 0);
            od[i] = (int8_t) ((ps[i] & 1u) + 1);
        }
        std::memcpy(out_score + to_at, score[p] + from_at, (size_t) c * 8);
    });
}

}  // extern "C"

// ---- result tables ------------------------------------------------------------------------------
// `motifscan scan` writes one row per region and one column per motif twice (site counts, best scores:
// io/__init__.py:12-38).  At 200,000 regions x 1,900 motifs that is 3.8e8 cells per table: the reference
// builds them from nested Python lists.  Here a block of rows is filled straight from the scan's
// motif-major arrays and formatted to text on host threads; numbers look exactly like Python's str().
namespace msb {

// str(float) of CPython (repr, shortest digits that round-trip; float_repr_style 'short'): fixed notation
// while -4 < decimal point position <= 16, else d.ddde+XX; always a ".0" on integral values in fixed form.
static int py_float_str(double v, char *out) {
    if (std::isnan(v)) { std::memcpy(out, "nan", 3); return 3; }
    if (std::isinf(v)) { const char *t = v < 0 ? "-inf" : "inf"; const int n = (int) std::strlen(t); std::memcpy(out, t, n); return n; }
    char buf[48];
    const auto res = std::to_chars(buf, buf + sizeof(buf), v, std::chars_format::scientific);
    const char *p = buf, *end = res.ptr;
    char *o = out;
    if (*p == '-') { *o++ = '-'; p++; }
    char digits[32];
    int nd = 0;
    while (p < end && *p != 'e') { if (*p != '.') digits[nd++] = *p; p++; }
    int e10 = 0;
    if (p < end) { p++; const bool neg = *p == '-'; if (*p == '+' || *p == '-') p++; while (p < end) e10 = e10 * 10 + (*p++ - '0'); if (neg) e10 = -e10; }
    while (nd > 1 && digits[nd - 1] == '0') nd--;          // to_chars never pads, but be safe
    const int decpt = e10 + 1;                              // value = 0.d1d2... x 10^decpt
    if (v == 0) { std::memcpy(o, "0.0", 3); return (int) (o - out) + 3; }
    if (decpt <= -4 || decpt > 16) {
        *o++ = digits[0];
        if (nd > 1) { *o++ = '.'; std::memcpy(o, digits + 1, nd - 1); o += nd - 1; }
        *o++ = 'e';
        *o++ = e10 < 0 ? '-' : '+';
        const int a = e10 < 0 ? -e10 : e10;
        if (a >= 100) *o++ = (char) ('0' + a / 100);
        *o++ = (char) ('0' + (a / 10) % 10);
        *o++ = (char) ('0' + a % 10);
    } else if (decpt <= 0) {
        *o++ = '0'; *o++ = '.';
        for (int i = 0; i < -decpt; i++) *o++ = '0';
        std::memcpy(o, digits, nd); o += nd;
    } else if (decpt >= nd) {
        std::memcpy(o, digits, nd); o += nd;
        for (int i = nd; i < decpt; i++) *o++ = '0';
        *o++ = '.'; *o++ = '0';
    } else {
        std::memcpy(o, digits, decpt); o += decpt;
        *o++ = '.';
        std::memcpy(o, digits + decpt, nd - decpt); o += nd - decpt;
    }
    return (int) (o - out);
}

static inline int fmt_int(int64_t v, char *out) {
    char tmp[24];
    int n = 0;
    uint64_t a = v < 0 ? (uint64_t) (-v) : (uint64_t) v;
    do { tmp[n++] = (char) ('0' + a % 10); a /= 10; } while (a);
    int k = 0;
    if (v < 0) out[k++] = '-';
    while (n) out[k++] = tmp[--n];
    return k;
}

template <typename Fn>
static void run_threads(int nt, Fn &fn) {
    std::vector<std::thread> pool;
    for (int t = 1; t < nt; t++) pool.emplace_back(fn, t);
    fn(0);
    for (auto &th : pool) th.join();
}

// Rows of the two tables from dense [row][motif] cells (count, best score) as text, on `nt` host threads.
template <typename Count>
static int format_cell_tables(int64_t n_rows, int32_t n_motifs, const Count *counts, const double *best, const char *lead,
                              const int64_t *lead_off, char **num_text, int64_t *num_len, char **score_text, int64_t *score_len,
                              int nt) {
    // a contiguous range of rows per thread, written with a bump pointer into a buffer sized for the worst case
    // (a count has at most 11 characters as int32, 20 as int64, a double at most 24)
    struct Part { char *num = nullptr, *score = nullptr; size_t n_num = 0, n_score = 0; };
    std::vector<Part> parts((size_t) nt);
    bool oom = false;
    auto format = [&](int t) {
        const int64_t a = n_rows * t / nt, b = n_rows * (t + 1) / nt;
        if (b <= a) return;
        const size_t lead_bytes = (size_t) (lead_off[b] - lead_off[a]);
        Part &P = parts[t];
        P.num = (char *) std::malloc(lead_bytes + (size_t) (b - a) * ((size_t) n_motifs * (sizeof(Count) == 4 ? 12 : 21) + 2));
        P.score = (char *) std::malloc(lead_bytes + (size_t) (b - a) * ((size_t) n_motifs * 26 + 2));
        if (!P.num || !P.score) { oom = true; return; }
        char *pn = P.num, *ps = P.score;
        for (int64_t r = a; r < b; r++) {
            const char *l = lead + lead_off[r];
            const size_t ln = (size_t) (lead_off[r + 1] - lead_off[r]);
            std::memcpy(pn, l, ln); pn += ln;
            std::memcpy(ps, l, ln); ps += ln;
            const Count *c = counts + (size_t) r * n_motifs;
            const double *s = best + (size_t) r * n_motifs;
            for (int32_t m = 0; m < n_motifs; m++) {
                if (m) { *pn++ = '\t'; *ps++ = '\t'; }
                const int64_t cnt = (int64_t) c[m];
                if (cnt == 0) {
                    *pn++ = '0';
                    *ps++ = 'N'; *ps++ = 'A';
                } else {
                    pn += fmt_int(cnt, pn);
                    ps += py_float_str(s[m], ps);
                }
            }
            *pn++ = '\n';
            *ps++ = '\n';
        }
        P.n_num = (size_t) (pn - P.num);
        P.n_score = (size_t) (ps - P.score);
    };
    run_threads(nt, format);
    size_t total_num = 0, total_score = 0;
    for (auto &P : parts) { total_num += P.n_num; total_score += P.n_score; }
    char *out_num = oom ? nullptr : (char *) std::malloc(std::max<size_t>(total_num, 1));
    char *out_score = oom ? nullptr : (char *) std::malloc(std::max<size_t>(total_score, 1));
    if (!out_num || !out_score) {
        for (auto &P : parts) { std::free(P.num); std::free(P.score); }
        std::free(out_num); std::free(out_score);
        set_error("out of host memory");
        return MSB_ENOMEM;
    }
    std::vector<size_t> at_num((size_t) nt), at_score((size_t) nt);
    size_t an = 0, as = 0;
    for (int t = 0; t < nt; t++) { at_num[t] = an; at_score[t] = as; an += parts[t].n_num; as += parts[t].n_score; }
    auto gather = [&](int t) {
        if (parts[t].n_num) std::memcpy(out_num + at_num[t], parts[t].num, parts[t].n_num);
        if (parts[t].n_score) std::memcpy(out_score + at_score[t], parts[t].score, parts[t].n_score);
        std::free(parts[t].num);
        std::free(parts[t].score);
    };
    run_threads(nt, gather);
    *num_text = out_num;
    *num_len = (int64_t) total_num;
    *score_text = out_score;
    *score_len = (int64_t) total_score;
    return MSB_OK;
}

}  // namespace msb

extern "C" {

int msb_format_site_tables(int32_t n_motifs, const int64_t *offsets, const int32_t *seq_idx, const double *score,
                           int64_t r0, int64_t r1, const char *lead, const int64_t *lead_off, char **num_text,
                           int64_t *num_len, char **score_text, int64_t *score_len, int32_t n_threads) {
    if (n_motifs < 0 || r1 < r0 || !offsets || !lead_off || !num_text || !num_len || !score_text || !score_len ||
        (offsets[n_motifs] > 0 && (!seq_idx || !score))) {
        set_error("msb_format_site_tables: bad argument");
        return MSB_EINVAL;
    }
    *num_text = *score_text = nullptr;
    *num_len = *score_len = 0;
    const int64_t n_rows = r1 - r0;
    if (n_rows == 0) return MSB_OK;
    const size_t cells = (size_t) n_rows * (size_t) n_motifs;
    std::vector<int32_t> counts;
    std::vector<double> best;
    try { counts.assign(cells, 0); best.assign(cells, -std::numeric_limits<double>::infinity()); }
    catch (const std::bad_alloc &) { set_error("out of host memory"); return MSB_ENOMEM; }
    const int nt = std::max(1, std::min<int>(n_threads, 64));
    // 1. the block's cells: a motif's sites are sorted by region, so its part of [r0, r1) is one slice.  A thread
    //    owns a contiguous range of motifs (= a contiguous run of cells in every row: no cache line ping-pong).
    auto fill = [&](int t) {
        for (int32_t m = (int32_t) ((int64_t) n_motifs * t / nt); m < (int32_t) ((int64_t) n_motifs * (t + 1) / nt); m++) {
            const int32_t *a = seq_idx + offsets[m], *b = seq_idx + offsets[m + 1];
            const int32_t *lo = std::lower_bound(a, b, (int32_t) r0), *hi = std::lower_bound(lo, b, (int32_t) std::min<int64_t>(r1, 0x7fffffff));
            for (const int32_t *q = lo; q < hi; q++) {
                const size_t cell = (size_t) (*q - r0) * n_motifs + m;
                counts[cell]++;
                const double sc = score[q - seq_idx];
                if (counts[cell] == 1 || sc > best[cell]) best[cell] = sc;   // max() keeps the first of equal scores
            }
        }
    };
    // 2. the rows as text
    run_threads(nt, fill);
    return format_cell_tables(n_rows, n_motifs, counts.data(), best.data(), lead, lead_off, num_text, num_len, score_text,
                              score_len, nt);
}

int msb_format_cell_tables(int64_t n_rows, int32_t n_motifs, const int64_t *counts, const double *best, const char *lead,
                           const int64_t *lead_off, char **num_text, int64_t *num_len, char **score_text, int64_t *score_len,
                           int32_t n_threads) {
    if (n_rows < 0 || n_motifs < 0 || !lead_off || !num_text || !num_len || !score_text || !score_len ||
        (n_rows && n_motifs && (!counts || !best))) {
        set_error("msb_format_cell_tables: bad argument");
        return MSB_EINVAL;
    }
    *num_text = *score_text = nullptr;
    *num_len = *score_len = 0;
    if (n_rows == 0) return MSB_OK;
    return format_cell_tables(n_rows, n_motifs, counts, best, lead, lead_off, num_text, num_len, score_text, score_len,
                              std::max(1, std::min<int>(n_threads, 64)));
}

int msb_write_sites_bed(const char *path, int64_t n, const int32_t *group, const int32_t *start, const int64_t *group_base,
                        const double *score, const int8_t *strand, int32_t length, int64_t n_groups, const char *names,
                        const int64_t *name_off, int32_t n_threads) {
    if (!path || n < 0 || n_groups < 0 || !name_off || (n && (!group || !start || !score || !strand))) {
        set_error("msb_write_sites_bed: bad argument");
        return MSB_EINVAL;
    }
    size_t name_max = 0;
    for (int64_t g = 0; g < n_groups; g++) name_max = std::max<size_t>(name_max, (size_t) (name_off[g + 1] - name_off[g]));
    for (int64_t i = 0; i < n; i++)
        if (group[i] < 0 || group[i] >= n_groups) { set_error("msb_write_sites_bed: group index out of range"); return MSB_EINVAL; }
    FILE *f = std::fopen(path, "wb");
    if (!f) { set_error(std::string("msb_write_sites_bed: cannot open ") + path); return MSB_EINVAL; }
    // blocks of sites formatted on host threads, written in order: one round of `nt` blocks at a time
    const int nt = std::max(1, std::min<int>(n_threads, 64));
    const int64_t block = 1 << 18;
    const size_t line_max = name_max + 2 * 21 + 3 + 25 + 4;
    std::vector<std::vector<char>> buf((size_t) nt);
    std::vector<size_t> used((size_t) nt);
    try { for (auto &b : buf) b.resize((size_t) std::min(n, block) * line_max); }
    catch (const std::bad_alloc &) { std::fclose(f); set_error("out of host memory"); return MSB_ENOMEM; }
    bool io_ok = true;
    for (int64_t r0 = 0; r0 < n && io_ok; r0 += block * nt) {
        auto format = [&](int t) {
            const int64_t a = std::min(n, r0 + block * t), b = std::min(n, a + block);
            char *o = buf[t].data();
            for (int64_t i = a; i < b; i++) {
                const int32_t g = group[i];
                const size_t ln = (size_t) (name_off[g + 1] - name_off[g]);
                std::memcpy(o, names + name_off[g], ln); o += ln;
                const int64_t s0 = (int64_t) start[i] + (group_base ? group_base[g] : 0);
                *o++ = '\t'; o += fmt_int(s0, o);
                *o++ = '\t'; o += fmt_int(s0 + length, o);
                *o++ = '\t'; *o++ = '.'; *o++ = '\t';
                o += py_float_str(score[i], o);
                *o++ = '\t'; *o++ = strand[i] == 1 ? '+' : '-'; *o++ = '\n';
            }
            used[t] = (size_t) (o - buf[t].data());
        };
        run_threads(nt, format);
        for (int t = 0; t < nt && io_ok; t++)
            if (used[t] && std::fwrite(buf[t].data(), 1, used[t], f) != used[t]) io_ok = false;
    }
    if (std::fclose(f) != 0) io_ok = false;
    if (!io_ok) { set_error(std::string("msb_write_sites_bed: write to ") + path + " failed"); return MSB_EINVAL; }
    return MSB_OK;
}

}  // extern "C"

// The end of a variant / haplotype table row: strand, ref_score, alt_score (printed like Python's str(); effect 6 has
// no ref window and 5 no alt window, the missing score is NA) and the effect name.
static const size_t kRowTailMax = 64;            // 2 + 2 x (1 + 25) + 6 bytes at most
static char *fmt_row_tail(char *o, int8_t strand, double ref_score, double alt_score, int eff) {
    static const char *const kEffect[4] = {"", "loss", "gain", "both"};
    *o++ = '\t'; *o++ = strand == 1 ? '+' : '-';
    *o++ = '\t';
    if (eff == 6) { std::memcpy(o, "NA", 2); o += 2; } else o += py_float_str(ref_score, o);
    *o++ = '\t';
    if (eff == 5) { std::memcpy(o, "NA", 2); o += 2; } else o += py_float_str(alt_score, o);
    *o++ = '\t';
    std::memcpy(o, kEffect[eff & 3], 4); o += 4;
    *o++ = '\n';
    return o;
}

static bool row_effect_ok(int8_t eff) { return eff >= 1 && eff <= 6 && eff != 4; }

// Writes `header` then n rows, row i formatted by row(i, o) (returns the end; at most line_max bytes) in blocks on up
// to n_threads host threads, written in order (msb_write_sites_bed's scheme).
template <class Row>
static int write_table_rows(const char *path, const char *header, int64_t n, size_t line_max, int32_t n_threads, Row row,
                            const char *what) {
    FILE *f = std::fopen(path, "wb");
    if (!f) { set_error(std::string(what) + ": cannot open " + path); return MSB_EINVAL; }
    bool io_ok = true;
    if (header) {
        const size_t hn = std::strlen(header);
        io_ok = std::fwrite(header, 1, hn, f) == hn;
    }
    const int nt = std::max(1, std::min<int>(n_threads, 64));
    const int64_t block = 1 << 17;
    std::vector<std::vector<char>> buf((size_t) nt);
    std::vector<size_t> used((size_t) nt);
    try { for (auto &b : buf) b.resize((size_t) std::min(n, block) * line_max); }
    catch (const std::bad_alloc &) { std::fclose(f); set_error("out of host memory"); return MSB_ENOMEM; }
    for (int64_t r0 = 0; r0 < n && io_ok; r0 += block * nt) {
        auto format = [&](int t) {
            const int64_t a = std::min(n, r0 + block * t), b = std::min(n, a + block);
            char *o = buf[t].data();
            for (int64_t i = a; i < b; i++) o = row(i, o);
            used[t] = (size_t) (o - buf[t].data());
        };
        run_threads(nt, format);
        for (int t = 0; t < nt && io_ok; t++)
            if (used[t] && std::fwrite(buf[t].data(), 1, used[t], f) != used[t]) io_ok = false;
    }
    if (std::fclose(f) != 0) io_ok = false;
    if (!io_ok) { set_error(std::string(what) + ": write to " + path + " failed"); return MSB_EINVAL; }
    return MSB_OK;
}

extern "C" {

int msb_write_variant_table(const char *path, const char *header, int64_t n, const int32_t *allele, const int32_t *motif,
                            const int32_t *start, const int8_t *strand, const double *ref_score, const double *alt_score,
                            const int8_t *effect, int64_t n_alleles, const char *lead, const int64_t *lead_off, int32_t n_motifs,
                            const char *motif_text, const int64_t *motif_off, const int32_t *motif_len, int32_t n_threads) {
    if (!path || n < 0 || n_alleles < 0 || n_motifs < 0 || !lead_off || !motif_off || (n_motifs && !motif_len) ||
        (n && (!allele || !motif || !start || !strand || !ref_score || !alt_score || !effect))) {
        set_error("msb_write_variant_table: bad argument");
        return MSB_EINVAL;
    }
    size_t lead_max = 0, motif_max = 0;
    for (int64_t a = 0; a < n_alleles; a++) lead_max = std::max<size_t>(lead_max, (size_t) (lead_off[a + 1] - lead_off[a]));
    for (int32_t m = 0; m < n_motifs; m++) motif_max = std::max<size_t>(motif_max, (size_t) (motif_off[m + 1] - motif_off[m]));
    for (int64_t i = 0; i < n; i++)
        if (allele[i] < 0 || allele[i] >= n_alleles || motif[i] < 0 || motif[i] >= n_motifs || !row_effect_ok(effect[i])) {
            set_error("msb_write_variant_table: row refers to an unknown allele, motif or effect");
            return MSB_EINVAL;
        }
    auto row = [&](int64_t i, char *o) {
        const int32_t al = allele[i], m = motif[i];
        const size_t ln = (size_t) (lead_off[al + 1] - lead_off[al]), mn = (size_t) (motif_off[m + 1] - motif_off[m]);
        std::memcpy(o, lead + lead_off[al], ln); o += ln;
        std::memcpy(o, motif_text + motif_off[m], mn); o += mn;
        o += fmt_int(start[i], o);
        *o++ = '\t'; o += fmt_int((int64_t) start[i] + motif_len[m], o);
        return fmt_row_tail(o, strand[i], ref_score[i], alt_score[i], effect[i]);
    };
    return write_table_rows(path, header, n, lead_max + motif_max + 2 * 22 + kRowTailMax, n_threads, row,
                            "msb_write_variant_table");
}

int msb_write_haplotype_table(const char *path, const char *header, int64_t n, const int32_t *cluster, const int32_t *motif,
                              const int64_t *ref_start, const int64_t *alt_start, const int8_t *strand, const double *ref_score,
                              const double *alt_score, const int8_t *effect, int64_t n_clusters, const char *lead,
                              const int64_t *lead_off, int32_t n_motifs, const char *motif_text, const int64_t *motif_off,
                              const int32_t *motif_len, int32_t n_threads) {
    if (!path || n < 0 || n_clusters < 0 || n_motifs < 0 || !lead_off || !motif_off || (n_motifs && !motif_len) ||
        (n && (!cluster || !motif || !ref_start || !alt_start || !strand || !ref_score || !alt_score || !effect))) {
        set_error("msb_write_haplotype_table: bad argument");
        return MSB_EINVAL;
    }
    size_t lead_max = 0, motif_max = 0;
    for (int64_t c = 0; c < n_clusters; c++) lead_max = std::max<size_t>(lead_max, (size_t) (lead_off[c + 1] - lead_off[c]));
    for (int32_t m = 0; m < n_motifs; m++) motif_max = std::max<size_t>(motif_max, (size_t) (motif_off[m + 1] - motif_off[m]));
    for (int64_t i = 0; i < n; i++)
        if (cluster[i] < 0 || cluster[i] >= n_clusters || motif[i] < 0 || motif[i] >= n_motifs || !row_effect_ok(effect[i])) {
            set_error("msb_write_haplotype_table: row refers to an unknown cluster, motif or effect");
            return MSB_EINVAL;
        }
    auto window = [](int64_t s, int32_t len, char *o) {                 // [s, s + len), or NA NA when s < 0
        if (s < 0) { std::memcpy(o, "NA\tNA", 5); return o + 5; }
        o += fmt_int(s, o);
        *o++ = '\t';
        return o + fmt_int(s + len, o);
    };
    auto row = [&](int64_t i, char *o) {
        const int32_t c = cluster[i], m = motif[i];
        const size_t ln = (size_t) (lead_off[c + 1] - lead_off[c]), mn = (size_t) (motif_off[m + 1] - motif_off[m]);
        std::memcpy(o, lead + lead_off[c], ln); o += ln;
        std::memcpy(o, motif_text + motif_off[m], mn); o += mn;
        o = window(ref_start[i], motif_len[m], o);
        *o++ = '\t';
        o = window(alt_start[i], motif_len[m], o);
        return fmt_row_tail(o, strand[i], ref_score[i], alt_score[i], effect[i]);
    };
    return write_table_rows(path, header, n, lead_max + motif_max + 4 * 22 + kRowTailMax, n_threads, row,
                            "msb_write_haplotype_table");
}

int msb_text_free(char *text) {
    std::free(text);
    return MSB_OK;
}

// ---- c_score -----------------------------------------------------------------------------------
static int check_score_args(msb_ctx *ctx, const msb_motifs *M, const msb_seqs *S, int strand) {
    if (!ctx || !M || !S) { set_error("msb_score: null argument"); return MSB_EINVAL; }
    if (strand < 1 || strand > 3) { set_error("msb_score: strand must be 1, 2 or 3"); return MSB_EINVAL; }
    if (M->ctx != ctx || S->ctx != ctx) { set_error("msb_score: motifs/seqs belong to another context"); return MSB_EINVAL; }
    MSB_CUDA(cudaSetDevice(ctx->device));
    MSB_TRY(seqs_ready(S));
    if (S->n > 0 && M->n > 0 && S->min_len < M->lmax) {
        // the reference reads lens[m] bases without a length check (cscore.c:195): undefined there
        set_error("msb_score: a sequence is shorter than the longest motif");
        return MSB_ESHORT;
    }
    return MSB_OK;
}

static int launch_score0(msb_ctx *ctx, const msb_motifs *M, const msb_seqs *S, int strand, int32_t m0,
                         int32_t m1, double *d_out) {
    dim3 grid((unsigned) ((S->n + 255) / 256), (unsigned) std::min<int32_t>(m1 - m0, 1024));
    score0_kernel<<<grid, 256, 0, ctx->stream>>>(S->view(), M->view(), strand, m0, m1, S->n, d_out);
    MSB_CUDA(cudaGetLastError());
    return MSB_OK;
}

int msb_score(msb_ctx *ctx, const msb_motifs *M, const msb_seqs *S, int strand, double *out) {
    MSB_TRY(check_score_args(ctx, M, S, strand));
    if (M->n == 0 || S->n == 0) return MSB_OK;
    if (!out) { set_error("msb_score: null out"); return MSB_EINVAL; }
    MSB_CUDA(cudaSetDevice(ctx->device));
    // motif slices bound the device buffer (n_motifs x n_seqs doubles can exceed HBM)
    const int64_t max_elems = (int64_t) 1 << 29;  // 4 GiB of doubles per slice
    const int32_t per = (int32_t) std::max<int64_t>(1, std::min<int64_t>(M->n, max_elems / std::max<int64_t>(S->n, 1)));
    MSB_TRY(ctx->scores.ensure((size_t) per * (size_t) S->n * 8));
    double total_ms = 0;
    for (int32_t m0 = 0; m0 < M->n; m0 += per) {
        const int32_t m1 = std::min(M->n, m0 + per);
        MSB_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
        MSB_TRY(launch_score0(ctx, M, S, strand, m0, m1, ctx->scores.as<double>()));
        MSB_CUDA(cudaEventRecord(ctx->ev[1], ctx->stream));
        MSB_CUDA(cudaMemcpyAsync(out + (size_t) m0 * S->n, ctx->scores.p, (size_t) (m1 - m0) * S->n * 8,
                                 cudaMemcpyDeviceToHost, ctx->stream));
        MSB_CUDA(cudaStreamSynchronize(ctx->stream));
        total_ms += ev_ms(ctx->ev[0], ctx->ev[1]);
    }
    ctx->t[MSB_T_SCORE] = total_ms;
    return MSB_OK;
}

// Radix select over `n_segs` segments (kernels.cuh, select_ranks_kernel): data = doubles or ready-made keys.
static int launch_select(msb_ctx *ctx, bool from_doubles, const void *data, const int64_t *d_seg_off, int64_t stride,
                         int32_t n_segs, const int64_t *d_ranks, int32_t n_ranks, const int64_t *d_live, int64_t max_seg_len,
                         double *d_out, int32_t *d_ok) {
    if (n_segs <= 0) return MSB_OK;
    const int smem_keys = (int) std::min<int64_t>(std::max<int64_t>(max_seg_len, 1), kSelSmemKeys);
    const size_t smem = (size_t) smem_keys * 8;
    if (from_doubles)
        select_ranks_kernel<true><<<(unsigned) n_segs, kSelThreads, smem, ctx->stream>>>(data, d_seg_off, stride, d_ranks, n_ranks, smem_keys, d_live, d_out, d_ok);
    else
        select_ranks_kernel<false><<<(unsigned) n_segs, kSelThreads, smem, ctx->stream>>>(data, d_seg_off, stride, d_ranks, n_ranks, smem_keys, d_live, d_out, d_ok);
    MSB_CUDA(cudaGetLastError());
    return MSB_OK;
}

// Every sample scored for motifs [m0, m1) and the order statistics selected from the score rows: the plain
// form of the step, used for small inputs and for the motifs the pilot scheme below could not serve.
static int score_select_direct(msb_ctx *ctx, const msb_motifs *M, const msb_seqs *S, int strand, int32_t m0, int32_t m1,
                               int32_t n_ranks, double *out, double *score_ms, double *select_ms) {
    cudaStream_t st = ctx->stream;
    const int64_t max_elems = (int64_t) 1 << 28;  // 2 GiB of doubles per slice
    const int32_t per = (int32_t) std::max<int64_t>(1, std::min<int64_t>(m1 - m0, max_elems / std::max<int64_t>(S->n, 1)));
    MSB_TRY(ctx->scores.ensure((size_t) per * (size_t) S->n * 8));
    MSB_TRY(ctx->sel.ensure((size_t) per * (size_t) n_ranks * 8));
    for (int32_t a = m0; a < m1; a += per) {
        const int32_t b = std::min(m1, a + per), cnt = b - a;
        MSB_CUDA(cudaEventRecord(ctx->ev[0], st));
        MSB_TRY(launch_score0(ctx, M, S, strand, a, b, ctx->scores.as<double>()));
        MSB_CUDA(cudaEventRecord(ctx->ev[1], st));
        MSB_TRY(launch_select(ctx, true, ctx->scores.p, nullptr, S->n, cnt, ctx->ranks.as<int64_t>(), n_ranks, nullptr, S->n,
                              ctx->sel.as<double>(), nullptr));
        MSB_CUDA(cudaEventRecord(ctx->ev[2], st));
        MSB_CUDA(cudaMemcpyAsync(out + (size_t) a * n_ranks, ctx->sel.p, (size_t) cnt * n_ranks * 8, cudaMemcpyDeviceToHost, st));
        MSB_CUDA(cudaStreamSynchronize(st));
        *score_ms += ev_ms(ctx->ev[0], ctx->ev[1]);
        *select_ms += ev_ms(ctx->ev[1], ctx->ev[2]);
    }
    return MSB_OK;
}

// The cutoff step of `motif --build` (cli/motif.py:133-137 + motif/__init__.py:378-401) without the score matrix.
//
// The reference scores every background sample for every motif (750 x 1e6 doubles = 6 GB), sorts each row and
// reads five indices, all in the top 1 %.  Here:
//   1. pilot: the first 24,576 samples are scored for all motifs (score0_kernel) and a radix select reads, per
//      motif, the pilot score tau_m at 1.5 x the deepest wanted quantile;
//   2. the scan path -- tensor-core prefilter + exact fp64 re-score -- runs over ALL samples with the tau_m as
//      cutoffs and a start limit of 1 (only the offset-0 window of a sample is a window of the distribution,
//      cscore.c:195-213): it returns exactly the samples whose score reaches tau_m, with the reference's doubles,
//      i.e. the top ~1.5 % of every row (a set that is closed upwards, so ranks inside it are ranks in the row);
//   3. per (motif, sample) the better strand (cscore.c:215-221), then a radix select per motif over those ~15,000
//      keys reads the wanted order statistics.
// A motif whose candidate set turns out smaller than the deepest rank (probability ~1e-9 per motif for iid
// samples; certain for NaN scores) is redone the plain way.  What crosses HBM is the 12 B/sample of packed
// sequence and ~16 B per candidate instead of 8 B per (motif, sample) twice.
int msb_score_select(msb_ctx *ctx, const msb_motifs *M, const msb_seqs *S, int strand, int32_t n_ranks,
                     const int64_t *ranks, double *out) {
    MSB_TRY(check_score_args(ctx, M, S, strand));
    if (n_ranks < 0 || (n_ranks > 0 && (!ranks || !out))) { set_error("msb_score_select: bad ranks"); return MSB_EINVAL; }
    if (n_ranks > kSelMaxRanks) { set_error("msb_score_select: at most 8 ranks per call"); return MSB_EINVAL; }
    int64_t deepest = 0;
    for (int32_t k = 0; k < n_ranks; k++) {
        if (ranks[k] < 0 || ranks[k] >= S->n) { set_error("msb_score_select: rank out of range"); return MSB_EINVAL; }
        deepest = std::max(deepest, ranks[k]);
    }
    if (M->n == 0 || n_ranks == 0) return MSB_OK;
    MSB_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    MSB_TRY(ctx->ranks.ensure((size_t) n_ranks * 8));
    MSB_CUDA(cudaMemcpyAsync(ctx->ranks.p, ranks, (size_t) n_ranks * 8, cudaMemcpyHostToDevice, st));
    double score_ms = 0, select_ms = 0;
    const int64_t kPilot = kSelSmemKeys;   // a pilot row fits the select kernel's shared-memory staging
    const bool pilot = ctx->opt_select_pilot && S->n >= 8 * kPilot && (deepest + 1) * 32 <= S->n;
    ctx->c[MSB_C_RETRIES] = 0;
    if (!pilot) {
        MSB_TRY(score_select_direct(ctx, M, S, strand, 0, M->n, n_ranks, out, &score_ms, &select_ms));
        ctx->t[MSB_T_SCORE] = score_ms;
        ctx->t[MSB_T_SELECT] = select_ms;
        return MSB_OK;
    }
    // ---- 1. pilot thresholds -------------------------------------------------------------------------------
    const int64_t q = (int64_t) (1.5 * (double) (deepest + 1) * (double) kPilot / (double) S->n) + 32;
    MSB_TRY(ctx->scores.ensure((size_t) M->n * (size_t) kPilot * 8));
    MSB_TRY(ctx->sel.ensure((size_t) M->n * (size_t) std::max(n_ranks, 1) * 8));
    MSB_TRY(ctx->sel_aux.ensure((size_t) (M->n + 1) * 32 + 64));
    int64_t *d_q = ctx->sel_aux.as<int64_t>();                                  // [1] pilot rank
    unsigned long long *d_dead = (unsigned long long *) (d_q + 1);              // [n] second-strand sites per motif
    int64_t *d_live = (int64_t *) (d_dead + M->n);                              // [n]
    int32_t *d_ok = (int32_t *) (d_live + M->n);                                // [n]
    MSB_CUDA(cudaMemcpyAsync(d_q, &q, 8, cudaMemcpyHostToDevice, st));
    MSB_CUDA(cudaMemsetAsync(d_dead, 0, (size_t) M->n * 8, st));
    MSB_CUDA(cudaEventRecord(ctx->ev[6], st));
    {
        SeqView head = S->view();
        head.n_seqs = kPilot;
        dim3 grid((unsigned) ((kPilot + 255) / 256), (unsigned) std::min<int32_t>(M->n, 1024));
        score0_kernel<<<grid, 256, 0, st>>>(head, M->view(), strand, 0, M->n, kPilot, ctx->scores.as<double>());
        MSB_CUDA(cudaGetLastError());
    }
    MSB_CUDA(cudaEventRecord(ctx->ev[7], st));
    MSB_TRY(launch_select(ctx, true, ctx->scores.p, nullptr, kPilot, M->n, d_q, 1, nullptr, kPilot, ctx->sel.as<double>(), nullptr));
    MSB_CUDA(cudaEventRecord(ctx->ev[5], st));
    std::vector<double> tau((size_t) M->n);
    MSB_CUDA(cudaMemcpyAsync(tau.data(), ctx->sel.p, (size_t) M->n * 8, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaStreamSynchronize(st));
    score_ms += ev_ms(ctx->ev[6], ctx->ev[7]);
    select_ms += ev_ms(ctx->ev[7], ctx->ev[5]);
    // ---- 2. the scan path over all samples, offset-0 windows only ---------------------------------------------
    // the site predicate is score - cutoff >= -1e-10 (cscore.c:358): any cutoff keeps the candidate set closed
    // upwards; tau is only a way to size it
    msb_motifs *Mt = nullptr;
    MSB_TRY(msb_motifs_create(ctx, M->n, M->lens.data(), M->mats.data(), M->mat_off.data(), tau.data(), &Mt));
    int rc = ctx->limit1.ensure((size_t) std::max<int64_t>(S->n, 1) * 4);
    if (rc == MSB_OK) {
        fill_i32_kernel<<<(unsigned) ((S->n + 255) / 256), 256, 0, st>>>(ctx->limit1.as<int32_t>(), S->n, 1);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) rc = cuda_fail(e, "fill_i32_kernel", __FILE__, __LINE__);
    }
    if (rc == MSB_OK) rc = scan_device(ctx, Mt, S, strand, 0, nullptr, nullptr, ctx->limit1.as<int32_t>(), 8);
    msb_motifs_destroy(Mt);
    MSB_TRY(rc);
    score_ms += ctx->t[MSB_T_PREFILTER] + ctx->t[MSB_T_EXACT] + ctx->t[MSB_T_ORDER];
    // ---- 3. better strand per sample, select per motif ---------------------------------------------------------
    const int64_t n_sites = ctx->last_sites;
    msb_ctx::FinSet &F = ctx->fin[ctx->fin_cur];
    std::vector<int64_t> offsets((size_t) M->n + 1, 0);
    MSB_CUDA(cudaEventRecord(ctx->ev[6], st));
    if (n_sites) {
        MSB_TRY(ctx->scores_sorted.ensure((size_t) n_sites * 8));
        sample_keys_kernel<<<(unsigned) ((n_sites + 255) / 256), 256, 0, st>>>(ctx->fin_key, ctx->fin_seq, ctx->fin_score, n_sites,
                                                                                ctx->last_key_shift, ctx->scores_sorted.as<uint64_t>(), d_dead);
        MSB_CUDA(cudaGetLastError());
        MSB_CUDA(cudaMemcpyAsync(offsets.data(), F.offsets.p, offsets.size() * 8, cudaMemcpyDeviceToHost, st));
    }
    live_counts_kernel<<<(unsigned) ((M->n + 255) / 256), 256, 0, st>>>(F.offsets.as<int64_t>(), d_dead, M->n, d_live);
    MSB_CUDA(cudaGetLastError());
    MSB_CUDA(cudaStreamSynchronize(st));
    int64_t longest = 1;
    for (int32_t m = 0; m < M->n; m++) longest = std::max(longest, offsets[m + 1] - offsets[m]);
    MSB_TRY(launch_select(ctx, false, n_sites ? ctx->scores_sorted.p : ctx->sel_aux.p, F.offsets.as<int64_t>(), 0, M->n,
                          ctx->ranks.as<int64_t>(), n_ranks, d_live, longest, ctx->sel.as<double>(), d_ok));
    MSB_CUDA(cudaEventRecord(ctx->ev[7], st));
    std::vector<int32_t> ok((size_t) M->n);
    MSB_CUDA(cudaMemcpyAsync(out, ctx->sel.p, (size_t) M->n * n_ranks * 8, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaMemcpyAsync(ok.data(), d_ok, (size_t) M->n * 4, cudaMemcpyDeviceToHost, st));
    MSB_CUDA(cudaStreamSynchronize(st));
    select_ms += ev_ms(ctx->ev[6], ctx->ev[7]);
    int64_t redone = 0;
    for (int32_t m = 0; m < M->n; m++)
        if (!ok[m]) {   // too few candidates (or NaN scores): this motif the plain way
            MSB_TRY(score_select_direct(ctx, M, S, strand, m, m + 1, n_ranks, out, &score_ms, &select_ms));
            redone++;
        }
    ctx->c[MSB_C_RETRIES] = redone;
    ctx->c[MSB_C_HITS] = n_sites;
    ctx->t[MSB_T_SCORE] = score_ms;
    ctx->t[MSB_T_SELECT] = select_ms;
    return MSB_OK;
}

// ---- one-shot mirrors --------------------------------------------------------------------------
// The reference's two methods take no handle (cscore.c:399, :231), so these need a context from
// somewhere: one per (calling host thread, device), created on first use and destroyed when the
// thread ends.  No process-wide table, no lock: concurrent callers never share a context.
struct ThreadContexts {
    std::vector<msb_ctx *> by_device;
    ~ThreadContexts() { for (msb_ctx *c : by_device) if (c) msb_ctx_destroy(c); }
};

static int default_ctx(int device, msb_ctx **out) {
    static thread_local ThreadContexts tls;
    if (device < 0 || device >= 1024) { set_error("device out of range"); return MSB_EINVAL; }
    if ((size_t) device >= tls.by_device.size()) tls.by_device.resize((size_t) device + 1, nullptr);
    if (!tls.by_device[device]) MSB_TRY(msb_ctx_create(device, nullptr, &tls.by_device[device]));
    *out = tls.by_device[device];
    return MSB_OK;
}

int msb_c_scan_motif(int device, int32_t n_motifs, const int32_t *lens, const double *mats,
                     const int64_t *mat_off, const double *cutoffs, int64_t n_seqs, const char *seq_bytes,
                     const int64_t *seq_off, int strand, msb_result **out) {
    msb_ctx *ctx = nullptr;
    MSB_TRY(default_ctx(device, &ctx));
    msb_motifs *M = nullptr;
    int rc = msb_motifs_create(ctx, n_motifs, lens, mats, mat_off, cutoffs, &M);
    if (rc == MSB_OK) rc = msb_scan_ascii(ctx, M, n_seqs, seq_bytes, seq_off, strand, 0, nullptr, out);
    // the result may outlive the calling thread (and with it the thread's context): it owns its pinned
    // block outright instead of handing it back to the context's pool
    if (rc == MSB_OK && out && *out) (*out)->ctx = nullptr;
    msb_motifs_destroy(M);
    return rc;
}

int msb_c_score(int device, int32_t n_motifs, const int32_t *lens, const double *mats, const int64_t *mat_off,
                int64_t n_seqs, const char *seq_bytes, const int64_t *seq_off, int strand, double *out) {
    msb_ctx *ctx = nullptr;
    MSB_TRY(default_ctx(device, &ctx));
    msb_motifs *M = nullptr;
    msb_seqs *S = nullptr;
    int rc = msb_motifs_create(ctx, n_motifs, lens, mats, mat_off, nullptr, &M);
    if (rc == MSB_OK) rc = msb_seqs_from_ascii(ctx, n_seqs, seq_bytes, seq_off, &S);
    if (rc == MSB_OK) rc = msb_score(ctx, M, S, strand, out);
    msb_seqs_destroy(S);
    msb_motifs_destroy(M);
    return rc;
}

}  // extern "C"
