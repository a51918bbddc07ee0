// vtx_api.cu -- C ABI of the engine (include/vartrix_b200.h): context, device memory, stream
// orchestration of the kernels in vtx_pipeline.cuh / vtx_sw.cuh.  CUDA only -- there is no CPU path.
#include "../../include/vartrix_b200.h"
#include "vtx_pipeline.cuh"
#include "vtx_sw.cuh"
#include "vtx_sw_band.cuh"
#include "vtx_inflate.cuh"
#include "vtx_stage.cuh"

#include <nvtx3/nvToolsExt.h>     // header-only; ranges cost nothing unless a profiler (nsys / ncu --nvtx) is attached

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

using namespace vtx;

namespace {

thread_local std::string g_create_error;

// NVTX range around a host-side phase of the API (submit: copies / validation / kernel enqueue; finish; gather)
struct Nvtx {
    explicit Nvtx(const char* name) { nvtxRangePushA(name); }
    ~Nvtx() { nvtxRangePop(); }
};
constexpr int kBandK = 6, kBandW = 20;       // K, W of banded::Aligner::new (main.rs:33-34, 899)

struct DBuf {
    void* p = nullptr;
    size_t cap = 0;
};

enum { EV_START = 0, EV_H2D, EV_C0, EV_PREP, EV_SW, EV_POST, EV_COUNT };

constexpr size_t kMaxCum = 4096;   // submits per finish that can stream their triplets out early

struct TimeRec {   // CUDA events of one submit
    cudaEvent_t ev[EV_COUNT] = {};
    bool had_h2d = false;
    uint64_t sw_launches = 0, launches = 0;
};

// device copies of one staged shard; two slots so that the copy of shard k+1 overlaps the kernels of shard k
struct InSlot {
    DBuf locus_row, hap, ref_off, ref_len, alt_off, alt_len, cand_start, read_nib, read_off, read_len, cb_bytes,
        read_cb_off, read_cb_len, read_umi, cand_read;
    DBuf read_off4, read_len16, read_cb_key, cb_off_ex;     // slim layout (vtx_batch2)
    cudaEvent_t copy_done = nullptr, free_ev = nullptr;
    bool used = false;
};

// device buffers of one shard staged on the device (vtx_submit_bam); two slots: shard k+1 is inflated and scanned while the
// Smith-Waterman kernels of shard k still read shard k's stream
struct StageSlot {
    DBuf comp, desc, status, stream, entry, seg_count, seg_first, rec_off, rec_tid, rec_pos, rec_end, rec_fm, l_start, l_end,
        locus_row, hap, ref_off, ref_len, alt_off, alt_len, cand_count, cand_first, cand_rec, used, read_off, read_len,
        read_cb_off, read_cb_len, read_umi, cand_start, scalars;
    cudaEvent_t staged = nullptr, free_ev = nullptr;
    bool used_once = false;
};

}  // namespace

struct vtx_ctx {
    vtx_config cfg{};
    int device = 0;
    int n_sm = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;

    // barcode table
    DBuf bc_slot, bc_bytes, bc_off;
    DBuf bck_key, bck_idx;            // the barcodes that have a vtx_pack_cb code, keyed by it
    uint32_t bck_cap = 0;
    DBuf x_read_off, x_read_len, x_units, x_off4;      // slim layout expanded to the internal read arrays
    DBuf band_scratch;                                  // VTX_BAND_MODEL work buffers, one slice per resident warp
    DBuf inf_comp, inf_out, inf_desc, inf_status;       // vtx_bgzf_inflate
    bool inflate_attr_set = false;
    StageSlot sslot[2];                                 // vtx_submit_bam
    uint64_t n_bam_submits = 0;
    cudaStream_t stage_stream = nullptr;
    DBuf bam_metrics;                                   // stage::LocusMetrics, cumulative
    DBuf stage_sums;                                    // block sums of the scans on the staging stream
    uint64_t* h_stage = nullptr;                        // pinned scalars read back between the staging phases
    uint32_t bc_cap = 0, n_barcodes = 0;
    bool have_barcodes = false;

    // staged inputs (device copies for vtx_submit): double-buffered, filled on a separate copy stream
    InSlot slot[2];
    uint64_t n_submits = 0;
    cudaStream_t copy_stream = nullptr;
    // work buffers
    DBuf read_col, keep, pidx, scan_sums, pair_read, pair_col, pair_umi, pair_locus, pair_start, tcount, tstart,
        pair_first, pair_cslot, pair_uslot, cslot_col, cslot_locus, uslot_cslot, ccnt, ucnt, keep2, oidx, tile_counters,
        scratch, pair_scores, d_metrics, d_res_n, big_list, slot_scratch;
    // results (device) + host mirrors
    DBuf r_row, r_col, r_ref, r_alt, r_unk, r_val, r_val2;
    size_t res_cap = 0;        // entries
    size_t res_ub = 0;         // upper bound of entries currently held
    bool finished = true;      // true: next submit starts a fresh result set
    void* h_res[7] = { nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr };
    size_t h_res_cap = 0;
    void* h_scalars = nullptr; // pinned: res_n (u64) + 3 metrics (u64)
    uint64_t last_n = 0;
    vtx_metrics last_metrics{};

    cudaStream_t fetch_stream = nullptr;                 // device->host copies of finished triplets
    unsigned long long* h_cum = nullptr;                 // host-mapped running triplet count after each submit
    unsigned long long* d_cum = nullptr;                 // device alias of h_cum
    std::vector<TimeRec> trecs;     // one per submit since the last finish (events are reused)
    size_t trec_used = 0;
    bool timing_valid = false;
    uint32_t last_tiles_nl = 0;       // loci of the most recent run_sw (vtx_last_tile_counts)
    bool last_tiles_valid = false;
    uint64_t t_pairs = 0;

    // multi-GPU (vtx_comm.cpp)
    void* comm = nullptr;
    int rank = 0, n_ranks = 1;
    void* g_host[7] = { nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr };
    size_t g_host_cap = 0;
    DBuf g_dev[7];
    DBuf g_counts;
    cudaStream_t comm_stream = nullptr;          // the gather runs here so that later submits overlap it
    cudaEvent_t ev_counts = nullptr, ev_gather = nullptr, ev_results = nullptr;
    uint64_t* h_counts = nullptr;                // pinned: [n_ranks + 1][4]
    bool gather_pending = false;                 // started, not yet waited for
    bool gather_guard = false;                   // ev_gather must be awaited (on the device) before r_* are overwritten
    vtx_result g_out{};
};

namespace {

int set_err(vtx_ctx* c, int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof(buf), fmt, ap); va_end(ap);
    if (c) c->err = buf; else g_create_error = buf;
    return code;
}

#define CK(call)                                                                                     \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess)                                                                       \
            return set_err(ctx, VTX_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

int ensure(vtx_ctx* ctx, DBuf& b, size_t bytes)
{
    if (bytes <= b.cap) return VTX_OK;
    if (b.p) {
        CK(cudaStreamSynchronize(ctx->stream));
        if (ctx->copy_stream) CK(cudaStreamSynchronize(ctx->copy_stream));
        CK(cudaFree(b.p)); b.p = nullptr; b.cap = 0;
    }
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) { b.p = nullptr; return set_err(ctx, VTX_E_NOMEM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e)); }
    b.cap = want;
    return VTX_OK;
}

#define ENS(buf, bytes) do { int rc_ = ensure(ctx, buf, (bytes)); if (rc_) return rc_; } while (0)

template <typename T> T* P(DBuf& b) { return static_cast<T*>(b.p); }

TimeRec* new_trec(vtx_ctx* ctx)
{
    if (ctx->finished) ctx->trec_used = 0;
    if (ctx->trec_used == ctx->trecs.size()) {
        TimeRec r;
        for (auto& e : r.ev) if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
        ctx->trecs.push_back(r);
    }
    TimeRec* r = &ctx->trecs[ctx->trec_used++];
    r->had_h2d = false; r->sw_launches = 0; r->launches = 0;
    return r;
}

inline unsigned blocks_for(uint64_t n, unsigned threads) { return unsigned((n + threads - 1) / threads); }

// exclusive scan wrapper: out has n + 1 entries
int scan_u32(vtx_ctx* ctx, const uint32_t* in, uint64_t n, uint32_t* out, uint64_t* launches)
{
    const unsigned nb = std::max(1u, blocks_for(n, kScanTile));
    ENS(ctx->scan_sums, size_t(nb) * 4);
    vtx_k_scan_tiles<<<nb, kScanThreads, 0, ctx->stream>>>(in, n, out, P<uint32_t>(ctx->scan_sums));
    vtx_k_scan_sums<<<1, kScanThreads, 0, ctx->stream>>>(P<uint32_t>(ctx->scan_sums), nb, out + n);
    vtx_k_scan_add<<<nb, kScanThreads, 0, ctx->stream>>>(out, n, P<uint32_t>(ctx->scan_sums));
    if (launches) *launches += 3;
    CK(cudaGetLastError());
    return VTX_OK;
}

struct DevBatch {   // device pointers
    uint32_t n_loci = 0; uint32_t n_reads = 0; uint64_t n_cand = 0;
    const uint32_t* locus_row; const uint8_t* hap; const uint32_t *ref_off, *ref_len, *alt_off, *alt_len;
    const uint64_t* cand_start; const uint8_t* read_nib; const uint64_t* read_off; const uint32_t* read_len;
    const uint8_t* cb_bytes; const uint32_t* read_cb_off; const uint16_t* read_cb_len; const uint64_t* read_umi;
    const uint32_t* cand_read;       // nullptr: candidate c is read c
    // slim layout: cell tags as codes (then cb_bytes / cb_off_ex hold the exotic tags only)
    const uint64_t* read_cb_key = nullptr; const uint32_t* cb_off_ex = nullptr;
    uint32_t class_mask = ~0u;       // tile classes that may get tiles (host batches: from the windows; device batches: all)
    uint32_t max_read_len = 0, max_hap_len = 0;
    uint64_t max_depth = ~0ull;      // most candidates of one locus (unknown for device batches: assume deep)
};

// the allow_* switches of run_sw, shared with the host-side class mask
struct SwAllow { bool split, multi, fold; };
SwAllow sw_allow(const vtx_ctx* ctx, uint32_t max_read, uint32_t max_hap)
{
    SwAllow a;
    a.split = max_read <= uint32_t(kSplitMaxRead) && !(ctx->cfg.flags & VTX_F_NO_SPLIT);
    a.multi = max_read <= uint32_t(kMultiMaxRead) && max_hap > uint32_t(class_max_n(kNumFastClasses - 1));
    a.fold = !(ctx->cfg.flags & (VTX_F_NO_SPLIT | VTX_F_NO_FOLD));
    return a;
}
template <int CLS>
int launch_sw_class(vtx_ctx* ctx, SwArgs a, uint64_t* launches)
{
    using TC = TileClass<CLS>;
    constexpr int PPW = 32 / TC::LPP, RS = TC::LPP * TC::CS;
    const size_t codes_bytes = (size_t(PPW) * (a.mcap + 2 * TC::LPP) * 2 + 7) & ~size_t(7);
    const size_t bnd_bytes = (CLS == kMultiClass && a.multi) ? size_t(PPW) * (a.mcap + 8) * 8 : 0;
    const size_t warp_bytes = (size_t(5 * RS) * 4 + codes_bytes + bnd_bytes + 15) & ~size_t(15);
    constexpr int kSwThreads = TC::THREADS;
    const size_t smem = warp_bytes * (kSwThreads / 32);
    auto kern = vtx_k_sw_pairs<CLS>;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    int per_sm = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kSwThreads, smem));
    if (per_sm < 1) return set_err(ctx, VTX_E_CUDA, "SW kernel class %d does not fit on an SM (smem %zu)", CLS, smem);
    kern<<<ctx->n_sm * per_sm, kSwThreads, smem, ctx->stream>>>(a);
    CK(cudaGetLastError());
    ++*launches;
    return VTX_OK;
}

template <int SCLS>
int launch_sw_split(vtx_ctx* ctx, SwArgs a, uint64_t* launches)
{
    using SC = SplitClass<SCLS>;
    const size_t smem = split_warp_bytes<SCLS>(a.mcap) * (SC::THREADS / 32);
    auto kern = vtx_k_sw_split<SCLS>;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    int per_sm = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, SC::THREADS, smem));
    if (per_sm < 1) return set_err(ctx, VTX_E_CUDA, "split SW kernel %d does not fit on an SM (smem %zu)", SCLS, smem);
    kern<<<ctx->n_sm * per_sm, SC::THREADS, smem, ctx->stream>>>(a);
    CK(cudaGetLastError());
    ++*launches;
    return VTX_OK;
}

int launch_sw_fold(vtx_ctx* ctx, SwArgs a, uint64_t* launches)
{
    // The allele table holds the widest window's allele columns: max_hap_len is exact for host batches and, for device
    // batches, a promise that vtx_k_locus_prep enforces (a wider locus gets no tiles).
    a.fold_mid_cap = std::min(std::max(int(a.max_hap) - 2 * kFoldP, 1), kFoldMaxMid);
    const size_t wb = fold_warp_bytes(a.fold_mid_cap);
    auto kern = vtx_k_sw_fold;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(wb * (kFoldThreads / 32))));
    // 9 warps per CTA when two such CTAs fit an SM (SNV windows), otherwise 8 (wide indel windows)
    int threads = kFoldThreads, per_sm = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, wb * (threads / 32)));
    if (per_sm < 2) {
        threads = kFoldThreadsNarrow;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, wb * (threads / 32)));
    }
    const size_t smem = wb * (threads / 32);
    if (per_sm < 1) return set_err(ctx, VTX_E_CUDA, "folded SW kernel does not fit on an SM (smem %zu)", smem);
    kern<<<ctx->n_sm * per_sm, threads, smem, ctx->stream>>>(a);
    CK(cudaGetLastError());
    ++*launches;
    return VTX_OK;
}

// classes + tiles + SW kernels, shared by submit and score_pairs.  pair_start must be ready.
int run_sw(vtx_ctx* ctx, const DevBatch& b, uint32_t n_pairs_ub, const uint32_t* pair_slot, uint32_t* counters,
           uint32_t* pair_scores, uint64_t* launches, uint64_t* sw_launches, TimeRec* tr)
{
    const uint32_t nl = b.n_loci;
    ENS(ctx->tcount, size_t(kNumClasses) * (nl + 1) * 4);
    ENS(ctx->tstart, size_t(kNumClasses) * (nl + 1) * 4);
    ENS(ctx->tile_counters, 64);
    const int force_slow = 0;       // reads of any supported length run on the single-phase classes (row blocks)
    const SwAllow allow = sw_allow(ctx, b.max_read_len, b.max_hap_len);
    const int allow_split = allow.split, allow_multi = allow.multi, allow_fold = allow.fold;   // fold: per locus, windows and read lengths decide
    vtx_k_locus_prep<<<blocks_for(uint64_t(nl) * 32, 256), 256, 0, ctx->stream>>>(
        nl, b.hap, b.ref_off, b.ref_len, b.alt_off, b.alt_len, P<uint32_t>(ctx->pair_start), P<uint32_t>(ctx->pair_read), b.read_len,
        force_slow, allow_split, allow_multi, allow_fold, b.max_read_len, b.max_hap_len, P<unsigned long long>(ctx->d_metrics) + 4,
        P<uint32_t>(ctx->tcount));
    ++*launches;
    vtx_k_scan_rows<<<kNumClasses, kScanThreads, 0, ctx->stream>>>(P<uint32_t>(ctx->tcount), P<uint32_t>(ctx->tstart), nl, nl + 1);
    ++*launches;
    CK(cudaGetLastError());
    CK(cudaMemsetAsync(ctx->tile_counters.p, 0, 64, ctx->stream));
    ctx->last_tiles_nl = nl;
    ctx->last_tiles_valid = true;
    if (tr) CK(cudaEventRecord(tr->ev[EV_PREP], ctx->stream));

    SwArgs a{};
    a.hap_bytes = b.hap; a.ref_off = b.ref_off; a.ref_len = b.ref_len; a.alt_off = b.alt_off; a.alt_len = b.alt_len;
    a.read_nib = b.read_nib; a.read_off = b.read_off; a.read_len = b.read_len;
    a.pair_read = P<uint32_t>(ctx->pair_read); a.pair_start = P<uint32_t>(ctx->pair_start);
    a.n_loci = nl; a.pair_slot = pair_slot; a.counters = counters; a.pair_scores = pair_scores;
    a.min_score = ctx->cfg.min_score;
    int mcap = int(std::min<uint32_t>(b.max_read_len, kFastMaxRead));
    mcap = std::max(2, (mcap + 1) & ~1);
    a.mcap = mcap;
    a.k64k = 65536u;
    a.one = 1u;
    a.multi = allow_multi;
    a.max_hap = b.max_hap_len;

    uint64_t before = *launches;
    if (ctx->cfg.band_mode == VTX_BAND_MODEL) {
        // optional slow path: every pair scored inside the k-mer-chain band model, one warp per pair (vtx_sw_band.cuh)
        BandArgs ba{};
        ba.sw = a; ba.n_pairs_ub = n_pairs_ub; ba.k = ctx->cfg.band_k; ba.w = ctx->cfg.band_w;
        ba.max_read = std::max<uint32_t>(b.max_read_len, 8); ba.max_hap = std::max<uint32_t>(b.max_hap_len, 8);
        const uint64_t all_hits = uint64_t(ba.max_read) * ba.max_hap;          // every position pair can be a hit at most
        ba.hit_cap = uint32_t(std::min<uint64_t>(all_hits, uint64_t(1) << 20));
        ba.hit_cap = std::min<uint32_t>(ba.hit_cap, 65535u * 16u);
        const size_t wb = band_warp_bytes(ba.max_read, ba.max_hap, ba.hit_cap);
        size_t warps = size_t(ctx->n_sm) * 16;
        const size_t budget = size_t(4) << 30;                                  // scratch budget: 4 GiB
        if (warps * wb > budget) warps = std::max<size_t>(size_t(ctx->n_sm), budget / wb);
        warps = std::max<size_t>(warps & ~size_t(3), 4);
        ENS(ctx->band_scratch, warps * wb);
        ba.scratch = P<uint8_t>(ctx->band_scratch);
        if (ba.max_hap >= 65536u || ba.max_read >= 65536u) return set_err(ctx, VTX_E_UNSUPPORTED, "band model: reads and windows must be shorter than 65536");
        ba.overflow = P<unsigned long long>(ctx->d_metrics) + 5;
        ba.bounds_violated = P<unsigned long long>(ctx->d_metrics) + 4;
        ba.cursor = P<uint32_t>(ctx->tile_counters);
        vtx_k_sw_band<<<unsigned(warps / (kBandThreads / 32)), kBandThreads, 0, ctx->stream>>>(ba);
        CK(cudaGetLastError());
        ++*launches;
        *sw_launches += *launches - before;
        return VTX_OK;
    }
    // b.class_mask: for host batches the classes the windows of this shard can select (scan_host_batch); all for device batches
    for (int c = 0; c < kNumFastClasses; ++c) {
        // a class whose narrowest window is wider than every window of this batch has no tiles: skip the empty launch
        // (max_hap_len is exact for host batches and a promised upper bound for device batches)
        if (c > 0 && b.max_hap_len <= uint32_t(class_max_n(c - 1))) continue;
        if (!(b.class_mask >> c & 1u)) continue;
        a.tile_start = P<uint32_t>(ctx->tstart) + size_t(c) * (nl + 1);
        a.tile_counter = P<uint32_t>(ctx->tile_counters) + c;
        int rc = VTX_OK;
        switch (c) {
        case 0: rc = launch_sw_class<0>(ctx, a, launches); break;
        case 1: rc = launch_sw_class<1>(ctx, a, launches); break;
        case 2: rc = launch_sw_class<2>(ctx, a, launches); break;
        case 3: rc = launch_sw_class<3>(ctx, a, launches); break;
        }
        if (rc) return rc;
    }
    if (allow_split) {
        for (int c = 0; c < kNumSplitClasses; ++c) {
            if (c > 0 && b.max_hap_len <= uint32_t(split_max_n(c - 1))) continue;
            if (!(b.class_mask >> (kSplitClass0 + c) & 1u)) continue;
            a.tile_start = P<uint32_t>(ctx->tstart) + size_t(kSplitClass0 + c) * (nl + 1);
            a.tile_counter = P<uint32_t>(ctx->tile_counters) + kSplitClass0 + c;
            int rc = c == 0 ? launch_sw_split<0>(ctx, a, launches) : launch_sw_split<1>(ctx, a, launches);
            if (rc) return rc;
        }
    }
    if (allow_fold && (b.class_mask >> kFoldClass & 1u)) {
        a.tile_start = P<uint32_t>(ctx->tstart) + size_t(kFoldClass) * (nl + 1);
        a.tile_counter = P<uint32_t>(ctx->tile_counters) + kFoldClass;
        int rc = launch_sw_fold(ctx, a, launches);
        if (rc) return rc;
    }
    if (b.class_mask >> kSlowClass & 1u) {   // generic class (rare)
        const unsigned blocks = unsigned(ctx->n_sm) * 4, threads = 128;
        const size_t warps = size_t(blocks) * threads / 32;
        ENS(ctx->scratch, warps * (size_t(b.max_hap_len) + 1) * 32 * 4);
        a.scratch = P<uint32_t>(ctx->scratch);
        a.tile_start = P<uint32_t>(ctx->tstart) + size_t(kSlowClass) * (nl + 1);
        a.tile_counter = P<uint32_t>(ctx->tile_counters) + kSlowClass;
        vtx_k_sw_generic<<<blocks, threads, 0, ctx->stream>>>(a);
        CK(cudaGetLastError());
        ++*launches;
    }
    *sw_launches += *launches - before;
    (void)n_pairs_ub;
    return VTX_OK;
}

int grow_results(vtx_ctx* ctx, size_t need)
{
    if (need <= ctx->res_cap) return VTX_OK;
    const size_t ncap = need + need / 4 + 1024;
    DBuf* bufs[7] = { &ctx->r_row, &ctx->r_col, &ctx->r_ref, &ctx->r_alt, &ctx->r_unk, &ctx->r_val, &ctx->r_val2 };
    const size_t esz[7] = { 4, 4, 4, 4, 4, 8, 8 };
    for (int i = 0; i < 7; ++i) {
        void* np = nullptr;
        cudaError_t e = cudaMalloc(&np, ncap * esz[i]);
        if (e != cudaSuccess) return set_err(ctx, VTX_E_NOMEM, "result cudaMalloc(%zu) failed: %s", ncap * esz[i], cudaGetErrorString(e));
        if (bufs[i]->p && ctx->res_ub && !ctx->finished)
            CK(cudaMemcpyAsync(np, bufs[i]->p, ctx->res_ub * esz[i], cudaMemcpyDeviceToDevice, ctx->stream));
        if (bufs[i]->p) {
            CK(cudaStreamSynchronize(ctx->stream));
            if (ctx->fetch_stream) CK(cudaStreamSynchronize(ctx->fetch_stream));
            if (ctx->comm_stream) CK(cudaStreamSynchronize(ctx->comm_stream));
            CK(cudaFree(bufs[i]->p));
        }
        bufs[i]->p = np; bufs[i]->cap = ncap * esz[i];
    }
    ctx->res_cap = ncap;
    return VTX_OK;
}

int process_batch(vtx_ctx* ctx, const DevBatch& b, TimeRec* tr)
{
    const uint64_t nc = b.n_cand;
    const uint32_t nl = b.n_loci, nr = b.n_reads;
    const int use_umi = ctx->cfg.use_umi ? 1 : 0;
    uint64_t launches = 0, sw_launches = 0;
    cudaStream_t st = ctx->stream;

    if (ctx->finished) {      // fresh result set
        CK(cudaMemsetAsync(ctx->d_res_n.p, 0, 8, st));
        CK(cudaMemsetAsync(ctx->d_metrics.p, 0, 48, st));
        ctx->res_ub = 0;
        ctx->finished = false;
    }
    int rc = grow_results(ctx, ctx->res_ub + nc);
    if (rc) return rc;

    const size_t ncp = size_t(nc) + 1;
    ENS(ctx->read_col, size_t(nr ? nr : 1) * 4);
    ENS(ctx->keep, ncp * 4); ENS(ctx->pidx, ncp * 4);
    ENS(ctx->pair_read, ncp * 4); ENS(ctx->pair_col, ncp * 4);
    if (use_umi) ENS(ctx->pair_umi, ncp * 8);
    ENS(ctx->pair_start, size_t(nl + 1) * 4);
    ENS(ctx->pair_first, ncp);
    ENS(ctx->pair_cslot, ncp * 4); ENS(ctx->cslot_col, ncp * 4); ENS(ctx->cslot_locus, ncp * 4);
    ENS(ctx->ccnt, ncp * 16);
    if (use_umi) { ENS(ctx->pair_uslot, ncp * 4); ENS(ctx->uslot_cslot, ncp * 4); ENS(ctx->ucnt, ncp * 16); }
    ENS(ctx->keep2, ncp * 4); ENS(ctx->oidx, ncp * 4);
    uint32_t* pair_scores = nullptr;
    if (ctx->cfg.flags & VTX_F_KEEP_SCORES) { ENS(ctx->pair_scores, ncp * 4); pair_scores = P<uint32_t>(ctx->pair_scores); }

    if (nl == 0 || nc == 0) {
        if (ctx->d_cum && ctx->trec_used - 1 < kMaxCum)     // an empty shard still publishes the running triplet count
            vtx_k_bump<<<1, 32, 0, st>>>(P<unsigned long long>(ctx->d_res_n), nullptr, ctx->d_cum + (ctx->trec_used - 1));
        CK(cudaEventRecord(tr->ev[EV_PREP], st)); CK(cudaEventRecord(tr->ev[EV_SW], st)); CK(cudaEventRecord(tr->ev[EV_POST], st));
        ctx->timing_valid = true;
        return VTX_OK;
    }

    Nvtx r_prep("vtx: prep kernels (CB lookup, filter, compaction, slots)");
    // ---- K1: CB lookup, filter, compaction --------------------------------------------------------
    BarcodeTable tab{ P<int32_t>(ctx->bc_slot), ctx->bc_cap - 1, P<uint8_t>(ctx->bc_bytes), P<uint32_t>(ctx->bc_off) };
    if (b.read_cb_key) {
        BarcodeKeyTable kt{ P<uint64_t>(ctx->bck_key), P<uint32_t>(ctx->bck_idx), ctx->bck_cap - 1 };
        vtx_k_cb_lookup_key<<<blocks_for(nr, 256), 256, 0, st>>>(tab, kt, nr, b.read_cb_key, b.cb_bytes, b.cb_off_ex, P<int32_t>(ctx->read_col));
    } else {
        vtx_k_cb_lookup<<<blocks_for(nr, 256), 256, 0, st>>>(tab, nr, b.cb_bytes, b.read_cb_off, b.read_cb_len, P<int32_t>(ctx->read_col));
    }
    vtx_k_cand_filter<<<blocks_for(nc, 256), 256, 0, st>>>(nc, b.cand_read, P<int32_t>(ctx->read_col), b.read_umi, use_umi,
                                                           P<uint32_t>(ctx->keep), P<unsigned long long>(ctx->d_metrics));
    launches += 2;
    rc = scan_u32(ctx, P<uint32_t>(ctx->keep), nc, P<uint32_t>(ctx->pidx), &launches);
    if (rc) return rc;
    vtx_k_compact<<<blocks_for(nc, 256), 256, 0, st>>>(nc, b.cand_read, P<uint32_t>(ctx->keep), P<uint32_t>(ctx->pidx),
                                                       P<int32_t>(ctx->read_col), b.read_umi, use_umi, P<uint32_t>(ctx->pair_read),
                                                       P<uint32_t>(ctx->pair_col), P<uint64_t>(ctx->pair_umi));
    vtx_k_pair_start<<<blocks_for(nl + 1, 256), 256, 0, st>>>(nl, b.cand_start, P<uint32_t>(ctx->pidx), P<uint32_t>(ctx->pair_start));
    launches += 2;
    const uint32_t* n_pairs_ptr = P<uint32_t>(ctx->pidx) + nc;

    // ---- slots: the (row, col[, umi]) structure is independent of the alignment results ----------
    ENS(ctx->big_list, size_t(nc / kSlotSmallMax + 2) * 4);
    CK(cudaMemsetAsync(ctx->big_list.p, 0, 4, st));
    if (b.max_depth > kSlotSmallMax) ENS(ctx->slot_scratch, size_t(kSlotBigWords) * nc * 4);
    CK(cudaMemsetAsync(ctx->cslot_col.p, 0xFF, size_t(nc) * 4, st));
    CK(cudaMemsetAsync(ctx->ccnt.p, 0, size_t(nc) * 16, st));
    if (use_umi) {
        CK(cudaMemsetAsync(ctx->uslot_cslot.p, 0xFF, size_t(nc) * 4, st));
        CK(cudaMemsetAsync(ctx->ucnt.p, 0, size_t(nc) * 16, st));
    }
    vtx_k_slots<<<std::min<uint32_t>(nl, 65535u * 8), kSlotThreads, 0, st>>>(
        nl, P<uint32_t>(ctx->pair_start), P<uint32_t>(ctx->pair_col), P<uint64_t>(ctx->pair_umi), use_umi,
        P<uint8_t>(ctx->pair_first), P<uint32_t>(ctx->pair_cslot), P<uint32_t>(ctx->pair_uslot),
        P<uint32_t>(ctx->cslot_col), P<uint32_t>(ctx->cslot_locus), P<uint32_t>(ctx->uslot_cslot), P<uint32_t>(ctx->big_list));
    ++launches;
    if (nc > kSlotSmallMax) {       // a locus deeper than kSlotSmallMax pairs can only exist in such a shard
        vtx_k_slots_big<<<ctx->n_sm, kSlotBigThreads, 0, st>>>(
            P<uint32_t>(ctx->big_list), P<uint32_t>(ctx->pair_start), P<uint32_t>(ctx->pair_col), P<uint64_t>(ctx->pair_umi), use_umi,
            P<uint32_t>(ctx->slot_scratch), P<uint32_t>(ctx->pair_cslot), P<uint32_t>(ctx->pair_uslot), P<uint32_t>(ctx->cslot_col),
            P<uint32_t>(ctx->cslot_locus), P<uint32_t>(ctx->uslot_cslot));
        ++launches;
    }
    CK(cudaGetLastError());

    // ---- K2 + K3: Smith-Waterman, call, atomic scatter ----------------------------------------------
    nvtxRangePop(); nvtxRangePushA("vtx: Smith-Waterman kernels");
    rc = run_sw(ctx, b, uint32_t(nc), use_umi ? P<uint32_t>(ctx->pair_uslot) : P<uint32_t>(ctx->pair_cslot),
                use_umi ? P<uint32_t>(ctx->ucnt) : P<uint32_t>(ctx->ccnt), pair_scores, &launches, &sw_launches, tr);
    if (rc) return rc;
    CK(cudaEventRecord(tr->ev[EV_SW], st));

    // ---- K4 + K5: UMI collapse, mode value, row-major emit ------------------------------------------
    nvtxRangePop(); nvtxRangePushA("vtx: post kernels (UMI collapse, finalize, emit)");
    if (use_umi) {
        vtx_k_umi_collapse<<<blocks_for(nc, 256), 256, 0, st>>>(uint32_t(nc), n_pairs_ptr, P<uint32_t>(ctx->uslot_cslot),
                                                                P<uint32_t>(ctx->ucnt), P<uint32_t>(ctx->ccnt));
        ++launches;
    }
    vtx_k_finalize<<<blocks_for(nc, 256), 256, 0, st>>>(uint32_t(nc), n_pairs_ptr, ctx->cfg.mode, P<uint32_t>(ctx->cslot_col),
                                                        P<uint32_t>(ctx->ccnt), P<uint32_t>(ctx->keep2));
    ++launches;
    rc = scan_u32(ctx, P<uint32_t>(ctx->keep2), nc, P<uint32_t>(ctx->oidx), &launches);
    if (rc) return rc;
    if (ctx->gather_guard) {       // a gather started after the previous finish may still be reading the local result arrays
        CK(cudaStreamWaitEvent(st, ctx->ev_gather, 0));
        ctx->gather_guard = false;
    }
    ResultArrays out{ P<uint32_t>(ctx->r_row), P<uint32_t>(ctx->r_col), P<uint32_t>(ctx->r_ref), P<uint32_t>(ctx->r_alt),
                      P<uint32_t>(ctx->r_unk), P<double>(ctx->r_val), P<double>(ctx->r_val2) };
    vtx_k_emit<<<blocks_for(nc, 256), 256, 0, st>>>(uint32_t(nc), ctx->cfg.mode, P<uint32_t>(ctx->keep2), P<uint32_t>(ctx->oidx),
                                                    P<unsigned long long>(ctx->d_res_n), P<uint32_t>(ctx->cslot_col),
                                                    P<uint32_t>(ctx->cslot_locus), b.locus_row, P<uint32_t>(ctx->ccnt), out);
    const size_t sub_idx = ctx->trec_used - 1;       // this submit's slot
    vtx_k_bump<<<1, 32, 0, st>>>(P<unsigned long long>(ctx->d_res_n), P<uint32_t>(ctx->oidx) + nc,
                                 (ctx->d_cum && sub_idx < kMaxCum) ? ctx->d_cum + sub_idx : nullptr);
    launches += 2;
    CK(cudaGetLastError());
    CK(cudaEventRecord(tr->ev[EV_POST], st));
    ctx->res_ub += nc;
    ctx->timing_valid = true;
    tr->sw_launches = sw_launches;
    tr->launches = launches;
    return VTX_OK;
}

// One view of a host batch for validation, whichever layout it arrived in.
struct HostView {
    uint32_t n_loci = 0, n_reads = 0; uint64_t n_cand = 0;
    const uint32_t *locus_row = nullptr, *ref_off = nullptr, *ref_len = nullptr, *alt_off = nullptr, *alt_len = nullptr;
    const uint64_t* cand_start = nullptr; const uint8_t* hap = nullptr; uint64_t hap_len = 0;
    uint64_t nib_len = 0, cb_bytes_len = 0;
    const uint64_t* read_off = nullptr; const uint32_t* read_len = nullptr; const uint32_t* cb_off = nullptr; const uint16_t* cb_len = nullptr;   // vtx_batch
    const uint32_t* read_off4 = nullptr; const uint16_t* read_len16 = nullptr; const uint64_t* cb_key = nullptr;                                // vtx_batch2
    uint32_t n_exotic = 0; const uint32_t* cb_off_ex = nullptr;
    const uint64_t* umi = nullptr; const uint32_t* cand_read = nullptr;
    bool v2 = false;
};

HostView view_of(const vtx_batch* b)
{
    HostView v;
    v.n_loci = b->n_loci; v.n_reads = b->n_reads; v.n_cand = b->n_cand;
    v.locus_row = b->locus_row; v.ref_off = b->ref_off; v.ref_len = b->ref_len; v.alt_off = b->alt_off; v.alt_len = b->alt_len;
    v.cand_start = b->cand_start; v.hap = b->hap_bytes; v.hap_len = b->hap_bytes_len; v.nib_len = b->read_nib_len; v.cb_bytes_len = b->cb_bytes_len;
    v.read_off = b->read_off; v.read_len = b->read_len; v.cb_off = b->read_cb_off; v.cb_len = b->read_cb_len;
    v.umi = b->read_umi_key; v.cand_read = b->cand_read;
    return v;
}
HostView view_of(const vtx_batch2* b)
{
    HostView v;
    v.v2 = true;
    v.n_loci = b->n_loci; v.n_reads = b->n_reads; v.n_cand = b->n_cand;
    v.locus_row = b->locus_row; v.ref_off = b->ref_off; v.ref_len = b->ref_len; v.alt_off = b->alt_off; v.alt_len = b->alt_len;
    v.cand_start = b->cand_start; v.hap = b->hap_bytes; v.hap_len = b->hap_bytes_len; v.nib_len = b->read_nib_len;
    v.read_off4 = b->read_off4; v.read_len16 = b->read_len; v.cb_key = b->read_cb_key; v.n_exotic = b->n_exotic_cb; v.cb_off_ex = b->cb_off;
    v.cb_bytes_len = (b->n_exotic_cb && b->cb_off) ? b->cb_off[b->n_exotic_cb] : 0;
    v.umi = b->read_umi_key; v.cand_read = b->cand_read;
    return v;
}

int validate_batch(vtx_ctx* ctx, const HostView& b, bool device)
{
    if (b.n_cand >= 0xFFFFFFF0ull) return set_err(ctx, VTX_E_INVALID, "n_cand %llu exceeds 2^32 per shard; split the shard", (unsigned long long)b.n_cand);
    if (b.n_loci && (!b.locus_row || !b.ref_off || !b.ref_len || !b.alt_off || !b.alt_len || !b.cand_start))
        return set_err(ctx, VTX_E_INVALID, "locus arrays missing");
    if (b.n_reads) {
        const bool reads_ok = b.v2 ? (b.read_len16 && b.cb_key) : (b.read_off && b.read_len && b.cb_off && b.cb_len);
        if (!reads_ok || (!b.umi && ctx->cfg.use_umi)) return set_err(ctx, VTX_E_INVALID, "read arrays missing");
    }
    if (b.v2 && b.n_exotic && !b.cb_off_ex) return set_err(ctx, VTX_E_INVALID, "cb_off missing for the exotic cell tags");
    if (b.n_cand && !b.cand_read && !(b.v2 && b.n_cand == b.n_reads)) return set_err(ctx, VTX_E_INVALID, "cand_read missing (NULL means identity and needs n_cand == n_reads in a vtx_batch2)");
    if (b.hap_len >= 0xFFFFFFFFull) return set_err(ctx, VTX_E_INVALID, "haplotype pool exceeds 4 GiB; split the shard");
    if (b.v2 && b.nib_len >= (uint64_t(1) << 34)) return set_err(ctx, VTX_E_INVALID, "read pool exceeds 16 GiB; split the shard");
    (void)device;
    return VTX_OK;
}

// Which Smith-Waterman tile classes can get tiles, from the windows alone: the same decision tree as vtx_k_locus_prep,
// with the one input the host does not have (the longest SCORED read of a fold-shaped locus) resolved conservatively.
// Index of the per-locus shape: bit 0 exotic, bit 1 common prefix, bit 2 fold-shaped windows, bits 3.. single-phase
// class (kNumFastClasses = none), then the two-phase class (kNumSplitClasses = none).
constexpr int kShapeFast = 3, kShapeSplit = kShapeFast + 3, kNumShapes = 1 << (kShapeSplit + 2);
uint32_t shape_of(const uint8_t* rh, uint32_t nr, const uint8_t* ah, uint32_t na)
{
    // The alphabet test of vtx_k_locus_prep ("=MRSVWYHKDBN" bytes send a locus to the generic kernel) is not repeated on
    // the host -- a byte-wise scan of every window would cost more than the launch it can save: the generic class is
    // always launched, and bit 0 stays clear.
    const bool same = nr >= uint32_t(kSplitP) && na >= uint32_t(kSplitP) && memcmp(rh, ah, kSplitP) == 0;
    const bool fold = same && std::min(nr, na) > uint32_t(2 * kFoldP) && std::max(nr, na) <= uint32_t(2 * kFoldP + kFoldMaxMid) &&
                      memcmp(rh + nr - kFoldP, ah + na - kFoldP, kFoldP) == 0;
    const uint32_t nmax = std::max(nr, na);
    uint32_t fast = kNumFastClasses, split = kNumSplitClasses;
    for (int c = kNumFastClasses - 1; c >= 0; --c) if (nmax <= uint32_t(class_max_n(c))) fast = uint32_t(c);
    for (int c = kNumSplitClasses - 1; c >= 0; --c) if (nmax <= uint32_t(split_max_n(c))) split = uint32_t(c);
    return (uint32_t(same) << 1) | (uint32_t(fold) << 2) | (fast << kShapeFast) | (split << kShapeSplit);
}
uint32_t class_mask_of(const bool* seen, bool allow_split, bool allow_multi, bool allow_fold, uint32_t max_read)
{
    uint32_t mask = 1u << kSlowClass;          // loci with IUPAC / "=" bytes are only recognised on the device
    for (int i = 0; i < kNumShapes; ++i) {
        if (!seen[i]) continue;
        const bool exotic = i & 1, same = i & 2, fold = i & 4;
        const uint32_t fast = (uint32_t(i) >> kShapeFast) & 7u, split = (uint32_t(i) >> kShapeSplit) & 3u;
        int cls = kSlowClass;
        if (!exotic) {
            if (fast < uint32_t(kNumFastClasses)) cls = int(fast);
            else if (allow_multi) cls = kMultiClass;
            if (same && allow_split && split < uint32_t(kNumSplitClasses)) cls = kSplitClass0 + int(split);
            if (fold && allow_fold) {
                mask |= 1u << kFoldClass;
                if (max_read <= uint32_t(kFoldMaxRead)) continue;        // every read fits: the locus cannot fall back
            }
        }
        mask |= 1u << cls;
    }
    return mask;
}

// host-side checks that need to touch the (host) arrays; also returns max lengths.  Runs on a few host
// threads while the shard's H2D copies are already in flight (the kernels are only enqueued afterwards).
int scan_host_batch(vtx_ctx* ctx, const HostView& b, uint32_t* max_read, uint32_t* max_hap, bool check_cands,
                    uint64_t* max_depth = nullptr, bool* shapes_seen = nullptr)
{
    if (check_cands && b.n_loci && (b.cand_start[0] != 0 || b.cand_start[b.n_loci] != b.n_cand))
        return set_err(ctx, VTX_E_INVALID, "cand_start must span [0, n_cand]");
    if (check_cands && !b.n_loci && b.n_cand) return set_err(ctx, VTX_E_INVALID, "candidates without loci");
    if (b.v2 && b.n_exotic) {
        for (uint32_t i = 0; i < b.n_exotic; ++i)
            if (b.cb_off_ex[i] > b.cb_off_ex[i + 1]) return set_err(ctx, VTX_E_INVALID, "cb_off must be ascending (exotic tag %u)", i);
    }
    const bool scan_cands = check_cands && b.cand_read != nullptr;
    const uint64_t work = uint64_t(b.n_reads) + (scan_cands ? b.n_cand : 0) + uint64_t(b.n_loci) * 64;
    unsigned nt = std::min<unsigned>(8u, std::max(1u, std::thread::hardware_concurrency()));
    if (work < (1u << 16)) nt = 1;
    struct Part { uint32_t mr = 0, mh = 0; uint64_t md = 0, units = 0; int bad = 0; uint64_t where = 0; bool seen[kNumShapes] = {}; };
    std::vector<Part> parts(nt);
    auto worker = [&](unsigned t) {
        Part& pt = parts[t];
        auto flag = [&](int code, uint64_t where) { if (!pt.bad) { pt.bad = code; pt.where = where; } };
        const uint32_t l0 = uint32_t(uint64_t(b.n_loci) * t / nt), l1 = uint32_t(uint64_t(b.n_loci) * (t + 1) / nt);
        for (uint32_t l = l0; l < l1; ++l) {
            if ((b.ref_off[l] & 15) || (b.alt_off[l] & 15)) { flag(10, l); continue; }
            if (uint64_t(b.ref_off[l]) + b.ref_len[l] > b.hap_len || uint64_t(b.alt_off[l]) + b.alt_len[l] > b.hap_len) { flag(11, l); continue; }
            if (l && b.locus_row[l] <= b.locus_row[l - 1]) flag(12, l);
            if (check_cands && b.cand_start[l] > b.cand_start[l + 1]) flag(13, l);
            if (check_cands) pt.md = std::max<uint64_t>(pt.md, b.cand_start[l + 1] - b.cand_start[l]);
            pt.mh = std::max(pt.mh, std::max(b.ref_len[l], b.alt_len[l]));
            if (shapes_seen) pt.seen[shape_of(b.hap + b.ref_off[l], b.ref_len[l], b.hap + b.alt_off[l], b.alt_len[l])] = true;
        }
        const uint32_t r0 = uint32_t(uint64_t(b.n_reads) * t / nt), r1 = uint32_t(uint64_t(b.n_reads) * (t + 1) / nt);
        for (uint32_t r = r0; r < r1; ++r) {
            uint32_t len;
            if (b.v2) {
                len = b.read_len16[r];
                const uint64_t nb = (uint64_t(len) + 1) / 2;
                if (b.read_off4) { if (uint64_t(b.read_off4[r]) * 4 + nb > b.nib_len) flag(2, r); }
                else pt.units += (nb + 3) / 4;
                const uint64_t k = b.cb_key[r];
                if (k != VTX_NO_CB_KEY && (k & VTX_CB_EXOTIC) && (k & ~VTX_CB_EXOTIC) >= b.n_exotic) flag(3, r);
                else if (k != VTX_NO_CB_KEY && !(k & VTX_CB_EXOTIC) && (k >> 60)) flag(6, r);
            } else {
                len = b.read_len[r];
                if (b.read_off[r] & 15) flag(1, r);
                else if (b.read_off[r] + (uint64_t(len) + 1) / 2 > b.nib_len) flag(2, r);
                else if (b.cb_off[r] != VTX_NO_CB && uint64_t(b.cb_off[r]) + b.cb_len[r] > b.cb_bytes_len) flag(3, r);
            }
            if (b.umi && b.umi[r] != VTX_NO_UMI && b.umi[r] > VTX_UMI_KEY_MAX) flag(4, r);
            pt.mr = std::max(pt.mr, len);
        }
        if (scan_cands) {
            const uint64_t c0 = b.n_cand * t / nt, c1 = b.n_cand * (t + 1) / nt;
            uint32_t worst = 0;
            for (uint64_t c = c0; c < c1; ++c) worst = std::max(worst, b.cand_read[c]);
            if (c1 > c0 && worst >= b.n_reads) flag(5, c0);
        }
    };
    if (nt == 1) worker(0);
    else {
        std::vector<std::thread> th;
        for (unsigned t = 1; t < nt; ++t) th.emplace_back(worker, t);
        worker(0);
        for (auto& x : th) x.join();
    }
    uint32_t mr = 0, mh = 0;
    uint64_t md = 0, units = 0;
    for (const Part& pt : parts) {
        mr = std::max(mr, pt.mr); mh = std::max(mh, pt.mh); md = std::max(md, pt.md); units += pt.units;
        if (shapes_seen) for (int i = 0; i < kNumShapes; ++i) shapes_seen[i] |= pt.seen[i];
        const unsigned long long w = (unsigned long long)pt.where;
        switch (pt.bad) {
        case 1: return set_err(ctx, VTX_E_INVALID, "read %llu: read_off must be a multiple of 16", w);
        case 2: return set_err(ctx, VTX_E_INVALID, "read %llu outside read_nib", w);
        case 3: return set_err(ctx, VTX_E_INVALID, "read %llu: CB outside cb_bytes", w);
        case 4: return set_err(ctx, VTX_E_INVALID, "read %llu: UMI key exceeds VTX_UMI_KEY_MAX", w);
        case 5: return set_err(ctx, VTX_E_INVALID, "cand_read out of range near candidate %llu", w);
        case 6: return set_err(ctx, VTX_E_INVALID, "read %llu: read_cb_key is not a vtx_pack_cb code", w);
        case 10: return set_err(ctx, VTX_E_INVALID, "locus %llu: haplotype offsets must be multiples of 16", w);
        case 11: return set_err(ctx, VTX_E_INVALID, "locus %llu: haplotype window outside hap_bytes", w);
        case 12: return set_err(ctx, VTX_E_INVALID, "locus_row must be strictly ascending (locus %llu)", w);
        case 13: return set_err(ctx, VTX_E_INVALID, "cand_start must be ascending (locus %llu)", w);
        default: break;
        }
    }
    if (b.v2 && !b.read_off4 && units * 4 > b.nib_len) return set_err(ctx, VTX_E_INVALID, "dense read pool is shorter than the reads it should hold");
    if (mr > uint32_t(kMaxRead)) return set_err(ctx, VTX_E_UNSUPPORTED, "reads longer than %d bases (biased int16 DP) are not supported (%u)", kMaxRead, mr);
    *max_read = mr; *max_hap = mh;
    if (max_depth) *max_depth = md;
    return VTX_OK;
}

uint32_t host_class_mask(const vtx_ctx* ctx, const bool* shapes, uint32_t max_read, uint32_t max_hap)
{
    const SwAllow a = sw_allow(ctx, max_read, max_hap);
    return class_mask_of(shapes, a.split, a.multi, a.fold, max_read);
}

int upload(vtx_ctx* ctx, DBuf& d, const void* h, size_t bytes)
{
    ENS(d, bytes ? bytes : 16);
    if (bytes) CK(cudaMemcpyAsync(d.p, h, bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
    return VTX_OK;
}

#define UP(buf, ptr, bytes) do { int rc_ = upload(ctx, buf, ptr, (bytes)); if (rc_) return rc_; } while (0)

// claim the next input slot: its previous user's kernels must have finished before the copy may overwrite it
int claim_slot(vtx_ctx* ctx, InSlot** out)
{
    InSlot* sl = &ctx->slot[ctx->n_submits & 1];
    ++ctx->n_submits;
    if (sl->used) CK(cudaStreamWaitEvent(ctx->copy_stream, sl->free_ev, 0));
    sl->used = true;
    *out = sl;
    return VTX_OK;
}

int upload_common(vtx_ctx* ctx, InSlot* sl, const vtx_batch* hb, DevBatch& d)
{
    const uint32_t nl = hb->n_loci, nr = hb->n_reads;
    UP(sl->locus_row, hb->locus_row, size_t(nl) * 4);
    UP(sl->hap, hb->hap_bytes, hb->hap_bytes_len);
    UP(sl->ref_off, hb->ref_off, size_t(nl) * 4); UP(sl->ref_len, hb->ref_len, size_t(nl) * 4);
    UP(sl->alt_off, hb->alt_off, size_t(nl) * 4); UP(sl->alt_len, hb->alt_len, size_t(nl) * 4);
    UP(sl->read_nib, hb->read_nib, hb->read_nib_len);
    UP(sl->read_off, hb->read_off, size_t(nr) * 8); UP(sl->read_len, hb->read_len, size_t(nr) * 4);
    d.n_loci = nl; d.n_reads = nr;
    d.locus_row = P<uint32_t>(sl->locus_row); d.hap = P<uint8_t>(sl->hap);
    d.ref_off = P<uint32_t>(sl->ref_off); d.ref_len = P<uint32_t>(sl->ref_len);
    d.alt_off = P<uint32_t>(sl->alt_off); d.alt_len = P<uint32_t>(sl->alt_len);
    d.read_nib = P<uint8_t>(sl->read_nib); d.read_off = P<uint64_t>(sl->read_off); d.read_len = P<uint32_t>(sl->read_len);
    return VTX_OK;
}

}  // namespace

// =================================================================================================
extern "C" {

int vtx_abi_version(void) { return VTX_ABI_VERSION; }

const char* vtx_last_error(const vtx_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int vtx_create(const vtx_config* cfg, vtx_ctx** out)
{
    vtx_ctx* ctx = nullptr;   // for CK/set_err before the ctx exists
    if (!cfg || !out) return set_err(nullptr, VTX_E_INVALID, "vtx_create: NULL argument");
    *out = nullptr;
    if (cfg->match != kMatch || cfg->mismatch != kMismatch || cfg->gap_open != kGapOpen || cfg->gap_extend != kGapExtend)
        return set_err(nullptr, VTX_E_UNSUPPORTED, "scoring constants are compiled in: match %d mismatch %d gap_open %d gap_extend %d (main.rs:35-38)",
                       kMatch, kMismatch, kGapOpen, kGapExtend);
    if (cfg->mode < 0 || cfg->mode > 2) return set_err(nullptr, VTX_E_INVALID, "unknown mode %d", cfg->mode);
    if (cfg->band_mode != VTX_BAND_FULL && cfg->band_mode != VTX_BAND_MODEL) return set_err(nullptr, VTX_E_INVALID, "unknown band_mode %d", cfg->band_mode);
    if (cfg->band_k < 0 || cfg->band_k > 8 || cfg->band_w < 0 || cfg->band_w > 4096)
        return set_err(nullptr, VTX_E_UNSUPPORTED, "band constants out of range: K %d (1..8; 0 = %d), W %d (0 = %d; main.rs:33-34)", cfg->band_k, kBandK, cfg->band_w, kBandW);
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0)
        return set_err(nullptr, VTX_E_CUDA, "no CUDA device available (%s); vartrix_b200 has no CPU fallback", cudaGetErrorString(e));
    if (cfg->device < 0 || cfg->device >= n_dev) return set_err(nullptr, VTX_E_INVALID, "device %d out of range (%d devices)", cfg->device, n_dev);
    CK(cudaSetDevice(cfg->device));
    ctx = new vtx_ctx();
    ctx->cfg = *cfg; ctx->device = cfg->device;
    if (ctx->cfg.band_k == 0) ctx->cfg.band_k = kBandK;
    if (ctx->cfg.band_w == 0) ctx->cfg.band_w = kBandW;
    cudaDeviceProp prop{};
    cudaError_t pe = cudaGetDeviceProperties(&prop, cfg->device);
    if (pe != cudaSuccess) { g_create_error = cudaGetErrorString(pe); delete ctx; return VTX_E_CUDA; }
    if (prop.major < 9) { g_create_error = "vartrix_b200 needs DPX (sm_90+); built for sm_100a"; delete ctx; return VTX_E_UNSUPPORTED; }
    ctx->n_sm = prop.multiProcessorCount;
    if (cfg->stream) { ctx->stream = static_cast<cudaStream_t>(cfg->stream); ctx->own_stream = false; }
    else {
        pe = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
        if (pe != cudaSuccess) { g_create_error = cudaGetErrorString(pe); delete ctx; return VTX_E_CUDA; }
        ctx->own_stream = true;
    }
    pe = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
    if (pe != cudaSuccess) { g_create_error = cudaGetErrorString(pe); vtx_destroy(ctx); return VTX_E_CUDA; }
    cudaStreamCreateWithFlags(&ctx->fetch_stream, cudaStreamNonBlocking);
    if (cudaHostAlloc(reinterpret_cast<void**>(&ctx->h_cum), kMaxCum * 8, cudaHostAllocMapped) == cudaSuccess) {
        if (cudaHostGetDevicePointer(reinterpret_cast<void**>(&ctx->d_cum), ctx->h_cum, 0) != cudaSuccess) ctx->d_cum = nullptr;
    } else { ctx->h_cum = nullptr; cudaGetLastError(); }
    for (auto& sl : ctx->slot) {
        cudaEventCreateWithFlags(&sl.copy_done, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&sl.free_ev, cudaEventDisableTiming);
    }
    bool ok = cudaMalloc(&ctx->d_metrics.p, 64) == cudaSuccess && cudaMalloc(&ctx->d_res_n.p, 64) == cudaSuccess &&
              cudaHostAlloc(&ctx->h_scalars, 64, cudaHostAllocDefault) == cudaSuccess;
    if (!ok) { g_create_error = "allocation of context scalars failed"; vtx_destroy(ctx); return VTX_E_NOMEM; }
    ctx->d_metrics.cap = 64; ctx->d_res_n.cap = 64;
    cudaMemsetAsync(ctx->d_metrics.p, 0, 64, ctx->stream);
    cudaMemsetAsync(ctx->d_res_n.p, 0, 64, ctx->stream);
    *out = ctx;
    return VTX_OK;
}

void vtx_comm_destroy_internal(vtx_ctx* ctx);   // vtx_comm.cpp

void vtx_destroy(vtx_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->comm_stream) cudaStreamSynchronize(ctx->comm_stream);
    vtx_comm_destroy_internal(ctx);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    for (auto& sl : ctx->slot) {
        DBuf* sb[] = { &sl.locus_row, &sl.hap, &sl.ref_off, &sl.ref_len, &sl.alt_off, &sl.alt_len, &sl.cand_start, &sl.read_nib,
                       &sl.read_off, &sl.read_len, &sl.cb_bytes, &sl.read_cb_off, &sl.read_cb_len, &sl.read_umi, &sl.cand_read,
                       &sl.read_off4, &sl.read_len16, &sl.read_cb_key, &sl.cb_off_ex };
        for (DBuf* b : sb) if (b->p) cudaFree(b->p);
        if (sl.copy_done) cudaEventDestroy(sl.copy_done);
        if (sl.free_ev) cudaEventDestroy(sl.free_ev);
    }
    DBuf* all[] = { &ctx->bc_slot, &ctx->bc_bytes, &ctx->bc_off, &ctx->bck_key, &ctx->bck_idx, &ctx->x_read_off, &ctx->x_read_len,
                    &ctx->x_units, &ctx->x_off4, &ctx->band_scratch, &ctx->inf_comp, &ctx->inf_out, &ctx->inf_desc, &ctx->inf_status, &ctx->read_col,
                    &ctx->keep, &ctx->pidx, &ctx->scan_sums, &ctx->pair_read, &ctx->pair_col, &ctx->pair_umi, &ctx->pair_locus,
                    &ctx->pair_start, &ctx->tcount, &ctx->tstart, &ctx->pair_first, &ctx->pair_cslot, &ctx->pair_uslot, &ctx->cslot_col,
                    &ctx->cslot_locus, &ctx->uslot_cslot, &ctx->ccnt, &ctx->ucnt, &ctx->keep2, &ctx->oidx, &ctx->tile_counters,
                    &ctx->scratch, &ctx->pair_scores, &ctx->big_list, &ctx->slot_scratch, &ctx->d_metrics, &ctx->d_res_n, &ctx->r_row, &ctx->r_col, &ctx->r_ref,
                    &ctx->r_alt, &ctx->r_unk, &ctx->r_val, &ctx->r_val2, &ctx->g_counts };
    for (DBuf* b : all) if (b->p) cudaFree(b->p);
    for (auto& b : ctx->g_dev) if (b.p) cudaFree(b.p);
    if (ctx->stage_stream) { cudaStreamSynchronize(ctx->stage_stream); cudaStreamDestroy(ctx->stage_stream); }
    for (auto& ss : ctx->sslot) {
        DBuf* sb[] = { &ss.comp, &ss.desc, &ss.status, &ss.stream, &ss.entry, &ss.seg_count, &ss.seg_first, &ss.rec_off, &ss.rec_tid, &ss.rec_pos, &ss.rec_end,
                       &ss.rec_fm, &ss.l_start, &ss.l_end, &ss.locus_row, &ss.hap, &ss.ref_off, &ss.ref_len, &ss.alt_off, &ss.alt_len, &ss.cand_count,
                       &ss.cand_first, &ss.cand_rec, &ss.used, &ss.read_off, &ss.read_len, &ss.read_cb_off, &ss.read_cb_len, &ss.read_umi, &ss.cand_start, &ss.scalars };
        for (DBuf* b : sb) if (b->p) cudaFree(b->p);
        if (ss.staged) cudaEventDestroy(ss.staged);
        if (ss.free_ev) cudaEventDestroy(ss.free_ev);
    }
    if (ctx->bam_metrics.p) cudaFree(ctx->bam_metrics.p);
    if (ctx->stage_sums.p) cudaFree(ctx->stage_sums.p);
    if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
    for (void* h : ctx->h_res) if (h) cudaFreeHost(h);
    for (void* h : ctx->g_host) if (h) cudaFreeHost(h);
    if (ctx->h_scalars) cudaFreeHost(ctx->h_scalars);
    for (auto& tr : ctx->trecs) for (auto& ev : tr.ev) if (ev) cudaEventDestroy(ev);
    if (ctx->comm_stream) { cudaStreamSynchronize(ctx->comm_stream); cudaStreamDestroy(ctx->comm_stream); }
    for (cudaEvent_t e : { ctx->ev_counts, ctx->ev_gather, ctx->ev_results }) if (e) cudaEventDestroy(e);
    if (ctx->h_counts) cudaFreeHost(ctx->h_counts);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->fetch_stream) cudaStreamDestroy(ctx->fetch_stream);
    if (ctx->h_cum) cudaFreeHost(ctx->h_cum);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int vtx_host_alloc(void** out, uint64_t bytes)
{
    if (!out) return VTX_E_INVALID;
    cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 16, cudaHostAllocDefault);
    if (e != cudaSuccess) { g_create_error = cudaGetErrorString(e); *out = nullptr; return VTX_E_NOMEM; }
    return VTX_OK;
}

int vtx_host_free(void* p) { return cudaFreeHost(p) == cudaSuccess ? VTX_OK : VTX_E_CUDA; }

int vtx_set_barcodes(vtx_ctx* ctx, const uint8_t* bytes, const uint32_t* off, uint32_t n)
{
    if (!ctx) return VTX_E_INVALID;
    if (!off || (n && !bytes && off[n] > 0)) return set_err(ctx, VTX_E_INVALID, "vtx_set_barcodes: NULL argument");
    if (n == 0) return set_err(ctx, VTX_E_INVALID, "Loaded 0 barcodes (main.rs:712-715)");
    CK(cudaSetDevice(ctx->device));
    uint32_t cap = 16;
    while (cap < 2ull * n + 1) cap <<= 1;
    std::vector<int32_t> slot(cap, -1);
    for (uint32_t i = 0; i < n; ++i) {
        if (off[i + 1] < off[i]) return set_err(ctx, VTX_E_INVALID, "barcode offsets must be ascending");
        const uint32_t len = off[i + 1] - off[i];
        if (len > 0xFFFF) return set_err(ctx, VTX_E_INVALID, "barcode %u longer than 65535 bytes", i);
        uint32_t h = uint32_t(fnv1a64(bytes + off[i], len)) & (cap - 1);
        for (;;) {
            const int32_t s = slot[h];
            if (s < 0) { slot[h] = int32_t(i); break; }
            const uint32_t l2 = off[s + 1] - off[s];
            if (l2 == len && memcmp(bytes + off[s], bytes + off[i], len) == 0)
                return set_err(ctx, VTX_E_INVALID, "duplicate barcode at index %u (first seen at %d); dedup first (main.rs:706-709)", i, s);
            h = (h + 1) & (cap - 1);
        }
    }
    // second table for the slim layout: the barcodes that have a vtx_pack_cb code, keyed by the code
    std::vector<uint64_t> kkey(cap, kNoCbKey);
    std::vector<uint32_t> kidx(cap, 0);
    for (uint32_t i = 0; i < n; ++i) {
        const uint64_t k = pack_cb(bytes + off[i], off[i + 1] - off[i]);
        if (k == kNoCbKey) continue;
        uint32_t h = uint32_t(mix64(k)) & (cap - 1);
        while (kkey[h] != kNoCbKey) h = (h + 1) & (cap - 1);       // codes are injective and the strings distinct: no equal key
        kkey[h] = k; kidx[h] = i;
    }
    UP(ctx->bc_slot, slot.data(), size_t(cap) * 4);
    UP(ctx->bc_bytes, bytes, off[n]);
    UP(ctx->bc_off, off, size_t(n + 1) * 4);
    UP(ctx->bck_key, kkey.data(), size_t(cap) * 8);
    UP(ctx->bck_idx, kidx.data(), size_t(cap) * 4);
    CK(cudaStreamSynchronize(ctx->copy_stream));   // the tables are locals; they must be resident before any submit
    ctx->bc_cap = cap; ctx->bck_cap = cap; ctx->n_barcodes = n; ctx->have_barcodes = true;
    return VTX_OK;
}

int vtx_submit(vtx_ctx* ctx, const vtx_batch* hb)
{
    Nvtx nvtx_range("vtx_submit");
    if (!ctx) return VTX_E_INVALID;
    if (!ctx->have_barcodes) return set_err(ctx, VTX_E_STATE, "vtx_set_barcodes must be called before vtx_submit");
    if (!hb) return set_err(ctx, VTX_E_INVALID, "batch is NULL");
    const HostView hv = view_of(hb);
    int rc = validate_batch(ctx, hv, false);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    TimeRec* tr = new_trec(ctx);
    if (!tr) return set_err(ctx, VTX_E_CUDA, "cudaEventCreate failed");
    InSlot* sl = nullptr;
    rc = claim_slot(ctx, &sl);
    if (rc) return rc;
    // 1. start the copies of this shard on the copy stream (they overlap the previous shard's kernels) ...
    DevBatch d{};
    CK(cudaEventRecord(tr->ev[EV_START], ctx->copy_stream));
    rc = upload_common(ctx, sl, hb, d);
    if (rc) return rc;
    const uint32_t nl = hb->n_loci, nr = hb->n_reads;
    UP(sl->cand_start, hb->cand_start, size_t(nl + 1) * 8);
    UP(sl->cb_bytes, hb->cb_bytes, hb->cb_bytes_len);
    UP(sl->read_cb_off, hb->read_cb_off, size_t(nr) * 4); UP(sl->read_cb_len, hb->read_cb_len, size_t(nr) * 2);
    if (hb->read_umi_key) UP(sl->read_umi, hb->read_umi_key, size_t(nr) * 8);
    UP(sl->cand_read, hb->cand_read, size_t(hb->n_cand) * 4);
    CK(cudaEventRecord(tr->ev[EV_H2D], ctx->copy_stream));
    CK(cudaEventRecord(sl->copy_done, ctx->copy_stream));
    tr->had_h2d = true;
    d.n_cand = hb->n_cand;
    d.cand_start = P<uint64_t>(sl->cand_start); d.cb_bytes = P<uint8_t>(sl->cb_bytes);
    d.read_cb_off = P<uint32_t>(sl->read_cb_off); d.read_cb_len = P<uint16_t>(sl->read_cb_len);
    d.read_umi = hb->read_umi_key ? P<uint64_t>(sl->read_umi) : nullptr; d.cand_read = P<uint32_t>(sl->cand_read);
    // 2. ... validate the host arrays meanwhile; nothing has been launched on them yet
    bool shapes[kNumShapes] = {};
    { Nvtx r_val("vtx: validate host batch (copies in flight)");
      rc = scan_host_batch(ctx, hv, &d.max_read_len, &d.max_hap_len, true, &d.max_depth, shapes); }
    if (rc) { cudaStreamSynchronize(ctx->copy_stream); --ctx->trec_used; return rc; }
    d.class_mask = host_class_mask(ctx, shapes, d.max_read_len, d.max_hap_len);
    // 3. kernels wait for the copy, and release the slot when done
    CK(cudaStreamWaitEvent(ctx->stream, sl->copy_done, 0));
    CK(cudaEventRecord(tr->ev[EV_C0], ctx->stream));
    rc = process_batch(ctx, d, tr);
    if (rc) return rc;
    CK(cudaEventRecord(sl->free_ev, ctx->stream));
    return VTX_OK;
}

// device batches carry their own bounds in the (otherwise unused) *_len fields of the pools:
// the caller must pass max read / haplotype lengths through vtx_submit_device_ex.
int vtx_submit_device_ex(vtx_ctx* ctx, const vtx_batch* db, uint32_t max_read_len, uint32_t max_hap_len)
{
    if (!ctx) return VTX_E_INVALID;
    if (!ctx->have_barcodes) return set_err(ctx, VTX_E_STATE, "vtx_set_barcodes must be called before vtx_submit_device");
    if (!db) return set_err(ctx, VTX_E_INVALID, "batch is NULL");
    int rc = validate_batch(ctx, view_of(db), true);
    if (rc) return rc;
    if (max_read_len > uint32_t(kMaxRead)) return set_err(ctx, VTX_E_UNSUPPORTED, "reads longer than %d bases are not supported", kMaxRead);
    CK(cudaSetDevice(ctx->device));
    DevBatch d{};
    d.n_loci = db->n_loci; d.n_reads = db->n_reads; d.n_cand = db->n_cand;
    d.locus_row = db->locus_row; d.hap = db->hap_bytes; d.ref_off = db->ref_off; d.ref_len = db->ref_len;
    d.alt_off = db->alt_off; d.alt_len = db->alt_len; d.cand_start = db->cand_start; d.read_nib = db->read_nib;
    d.read_off = db->read_off; d.read_len = db->read_len; d.cb_bytes = db->cb_bytes; d.read_cb_off = db->read_cb_off;
    d.read_cb_len = db->read_cb_len; d.read_umi = db->read_umi_key; d.cand_read = db->cand_read;
    d.max_read_len = max_read_len; d.max_hap_len = max_hap_len;
    TimeRec* tr = new_trec(ctx);
    if (!tr) return set_err(ctx, VTX_E_CUDA, "cudaEventCreate failed");
    CK(cudaEventRecord(tr->ev[EV_C0], ctx->stream));
    return process_batch(ctx, d, tr);
}

int vtx_submit_device(vtx_ctx* ctx, const vtx_batch* db)
{
    // conservative bounds when the caller does not state them: the largest fast-path read and the
    // widest haplotype any tile class takes (wider inputs need vtx_submit_device_ex)
    return vtx_submit_device_ex(ctx, db, kFastMaxRead, class_max_n(kNumFastClasses - 1));
}

// ---- slim layout -------------------------------------------------------------------------------------------------
namespace {
// slim read arrays (device) -> the engine's internal read_off (u64 bytes) / read_len (u32)
int expand_reads(vtx_ctx* ctx, uint32_t nr, const uint16_t* d_len16, const uint32_t* d_off4, DevBatch& d, uint64_t* launches_unused = nullptr)
{
    (void)launches_unused;
    ENS(ctx->x_read_off, size_t(nr ? nr : 1) * 8); ENS(ctx->x_read_len, size_t(nr ? nr : 1) * 4);
    if (nr) {
        if (!d_off4) {          // dense pool: offsets are the running sum of the 4-byte units of the reads before
            ENS(ctx->x_units, size_t(nr) * 4); ENS(ctx->x_off4, size_t(nr + 1) * 4);
            vtx_k_read_units<<<blocks_for(nr, 256), 256, 0, ctx->stream>>>(nr, d_len16, P<uint32_t>(ctx->x_units));
            int rc = scan_u32(ctx, P<uint32_t>(ctx->x_units), nr, P<uint32_t>(ctx->x_off4), nullptr);
            if (rc) return rc;
            d_off4 = P<uint32_t>(ctx->x_off4);
        }
        vtx_k_expand_reads<<<blocks_for(nr, 256), 256, 0, ctx->stream>>>(nr, d_len16, d_off4, P<uint64_t>(ctx->x_read_off), P<uint32_t>(ctx->x_read_len));
        CK(cudaGetLastError());
    }
    d.read_off = P<uint64_t>(ctx->x_read_off); d.read_len = P<uint32_t>(ctx->x_read_len);
    return VTX_OK;
}
}  // namespace

int vtx_submit2(vtx_ctx* ctx, const vtx_batch2* hb)
{
    Nvtx nvtx_range("vtx_submit2");
    if (!ctx) return VTX_E_INVALID;
    if (!ctx->have_barcodes) return set_err(ctx, VTX_E_STATE, "vtx_set_barcodes must be called before vtx_submit2");
    if (!hb) return set_err(ctx, VTX_E_INVALID, "batch is NULL");
    const HostView hv = view_of(hb);
    int rc = validate_batch(ctx, hv, false);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    TimeRec* tr = new_trec(ctx);
    if (!tr) return set_err(ctx, VTX_E_CUDA, "cudaEventCreate failed");
    InSlot* sl = nullptr;
    rc = claim_slot(ctx, &sl);
    if (rc) return rc;
    DevBatch d{};
    const uint32_t nl = hb->n_loci, nr = hb->n_reads;
    CK(cudaEventRecord(tr->ev[EV_START], ctx->copy_stream));
    UP(sl->locus_row, hb->locus_row, size_t(nl) * 4);
    UP(sl->hap, hb->hap_bytes, hb->hap_bytes_len);
    UP(sl->ref_off, hb->ref_off, size_t(nl) * 4); UP(sl->ref_len, hb->ref_len, size_t(nl) * 4);
    UP(sl->alt_off, hb->alt_off, size_t(nl) * 4); UP(sl->alt_len, hb->alt_len, size_t(nl) * 4);
    UP(sl->cand_start, hb->cand_start, size_t(nl + 1) * 8);
    UP(sl->read_nib, hb->read_nib, hb->read_nib_len);
    if (hb->read_off4) UP(sl->read_off4, hb->read_off4, size_t(nr) * 4);
    UP(sl->read_len16, hb->read_len, size_t(nr) * 2);
    UP(sl->read_cb_key, hb->read_cb_key, size_t(nr) * 8);
    if (hb->n_exotic_cb) { UP(sl->cb_bytes, hb->cb_bytes, hv.cb_bytes_len); UP(sl->cb_off_ex, hb->cb_off, size_t(hb->n_exotic_cb + 1) * 4); }
    if (hb->read_umi_key) UP(sl->read_umi, hb->read_umi_key, size_t(nr) * 8);
    if (hb->cand_read) UP(sl->cand_read, hb->cand_read, size_t(hb->n_cand) * 4);
    CK(cudaEventRecord(tr->ev[EV_H2D], ctx->copy_stream));
    CK(cudaEventRecord(sl->copy_done, ctx->copy_stream));
    tr->had_h2d = true;
    d.n_loci = nl; d.n_reads = nr; d.n_cand = hb->n_cand;
    d.locus_row = P<uint32_t>(sl->locus_row); d.hap = P<uint8_t>(sl->hap);
    d.ref_off = P<uint32_t>(sl->ref_off); d.ref_len = P<uint32_t>(sl->ref_len);
    d.alt_off = P<uint32_t>(sl->alt_off); d.alt_len = P<uint32_t>(sl->alt_len);
    d.cand_start = P<uint64_t>(sl->cand_start); d.read_nib = P<uint8_t>(sl->read_nib);
    d.read_cb_key = P<uint64_t>(sl->read_cb_key);
    d.cb_bytes = hb->n_exotic_cb ? P<uint8_t>(sl->cb_bytes) : nullptr; d.cb_off_ex = hb->n_exotic_cb ? P<uint32_t>(sl->cb_off_ex) : nullptr;
    d.read_cb_off = nullptr; d.read_cb_len = nullptr;
    d.read_umi = hb->read_umi_key ? P<uint64_t>(sl->read_umi) : nullptr;
    d.cand_read = hb->cand_read ? P<uint32_t>(sl->cand_read) : nullptr;
    bool shapes[kNumShapes] = {};
    { Nvtx r_val("vtx: validate host batch (copies in flight)");
      rc = scan_host_batch(ctx, hv, &d.max_read_len, &d.max_hap_len, true, &d.max_depth, shapes); }
    if (rc) { cudaStreamSynchronize(ctx->copy_stream); --ctx->trec_used; return rc; }
    d.class_mask = host_class_mask(ctx, shapes, d.max_read_len, d.max_hap_len);
    CK(cudaStreamWaitEvent(ctx->stream, sl->copy_done, 0));
    CK(cudaEventRecord(tr->ev[EV_C0], ctx->stream));
    rc = expand_reads(ctx, nr, P<uint16_t>(sl->read_len16), hb->read_off4 ? P<uint32_t>(sl->read_off4) : nullptr, d);
    if (rc) return rc;
    rc = process_batch(ctx, d, tr);
    if (rc) return rc;
    CK(cudaEventRecord(sl->free_ev, ctx->stream));
    return VTX_OK;
}

int vtx_submit2_device(vtx_ctx* ctx, const vtx_batch2* db, uint32_t max_read_len, uint32_t max_hap_len)
{
    if (!ctx) return VTX_E_INVALID;
    if (!ctx->have_barcodes) return set_err(ctx, VTX_E_STATE, "vtx_set_barcodes must be called before vtx_submit2_device");
    if (!db) return set_err(ctx, VTX_E_INVALID, "batch is NULL");
    HostView hv = view_of(db); hv.cb_bytes_len = 0;       // device pointers: nothing may be dereferenced here
    hv.cb_off_ex = db->cb_off;
    int rc = validate_batch(ctx, hv, true);
    if (rc) return rc;
    if (max_read_len > uint32_t(kMaxRead)) return set_err(ctx, VTX_E_UNSUPPORTED, "reads longer than %d bases are not supported", kMaxRead);
    CK(cudaSetDevice(ctx->device));
    DevBatch d{};
    d.n_loci = db->n_loci; d.n_reads = db->n_reads; d.n_cand = db->n_cand;
    d.locus_row = db->locus_row; d.hap = db->hap_bytes; d.ref_off = db->ref_off; d.ref_len = db->ref_len;
    d.alt_off = db->alt_off; d.alt_len = db->alt_len; d.cand_start = db->cand_start; d.read_nib = db->read_nib;
    d.read_cb_key = db->read_cb_key; d.cb_bytes = db->cb_bytes; d.cb_off_ex = db->cb_off; d.read_cb_off = nullptr; d.read_cb_len = nullptr;
    d.read_umi = db->read_umi_key; d.cand_read = db->cand_read;
    d.max_read_len = max_read_len; d.max_hap_len = max_hap_len;
    TimeRec* tr = new_trec(ctx);
    if (!tr) return set_err(ctx, VTX_E_CUDA, "cudaEventCreate failed");
    CK(cudaEventRecord(tr->ev[EV_C0], ctx->stream));
    rc = expand_reads(ctx, db->n_reads, db->read_len, db->read_off4, d);
    if (rc) return rc;
    return process_batch(ctx, d, tr);
}

static int inflate_attr(vtx_ctx* ctx)        // the inflate kernel's tables + input windows need the opt-in shared-memory size
{
    if (ctx->inflate_attr_set) return VTX_OK;
    CK(cudaFuncSetAttribute(inflate::vtx_k_bgzf_inflate, cudaFuncAttributeMaxDynamicSharedMemorySize, int(inflate::inflate_smem_bytes())));
    ctx->inflate_attr_set = true;
    return VTX_OK;
}

int vtx_bgzf_inflate(vtx_ctx* ctx, const vtx_bgzf_block* blocks, uint32_t n_blocks, const uint8_t* comp, uint64_t comp_len,
                     uint8_t* out, uint64_t out_len, int32_t* status, uint32_t flags)
{
    if (!ctx) return VTX_E_INVALID;
    Nvtx nvtx_range("vtx_bgzf_inflate");
    if (n_blocks == 0) return VTX_OK;
    if (!blocks || !comp || !status || (!out && out_len)) return set_err(ctx, VTX_E_INVALID, "vtx_bgzf_inflate: NULL argument");
    static_assert(sizeof(vtx_bgzf_block) == sizeof(inflate::BlockDesc), "descriptor layouts must agree");
    for (uint32_t i = 0; i < n_blocks; ++i) {
        const vtx_bgzf_block& b = blocks[i];
        if ((b.in_off & 3) || b.in_off + b.in_len + 8 > comp_len + 8 || b.in_off + b.in_len > comp_len)
            return set_err(ctx, VTX_E_INVALID, "vtx_bgzf_inflate: member %u: payload must start on a 4-byte boundary inside comp", i);
        if (b.out_len > 65536u || b.out_off + b.out_len > out_len) return set_err(ctx, VTX_E_INVALID, "vtx_bgzf_inflate: member %u: output outside out / ISIZE above 64 KiB", i);
    }
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    ENS(ctx->inf_comp, size_t(comp_len) + 16); ENS(ctx->inf_out, size_t(out_len) + 16);
    ENS(ctx->inf_desc, size_t(n_blocks) * sizeof(vtx_bgzf_block)); ENS(ctx->inf_status, size_t(n_blocks) * 4 + 16);
    ENS(ctx->tile_counters, 64);
    CK(cudaMemsetAsync(static_cast<uint8_t*>(ctx->inf_comp.p) + comp_len, 0, 16, st));              // the readable padding
    CK(cudaMemcpyAsync(ctx->inf_comp.p, comp, comp_len, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->inf_desc.p, blocks, size_t(n_blocks) * sizeof(vtx_bgzf_block), cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(ctx->tile_counters.p, 0, 64, st));
    const unsigned ctas = unsigned(std::min<uint64_t>((n_blocks + inflate::kInflateWarps - 1) / inflate::kInflateWarps, uint64_t(ctx->n_sm) * 6));
    if (int rc_attr = inflate_attr(ctx)) return rc_attr;
    inflate::vtx_k_bgzf_inflate<<<ctas, inflate::kInflateWarps * 32, inflate::inflate_smem_bytes(), st>>>(
        P<inflate::BlockDesc>(ctx->inf_desc), n_blocks, P<uint8_t>(ctx->inf_comp), P<uint8_t>(ctx->inf_out), P<int32_t>(ctx->inf_status),
        P<uint32_t>(ctx->tile_counters), (flags & VTX_BGZF_CHECK_CRC) ? 1 : 0);
    CK(cudaGetLastError());
    if (out_len) CK(cudaMemcpyAsync(out, ctx->inf_out.p, out_len, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(status, ctx->inf_status.p, size_t(n_blocks) * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (uint32_t i = 0; i < n_blocks; ++i)
        if (status[i] != 0) return set_err(ctx, VTX_E_INVALID, "vtx_bgzf_inflate: member %u failed with decoder status %d (corrupt data)", i, status[i]);
    return VTX_OK;
}

// -------------------------------------------------------------------------------------------------
// vtx_submit_bam: inflate + record scan + fetch + filters + tags on the device (vtx_inflate.cuh, vtx_stage.cuh)
// -------------------------------------------------------------------------------------------------
namespace {
int scan_u32_on(vtx_ctx* ctx, cudaStream_t st, const uint32_t* in, uint64_t n, uint32_t* out, DBuf& sums)
{
    const unsigned nb = std::max(1u, blocks_for(n, kScanTile));
    int rc = ensure(ctx, sums, size_t(nb) * 4);
    if (rc) return rc;
    vtx_k_scan_tiles<<<nb, kScanThreads, 0, st>>>(in, n, out, P<uint32_t>(sums));
    vtx_k_scan_sums<<<1, kScanThreads, 0, st>>>(P<uint32_t>(sums), nb, out + n);
    vtx_k_scan_add<<<nb, kScanThreads, 0, st>>>(out, n, P<uint32_t>(sums));
    CK(cudaGetLastError());
    return VTX_OK;
}
}  // namespace

int vtx_submit_bam(vtx_ctx* ctx, const vtx_bam_shard* sh)
{
    if (!ctx) return VTX_E_INVALID;
    Nvtx nvtx_range("vtx_submit_bam");
    if (!ctx->have_barcodes) return set_err(ctx, VTX_E_STATE, "vtx_set_barcodes must be called before vtx_submit_bam");
    if (!sh) return set_err(ctx, VTX_E_INVALID, "shard is NULL");
    const uint32_t nl = sh->n_loci, nm = sh->n_members, ne = sh->n_entry;
    if (nl && (!sh->locus_row || !sh->locus_start || !sh->locus_end || !sh->ref_off || !sh->ref_len || !sh->alt_off || !sh->alt_len))
        return set_err(ctx, VTX_E_INVALID, "vtx_submit_bam: locus arrays missing");
    if (nm && (!sh->members || !sh->comp)) return set_err(ctx, VTX_E_INVALID, "vtx_submit_bam: members missing");
    if ((ne == 1) || (ne && !sh->entry_off)) return set_err(ctx, VTX_E_INVALID, "vtx_submit_bam: entry_off needs at least a start and an end");
    if (sh->hap_bytes_len >= 0xFFFFFFFFull) return set_err(ctx, VTX_E_INVALID, "haplotype pool exceeds 4 GiB; split the shard");
    uint64_t stream_len = 0;
    uint32_t max_hap = 0;
    for (uint32_t i = 0; i < nm; ++i) {
        const vtx_bgzf_block& b = sh->members[i];
        if ((b.in_off & 3) || b.in_off + b.in_len > sh->comp_len || b.out_len > 65536u || b.out_off != stream_len)
            return set_err(ctx, VTX_E_INVALID, "vtx_submit_bam: member %u: payload on a 4-byte boundary inside comp, out_off = running sum of out_len", i);
        stream_len += b.out_len;
    }
    if (stream_len >= 0xFFFFFFFFull) return set_err(ctx, VTX_E_INVALID, "vtx_submit_bam: more than 4 GiB of records in one shard; split the shard");
    for (uint32_t i = 0; i < ne; ++i)
        if (sh->entry_off[i] > stream_len || (i && sh->entry_off[i] <= sh->entry_off[i - 1])) return set_err(ctx, VTX_E_INVALID, "vtx_submit_bam: entry_off must ascend inside the stream");
    for (uint32_t l = 0; l < nl; ++l) {
        if ((sh->ref_off[l] & 15) || (sh->alt_off[l] & 15) || uint64_t(sh->ref_off[l]) + sh->ref_len[l] > sh->hap_bytes_len ||
            uint64_t(sh->alt_off[l]) + sh->alt_len[l] > sh->hap_bytes_len) return set_err(ctx, VTX_E_INVALID, "vtx_submit_bam: locus %u: bad haplotype window", l);
        if (l && (sh->locus_row[l] <= sh->locus_row[l - 1])) return set_err(ctx, VTX_E_INVALID, "locus_row must be strictly ascending (locus %u)", l);
        max_hap = std::max(max_hap, std::max(sh->ref_len[l], sh->alt_len[l]));
    }
    CK(cudaSetDevice(ctx->device));
    if (!ctx->stage_stream) {
        CK(cudaStreamCreateWithFlags(&ctx->stage_stream, cudaStreamNonBlocking));
        for (auto& ss : ctx->sslot) { CK(cudaEventCreateWithFlags(&ss.staged, cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&ss.free_ev, cudaEventDisableTiming)); }
        ENS(ctx->bam_metrics, sizeof(stage::LocusMetrics));
        CK(cudaMemsetAsync(ctx->bam_metrics.p, 0, sizeof(stage::LocusMetrics), ctx->stage_stream));
        CK(cudaHostAlloc(reinterpret_cast<void**>(&ctx->h_stage), 256, cudaHostAllocDefault));
    }
    cudaStream_t ss = ctx->stage_stream;
    StageSlot& sl = ctx->sslot[ctx->n_bam_submits & 1];
    ++ctx->n_bam_submits;
    if (sl.used_once) CK(cudaEventSynchronize(sl.free_ev));       // the kernels that read this slot's stream two shards ago are done
    sl.used_once = true;
    TimeRec* tr = new_trec(ctx);
    if (!tr) return set_err(ctx, VTX_E_CUDA, "cudaEventCreate failed");
    auto fail_out = [&](int code) { --ctx->trec_used; sl.used_once = false; return code; };

    // ---- copies (staging stream) ----
    auto up = [&](DBuf& d, const void* h, size_t bytes) -> int {
        int rc = ensure(ctx, d, bytes ? bytes + 16 : 16);
        if (rc) return rc;
        if (bytes && cudaMemcpyAsync(d.p, h, bytes, cudaMemcpyHostToDevice, ss) != cudaSuccess) return set_err(ctx, VTX_E_CUDA, "cudaMemcpyAsync failed in vtx_submit_bam");
        return VTX_OK;
    };
    CK(cudaEventRecord(tr->ev[EV_START], ss));
    int rc;
    if ((rc = up(sl.comp, sh->comp, sh->comp_len)) || (rc = up(sl.desc, sh->members, size_t(nm) * sizeof(vtx_bgzf_block))) ||
        (rc = up(sl.entry, sh->entry_off, size_t(ne) * 8)) || (rc = up(sl.l_start, sh->locus_start, size_t(nl) * 8)) ||
        (rc = up(sl.l_end, sh->locus_end, size_t(nl) * 8)) || (rc = up(sl.locus_row, sh->locus_row, size_t(nl) * 4)) ||
        (rc = up(sl.hap, sh->hap_bytes, sh->hap_bytes_len)) || (rc = up(sl.ref_off, sh->ref_off, size_t(nl) * 4)) ||
        (rc = up(sl.ref_len, sh->ref_len, size_t(nl) * 4)) || (rc = up(sl.alt_off, sh->alt_off, size_t(nl) * 4)) ||
        (rc = up(sl.alt_len, sh->alt_len, size_t(nl) * 4))) return fail_out(rc);
    CK(cudaMemsetAsync(static_cast<uint8_t*>(sl.comp.p) + sh->comp_len, 0, 16, ss));
    CK(cudaEventRecord(tr->ev[EV_H2D], ss));
    tr->had_h2d = true;
    // ---- inflate into one contiguous stream ----
    ENS(sl.stream, size_t(stream_len) + stage::kWalkWindow + 64);      // the walkers read whole windows
    ENS(sl.status, size_t(nm) * 4 + 16); ENS(sl.scalars, 256);
    uint32_t* d_sc = P<uint32_t>(sl.scalars);       // [0] walk cursor / inflate cursor, [1] err, [2] max_span, [3] max read, [4..] spare
    CK(cudaMemsetAsync(sl.scalars.p, 0, 256, ss));
    if (nm) {
        const unsigned ctas = unsigned(std::min<uint64_t>((nm + inflate::kInflateWarps - 1) / inflate::kInflateWarps, uint64_t(ctx->n_sm) * 6));
        if (int rc_attr = inflate_attr(ctx)) return fail_out(rc_attr);
        inflate::vtx_k_bgzf_inflate<<<ctas, inflate::kInflateWarps * 32, inflate::inflate_smem_bytes(), ss>>>(P<inflate::BlockDesc>(sl.desc), nm, P<uint8_t>(sl.comp), P<uint8_t>(sl.stream),
                                                                                 P<int32_t>(sl.status), d_sc, 1);
        CK(cudaGetLastError());
    }
    stage::Params sp{};
    sp.s = P<uint8_t>(sl.stream); sp.s_len = stream_len; sp.tid = sh->tid; sp.mapq_min = sh->mapq; sp.primary_only = sh->primary_only;
    sp.no_duplicates = sh->no_duplicates; sp.want_umi = ctx->cfg.use_umi ? 1 : 0; sp.tag0 = uint8_t(sh->bam_tag[0]); sp.tag1 = uint8_t(sh->bam_tag[1]);
    // ---- record boundaries ----
    const uint32_t n_seg = ne ? ne - 1 : 0;
    ENS(sl.seg_count, size_t(n_seg + 1) * 4); ENS(sl.seg_first, size_t(n_seg + 2) * 4);
    uint32_t n_rec = 0;
    std::vector<int32_t> h_status(nm);
    if (n_seg) {
        stage::vtx_k_walk<<<blocks_for(n_seg, stage::kWalkWarps), stage::kWalkWarps * 32, 0, ss>>>(sp, n_seg, P<uint64_t>(sl.entry), 0, P<uint32_t>(sl.seg_count), nullptr, nullptr, d_sc + 1);
        rc = scan_u32_on(ctx, ss, P<uint32_t>(sl.seg_count), n_seg, P<uint32_t>(sl.seg_first), ctx->stage_sums);
        if (rc) return fail_out(rc);
    }
    // wait #1 (staging stream only): inflate status, walk errors, number of records
    uint32_t* hs = reinterpret_cast<uint32_t*>(ctx->h_stage);
    if (n_seg) CK(cudaMemcpyAsync(hs, P<uint32_t>(sl.seg_first) + n_seg, 4, cudaMemcpyDeviceToHost, ss)); else hs[0] = 0;
    CK(cudaMemcpyAsync(hs + 1, d_sc + 1, 4, cudaMemcpyDeviceToHost, ss));
    if (nm) CK(cudaMemcpyAsync(h_status.data(), sl.status.p, size_t(nm) * 4, cudaMemcpyDeviceToHost, ss));
    CK(cudaStreamSynchronize(ss));
    for (uint32_t i = 0; i < nm; ++i)
        if (h_status[i] != 0) return fail_out(set_err(ctx, VTX_E_INVALID, "vtx_submit_bam: BGZF member %u failed with decoder status %d (corrupt data)", i, h_status[i]));
    if (hs[1] & (stage::kErrWalk | stage::kErrRecord))
        return fail_out(set_err(ctx, VTX_E_INVALID, "vtx_submit_bam: the record walk did not land on the index's record boundaries (corrupt BAM record or index; flags %u)", hs[1]));
    n_rec = hs[0];
    const size_t nrp = size_t(n_rec) + 1;
    ENS(sl.rec_off, nrp * 8); ENS(sl.rec_tid, nrp * 4); ENS(sl.rec_pos, nrp * 4); ENS(sl.rec_end, nrp * 4); ENS(sl.rec_fm, nrp * 4); ENS(sl.used, nrp * 4);
    ENS(sl.cand_count, size_t(nl + 1) * 4); ENS(sl.cand_first, size_t(nl + 2) * 4); ENS(sl.cand_start, size_t(nl + 2) * 8);
    stage::LocusMetrics* d_met = P<stage::LocusMetrics>(ctx->bam_metrics);
    uint64_t n_cand = 0;
    uint32_t max_read = 0;
    if (n_rec) {
        stage::vtx_k_walk<<<blocks_for(n_seg, stage::kWalkWarps), stage::kWalkWarps * 32, 0, ss>>>(sp, n_seg, P<uint64_t>(sl.entry), 1, nullptr, P<uint32_t>(sl.seg_first), P<uint64_t>(sl.rec_off), d_sc + 1);
        stage::vtx_k_parse<<<blocks_for(n_rec, 256), 256, 0, ss>>>(sp, n_rec, P<uint64_t>(sl.rec_off), P<int32_t>(sl.rec_tid), P<int32_t>(sl.rec_pos),
                                                                   P<int32_t>(sl.rec_end), P<uint32_t>(sl.rec_fm), d_sc + 2);
        CK(cudaMemsetAsync(sl.used.p, 0, nrp * 4, ss));
    }
    if (nl) {
        // counts first; the per-locus metric counters of this pass only become final if the shard is accepted, so they go to a scratch copy
        ENS(sl.status, std::max<size_t>(size_t(nm) * 4 + 16, sizeof(stage::LocusMetrics) + 16));
        stage::LocusMetrics* d_tmp = reinterpret_cast<stage::LocusMetrics*>(sl.status.p);
        CK(cudaMemsetAsync(d_tmp, 0, sizeof(stage::LocusMetrics), ss));
        stage::vtx_k_locus_cands<<<blocks_for(nl, 64), 64, 0, ss>>>(sp, nl, P<int64_t>(sl.l_start), P<int64_t>(sl.l_end), n_rec, P<uint64_t>(sl.rec_off),
                                                                   P<int32_t>(sl.rec_tid), P<int32_t>(sl.rec_pos), P<int32_t>(sl.rec_end), P<uint32_t>(sl.rec_fm),
                                                                   d_sc + 2, d_sc + 3, 0, P<uint32_t>(sl.cand_count), nullptr, nullptr, nullptr, d_tmp);
        rc = scan_u32_on(ctx, ss, P<uint32_t>(sl.cand_count), nl, P<uint32_t>(sl.cand_first), ctx->stage_sums);
        if (rc) return fail_out(rc);
        CK(cudaMemcpyAsync(hs, P<uint32_t>(sl.cand_first) + nl, 4, cudaMemcpyDeviceToHost, ss));
    } else hs[0] = 0;
    CK(cudaMemcpyAsync(hs + 1, d_sc + 1, 12, cudaMemcpyDeviceToHost, ss));      // err, max_span, max read
    CK(cudaStreamSynchronize(ss));                                               // wait #2: number of candidates, longest read
    n_cand = hs[0]; max_read = hs[3];
    if (hs[1] & (stage::kErrWalk | stage::kErrRecord)) return fail_out(set_err(ctx, VTX_E_INVALID, "vtx_submit_bam: corrupt BAM record (flags %u)", hs[1]));
    if (max_read > uint32_t(kMaxRead)) return fail_out(set_err(ctx, VTX_E_UNSUPPORTED, "reads longer than %d bases (biased int16 DP) are not supported (%u)", kMaxRead, max_read));
    if (n_cand >= 0xFFFFFFF0ull) return fail_out(set_err(ctx, VTX_E_INVALID, "n_cand exceeds 2^32 per shard; split the shard"));
    const size_t ncp = size_t(n_cand) + 1;
    ENS(sl.cand_rec, ncp * 4); ENS(sl.read_off, nrp * 8); ENS(sl.read_len, nrp * 4); ENS(sl.read_cb_off, nrp * 4); ENS(sl.read_cb_len, nrp * 2 + 2);
    if (ctx->cfg.use_umi) ENS(sl.read_umi, nrp * 8);
    if (nl) {
        stage::LocusMetrics* d_tmp = reinterpret_cast<stage::LocusMetrics*>(sl.status.p);
        stage::vtx_k_locus_cands<<<blocks_for(nl, 64), 64, 0, ss>>>(sp, nl, P<int64_t>(sl.l_start), P<int64_t>(sl.l_end), n_rec, P<uint64_t>(sl.rec_off),
                                                                   P<int32_t>(sl.rec_tid), P<int32_t>(sl.rec_pos), P<int32_t>(sl.rec_end), P<uint32_t>(sl.rec_fm),
                                                                   d_sc + 2, d_sc + 3, 1, nullptr, P<uint32_t>(sl.cand_first), P<uint32_t>(sl.cand_rec), P<uint32_t>(sl.used), d_tmp);
        stage::vtx_k_widen<<<blocks_for(nl + 1, 256), 256, 0, ss>>>(nl + 1, P<uint32_t>(sl.cand_first), P<uint64_t>(sl.cand_start));
    }
    if (n_rec)
        stage::vtx_k_read_emit<<<blocks_for(n_rec, 128), 128, 0, ss>>>(sp, n_rec, P<uint64_t>(sl.rec_off), P<uint32_t>(sl.used), P<uint64_t>(sl.read_off),
                                                                       P<uint32_t>(sl.read_len), P<uint32_t>(sl.read_cb_off), P<uint16_t>(sl.read_cb_len),
                                                                       P<uint64_t>(sl.read_umi), d_sc + 1);
    CK(cudaGetLastError());
    if (ctx->cfg.use_umi && n_rec) {      // wait #3 only with --umi: a UB string the device cannot key sends the shard back to the host
        CK(cudaMemcpyAsync(hs + 1, d_sc + 1, 4, cudaMemcpyDeviceToHost, ss));
        CK(cudaStreamSynchronize(ss));
        if (hs[1] & stage::kErrExoticUmi) return fail_out(set_err(ctx, VTX_E_UNSUPPORTED, "vtx_submit_bam: a UB tag outside vtx_pack_umi's alphabet needs the host's interner; stage this shard on the host"));
    }
    if (nl) {                             // the shard is accepted: its filter counters join the running totals
        stage::LocusMetrics* d_tmp = reinterpret_cast<stage::LocusMetrics*>(sl.status.p);
        vtx_k_add_u64<<<1, 32, 0, ss>>>(reinterpret_cast<unsigned long long*>(d_met), reinterpret_cast<const unsigned long long*>(d_tmp), 5);
    }
    CK(cudaEventRecord(sl.staged, ss));
    // ---- the usual pipeline, on the engine stream, reading reads and tags inside the stream ----
    DevBatch d{};
    d.n_loci = nl; d.n_reads = n_rec; d.n_cand = n_cand;
    d.locus_row = P<uint32_t>(sl.locus_row); d.hap = P<uint8_t>(sl.hap); d.ref_off = P<uint32_t>(sl.ref_off); d.ref_len = P<uint32_t>(sl.ref_len);
    d.alt_off = P<uint32_t>(sl.alt_off); d.alt_len = P<uint32_t>(sl.alt_len); d.cand_start = P<uint64_t>(sl.cand_start);
    d.read_nib = P<uint8_t>(sl.stream); d.read_off = P<uint64_t>(sl.read_off); d.read_len = P<uint32_t>(sl.read_len);
    d.cb_bytes = P<uint8_t>(sl.stream); d.read_cb_off = P<uint32_t>(sl.read_cb_off); d.read_cb_len = P<uint16_t>(sl.read_cb_len);
    d.read_umi = ctx->cfg.use_umi ? P<uint64_t>(sl.read_umi) : nullptr; d.cand_read = P<uint32_t>(sl.cand_rec);
    d.max_read_len = max_read; d.max_hap_len = max_hap;
    CK(cudaStreamWaitEvent(ctx->stream, sl.staged, 0));
    CK(cudaEventRecord(tr->ev[EV_C0], ctx->stream));
    rc = process_batch(ctx, d, tr);
    if (rc) return rc;
    CK(cudaEventRecord(sl.free_ev, ctx->stream));
    return VTX_OK;
}

int vtx_bam_metrics_get(vtx_ctx* ctx, vtx_bam_metrics* out)
{
    if (!ctx || !out) return VTX_E_INVALID;
    memset(out, 0, sizeof(*out));
    if (!ctx->stage_stream) return VTX_OK;
    CK(cudaSetDevice(ctx->device));
    static_assert(sizeof(vtx_bam_metrics) == sizeof(stage::LocusMetrics), "metric layouts must agree");
    CK(cudaMemcpyAsync(out, ctx->bam_metrics.p, sizeof(*out), cudaMemcpyDeviceToHost, ctx->stage_stream));
    CK(cudaStreamSynchronize(ctx->stage_stream));
    return VTX_OK;
}

uint64_t vtx_pack_cb(const uint8_t* s, uint32_t len) { return (s || len == 0) ? pack_cb(s, len) : VTX_NO_CB_KEY; }

int vtx_sync(vtx_ctx* ctx)
{
    if (!ctx) return VTX_E_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    return VTX_OK;
}

int vtx_wait_copies(vtx_ctx* ctx)
{
    if (!ctx) return VTX_E_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->copy_stream));
    return VTX_OK;
}

static int finish_scalars(vtx_ctx* ctx)
{
    CK(cudaSetDevice(ctx->device));
    uint64_t* hs = static_cast<uint64_t*>(ctx->h_scalars);
    CK(cudaMemcpyAsync(hs, ctx->d_res_n.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(hs + 1, ctx->d_metrics.p, 48, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const uint64_t violated = ctx->finished ? 0 : hs[5], band_overflow = ctx->finished ? 0 : hs[6];
    ctx->last_n = ctx->finished ? 0 : hs[0];
    ctx->last_metrics.num_not_cell_bc = ctx->finished ? 0 : hs[1];
    ctx->last_metrics.num_non_umi = ctx->finished ? 0 : hs[2];
    ctx->last_metrics.num_scored = ctx->finished ? 0 : hs[3];
    ctx->t_pairs = ctx->last_metrics.num_scored;
    ctx->finished = true;
    if (band_overflow)
        return set_err(ctx, VTX_E_UNSUPPORTED, "band model: %llu alignments had more k-mer hits than the work buffers hold (reads x windows too large); "
                                               "they were scored with the full matrix", (unsigned long long)band_overflow);
    if (violated)
        return set_err(ctx, VTX_E_INVALID, "%llu loci of a device batch exceeded the bounds given to vtx_submit_device(_ex) (longest read / widest "
                                           "haplotype window); they were skipped, the result is incomplete", (unsigned long long)violated);
    return VTX_OK;
}

int vtx_finish_device(vtx_ctx* ctx, vtx_result* out)
{
    Nvtx nvtx_range("vtx_finish_device");
    if (!ctx || !out) return VTX_E_INVALID;
    int rc = finish_scalars(ctx);
    if (rc) return rc;
    out->n = ctx->last_n;
    out->row = P<uint32_t>(ctx->r_row); out->col = P<uint32_t>(ctx->r_col); out->ref_cnt = P<uint32_t>(ctx->r_ref);
    out->alt_cnt = P<uint32_t>(ctx->r_alt); out->unk_cnt = P<uint32_t>(ctx->r_unk);
    out->val = P<double>(ctx->r_val); out->val2 = P<double>(ctx->r_val2);
    out->metrics = ctx->last_metrics;
    return VTX_OK;
}

static int ensure_host_results(vtx_ctx* ctx, size_t n);

static int fetch_to(vtx_ctx* ctx, const vtx_result* dev, vtx_result* out, void** hbuf, size_t* hcap)
{
    const size_t n = dev->n;
    const size_t esz[7] = { 4, 4, 4, 4, 4, 8, 8 };
    const bool values_only = (ctx->cfg.flags & VTX_F_VALUES_ONLY) != 0;
    bool want[7] = { true, true, !values_only, !values_only, !values_only, true, !values_only || ctx->cfg.mode == VTX_MODE_COVERAGE };
    if (n > *hcap) {
        const size_t ncap = n + n / 4 + 1024;
        for (int i = 0; i < 7; ++i) {
            if (hbuf[i]) { cudaFreeHost(hbuf[i]); hbuf[i] = nullptr; }
            if (!want[i]) continue;
            cudaError_t e = cudaHostAlloc(&hbuf[i], ncap * esz[i], cudaHostAllocDefault);
            if (e != cudaSuccess) { *hcap = 0; return set_err(ctx, VTX_E_NOMEM, "pinned result alloc failed: %s", cudaGetErrorString(e)); }
        }
        *hcap = ncap;
    }
    const void* src[7] = { dev->row, dev->col, dev->ref_cnt, dev->alt_cnt, dev->unk_cnt, dev->val, dev->val2 };
    if (n) {
        for (int i = 0; i < 7; ++i)
            if (want[i] && src[i]) CK(cudaMemcpyAsync(hbuf[i], src[i], n * esz[i], cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    out->n = n;
    out->row = static_cast<uint32_t*>(hbuf[0]); out->col = static_cast<uint32_t*>(hbuf[1]);
    out->ref_cnt = want[2] ? static_cast<uint32_t*>(hbuf[2]) : nullptr; out->alt_cnt = want[3] ? static_cast<uint32_t*>(hbuf[3]) : nullptr;
    out->unk_cnt = want[4] ? static_cast<uint32_t*>(hbuf[4]) : nullptr;
    out->val = static_cast<double*>(hbuf[5]); out->val2 = want[6] ? static_cast<double*>(hbuf[6]) : nullptr;
    out->metrics = dev->metrics;
    return VTX_OK;
}

int vtx_fetch(vtx_ctx* ctx, const vtx_result* device_result, vtx_result* out)
{
    Nvtx nvtx_range("vtx_fetch");
    if (!ctx || !device_result || !out) return VTX_E_INVALID;
    CK(cudaSetDevice(ctx->device));
    // gathered results get their own host buffers so that a local and a gathered copy can coexist
    const bool gathered = device_result->row == ctx->g_dev[0].p && ctx->g_dev[0].p != nullptr;
    return gathered ? fetch_to(ctx, device_result, out, ctx->g_host, &ctx->g_host_cap)
                    : fetch_to(ctx, device_result, out, ctx->h_res, &ctx->h_res_cap);
}

// host pinned result arrays with room for `n` triplets
static int ensure_host_results(vtx_ctx* ctx, size_t n)
{
    if (n <= ctx->h_res_cap) return VTX_OK;
    const size_t esz[7] = { 4, 4, 4, 4, 4, 8, 8 };
    const size_t ncap = n + n / 4 + 1024;
    const bool values_only = (ctx->cfg.flags & VTX_F_VALUES_ONLY) != 0;       // then the three count arrays never leave the device
    const bool want[7] = { true, true, !values_only, !values_only, !values_only, true, !values_only || ctx->cfg.mode == VTX_MODE_COVERAGE };
    for (int i = 0; i < 7; ++i) {
        if (ctx->h_res[i]) { cudaFreeHost(ctx->h_res[i]); ctx->h_res[i] = nullptr; }
        if (!want[i]) continue;
        cudaError_t e = cudaHostAlloc(&ctx->h_res[i], ncap * esz[i], cudaHostAllocDefault);
        if (e != cudaSuccess) { ctx->h_res_cap = 0; return set_err(ctx, VTX_E_NOMEM, "pinned result alloc failed: %s", cudaGetErrorString(e)); }
    }
    ctx->h_res_cap = ncap;
    return VTX_OK;
}

int vtx_finish(vtx_ctx* ctx, vtx_result* out)
{
    Nvtx nvtx_range("vtx_finish");
    if (!ctx || !out) return VTX_E_INVALID;
    CK(cudaSetDevice(ctx->device));
    // Stream the triplets out submit by submit: the kernels of later submits are usually still running when the
    // host gets here, so the device->host copy of everything but the last shard hides behind them.
    const size_t esz[7] = { 4, 4, 4, 4, 4, 8, 8 };
    DBuf* bufs[7] = { &ctx->r_row, &ctx->r_col, &ctx->r_ref, &ctx->r_alt, &ctx->r_unk, &ctx->r_val, &ctx->r_val2 };
    const bool values_only = (ctx->cfg.flags & VTX_F_VALUES_ONLY) != 0;
    const bool want[7] = { true, true, !values_only, !values_only, !values_only, true, !values_only || ctx->cfg.mode == VTX_MODE_COVERAGE };
    size_t fetched = 0;
    const bool streamed = !ctx->finished && ctx->h_cum && ctx->fetch_stream && ctx->trec_used > 0 && ctx->trec_used <= kMaxCum;
    if (streamed) {
        int rc = ensure_host_results(ctx, ctx->res_ub);
        if (rc) return rc;
        for (size_t i = 0; i < ctx->trec_used; ++i) {
            CK(cudaEventSynchronize(ctx->trecs[i].ev[EV_POST]));
            const size_t n_i = size_t(ctx->h_cum[i]);
            if (n_i > fetched && n_i <= ctx->h_res_cap) {
                for (int a = 0; a < 7; ++a)
                    if (want[a]) CK(cudaMemcpyAsync(static_cast<uint8_t*>(ctx->h_res[a]) + fetched * esz[a], static_cast<uint8_t*>(bufs[a]->p) + fetched * esz[a],
                                                    (n_i - fetched) * esz[a], cudaMemcpyDeviceToHost, ctx->fetch_stream));
                fetched = n_i;
            }
        }
    }
    vtx_result dev{};
    int rc = vtx_finish_device(ctx, &dev);
    if (rc) return rc;
    const size_t n = dev.n;
    rc = ensure_host_results(ctx, n);          // no-op when streamed (res_ub >= n)
    if (rc) return rc;
    if (n > fetched)
        for (int a = 0; a < 7; ++a)
            if (want[a]) CK(cudaMemcpyAsync(static_cast<uint8_t*>(ctx->h_res[a]) + fetched * esz[a], static_cast<uint8_t*>(bufs[a]->p) + fetched * esz[a],
                                            (n - fetched) * esz[a], cudaMemcpyDeviceToHost, ctx->fetch_stream ? ctx->fetch_stream : ctx->stream));
    CK(cudaStreamSynchronize(ctx->fetch_stream ? ctx->fetch_stream : ctx->stream));
    out->n = n;
    out->row = static_cast<uint32_t*>(ctx->h_res[0]); out->col = static_cast<uint32_t*>(ctx->h_res[1]);
    out->ref_cnt = want[2] ? static_cast<uint32_t*>(ctx->h_res[2]) : nullptr; out->alt_cnt = want[3] ? static_cast<uint32_t*>(ctx->h_res[3]) : nullptr;
    out->unk_cnt = want[4] ? static_cast<uint32_t*>(ctx->h_res[4]) : nullptr;
    out->val = static_cast<double*>(ctx->h_res[5]); out->val2 = want[6] ? static_cast<double*>(ctx->h_res[6]) : nullptr;
    out->metrics = dev.metrics;
    return VTX_OK;
}

int vtx_last_tile_counts(vtx_ctx* ctx, uint32_t* out, uint32_t n_out)
{
    if (!ctx || !out) return VTX_E_INVALID;
    if (!ctx->last_tiles_valid) return set_err(ctx, VTX_E_STATE, "no Smith-Waterman pass has run yet");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    const uint32_t nl = ctx->last_tiles_nl;
    for (uint32_t c = 0; c < n_out; ++c) {
        out[c] = 0;
        if (c < uint32_t(kNumClasses))
            CK(cudaMemcpy(out + c, P<uint32_t>(ctx->tstart) + size_t(c) * (nl + 1) + nl, 4, cudaMemcpyDeviceToHost));
    }
    return kNumClasses;
}

int vtx_last_timing(vtx_ctx* ctx, vtx_timing* t)
{
    if (!ctx || !t) return VTX_E_INVALID;
    if (!ctx->timing_valid || ctx->trec_used == 0) return set_err(ctx, VTX_E_STATE, "no finished submit to time");
    CK(cudaSetDevice(ctx->device));
    memset(t, 0, sizeof(*t));
    for (size_t i = 0; i < ctx->trec_used; ++i) {      // summed over every submit since the last finish
        TimeRec& r = ctx->trecs[i];
        CK(cudaEventSynchronize(r.ev[EV_POST]));
        float ms = 0;
        if (r.had_h2d) { CK(cudaEventElapsedTime(&ms, r.ev[EV_START], r.ev[EV_H2D])); t->h2d_ms += ms; }
        CK(cudaEventElapsedTime(&ms, r.ev[EV_C0], r.ev[EV_PREP])); t->prep_ms += ms;
        CK(cudaEventElapsedTime(&ms, r.ev[EV_PREP], r.ev[EV_SW])); t->sw_ms += ms;
        CK(cudaEventElapsedTime(&ms, r.ev[EV_SW], r.ev[EV_POST])); t->post_ms += ms;
        t->sw_launches += r.sw_launches; t->total_launches += r.launches;
    }
    t->n_pairs = ctx->t_pairs;
    return VTX_OK;
}

int vtx_score_pairs(vtx_ctx* ctx, const vtx_batch* hb, uint64_t n_pairs, const uint32_t* pair_read,
                    const uint32_t* pair_locus, int16_t* ref_score, int16_t* alt_score)
{
    Nvtx nvtx_range("vtx_score_pairs");
    if (!ctx) return VTX_E_INVALID;
    if (!hb) return set_err(ctx, VTX_E_INVALID, "batch is NULL");
    const HostView hv = view_of(hb);
    HostView hv0 = hv; hv0.n_cand = 0; hv0.cand_read = nullptr;          // the cand_* fields are ignored here
    int rc = validate_batch(ctx, hv0, false);
    if (rc) return rc;
    if (n_pairs >= 0xFFFFFFF0ull) return set_err(ctx, VTX_E_INVALID, "too many pairs");
    if (n_pairs && (!pair_read || !pair_locus || !ref_score || !alt_score)) return set_err(ctx, VTX_E_INVALID, "NULL pair arrays");
    DevBatch d{};
    rc = scan_host_batch(ctx, hv0, &d.max_read_len, &d.max_hap_len, false);
    if (rc) return rc;
    if (n_pairs == 0) return VTX_OK;
    const uint32_t nl = hb->n_loci;
    // counting sort by locus (tiles need the pairs of a locus to be contiguous)
    std::vector<uint32_t> start(size_t(nl) + 2, 0), order(n_pairs), s_read(n_pairs), s_locus(n_pairs);
    for (uint64_t i = 0; i < n_pairs; ++i) {
        if (pair_locus[i] >= nl || pair_read[i] >= hb->n_reads) return set_err(ctx, VTX_E_INVALID, "pair %llu out of range", (unsigned long long)i);
        ++start[pair_locus[i] + 1];
    }
    for (uint32_t l = 0; l < nl; ++l) start[l + 1] += start[l];
    {
        std::vector<uint32_t> cur(start.begin(), start.begin() + nl + 1);
        for (uint64_t i = 0; i < n_pairs; ++i) { const uint32_t p = cur[pair_locus[i]]++; order[p] = uint32_t(i); s_read[p] = pair_read[i]; s_locus[p] = pair_locus[i]; }
    }
    CK(cudaSetDevice(ctx->device));
    InSlot* sl = nullptr;
    rc = claim_slot(ctx, &sl);
    if (rc) return rc;
    rc = upload_common(ctx, sl, hb, d);
    if (rc) return rc;
    CK(cudaEventRecord(sl->copy_done, ctx->copy_stream));
    CK(cudaStreamWaitEvent(ctx->stream, sl->copy_done, 0));
    ENS(ctx->pair_read, n_pairs * 4 + 4); ENS(ctx->pair_locus, n_pairs * 4 + 4); ENS(ctx->pair_start, size_t(nl + 1) * 4);
    ENS(ctx->pair_scores, n_pairs * 4 + 4);
    CK(cudaMemcpyAsync(ctx->pair_read.p, s_read.data(), n_pairs * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->pair_locus.p, s_locus.data(), n_pairs * 4, cudaMemcpyHostToDevice, ctx->stream));
    vtx_k_pair_start_explicit<<<blocks_for(nl + 1, 256), 256, 0, ctx->stream>>>(nl, uint32_t(n_pairs), P<uint32_t>(ctx->pair_locus),
                                                                                P<uint32_t>(ctx->pair_start));
    uint64_t launches = 1, sw_launches = 0;
    rc = run_sw(ctx, d, uint32_t(n_pairs), nullptr, nullptr, P<uint32_t>(ctx->pair_scores), &launches, &sw_launches, nullptr);
    if (rc) return rc;
    CK(cudaEventRecord(sl->free_ev, ctx->stream));
    std::vector<uint32_t> packed(n_pairs);
    CK(cudaMemcpyAsync(packed.data(), ctx->pair_scores.p, n_pairs * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (uint64_t p = 0; p < n_pairs; ++p) {
        ref_score[order[p]] = int16_t(packed[p] & 0xFFFF);
        alt_score[order[p]] = int16_t(packed[p] >> 16);
    }
    return VTX_OK;
}

uint64_t vtx_pack_umi(const uint8_t* s, uint32_t len)
{
    if (len > 18) return VTX_NO_UMI;
    uint64_t k = 0;
    for (uint32_t i = 0; i < len; ++i) {
        uint64_t c;
        switch (s[i]) { case 'A': c = 0; break; case 'C': c = 1; break; case 'G': c = 2; break; case 'T': c = 3; break; case 'N': c = 4; break; default: return VTX_NO_UMI; }
        k = (k << 3) | c;
    }
    return (k << 5) | len;      // < 2^59: bits 59..61 stay clear for caller-interned ids
}


// -------------------------------------------------------------------------------------------------
// multi-GPU: one allgatherv of the finished triplets over NCCL (NVLink 5 / NVSwitch).  NCCL has no
// native "v" collective: ncclAllGather of the per-rank counts, then one grouped set of exact-size
// ncclBroadcast calls (7 arrays x n_ranks roots).  NCCL is dlopen'ed so that single-GPU users (and
// CPU-only build hosts) never need the library.
// -------------------------------------------------------------------------------------------------
}  // extern "C"

#include <dlfcn.h>
namespace {
typedef struct { char internal[128]; } nccl_uid;
typedef void* nccl_comm;
struct NcclApi {
    void* h = nullptr;
    int (*GetUniqueId)(nccl_uid*) = nullptr;
    int (*CommInitRank)(nccl_comm*, int, nccl_uid, int) = nullptr;
    int (*CommDestroy)(nccl_comm) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, nccl_comm, cudaStream_t) = nullptr;
    int (*Broadcast)(const void*, void*, size_t, int, int, nccl_comm, cudaStream_t) = nullptr;
    int (*Send)(const void*, size_t, int, int, nccl_comm, cudaStream_t) = nullptr;
    int (*Recv)(void*, size_t, int, int, nccl_comm, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    bool ok = false;
};
NcclApi g_nccl;
constexpr int kNcclUint8 = 1, kNcclUint64 = 5;

bool load_nccl(std::string* why)
{
    if (g_nccl.ok) return true;
    const char* names[] = { "libnccl.so.2", "libnccl.so" };
    for (const char* n : names) { g_nccl.h = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (g_nccl.h) break; }
    if (!g_nccl.h) { *why = std::string("dlopen(libnccl.so.2) failed: ") + dlerror(); return false; }
#define SYM(field, name) *(void**)(&g_nccl.field) = dlsym(g_nccl.h, name); if (!g_nccl.field) { *why = std::string("missing symbol ") + name; return false; }
    SYM(GetUniqueId, "ncclGetUniqueId") SYM(CommInitRank, "ncclCommInitRank") SYM(CommDestroy, "ncclCommDestroy")
    SYM(AllGather, "ncclAllGather") SYM(Broadcast, "ncclBroadcast") SYM(GroupStart, "ncclGroupStart")
    SYM(GroupEnd, "ncclGroupEnd") SYM(GetErrorString, "ncclGetErrorString") SYM(Send, "ncclSend") SYM(Recv, "ncclRecv")
#undef SYM
    g_nccl.ok = true;
    return true;
}
#define NK(call) do { int r_ = (call); if (r_ != 0) return set_err(ctx, VTX_E_NCCL, "%s failed: %s", #call, g_nccl.GetErrorString(r_)); } while (0)
}  // namespace

extern "C" {

void vtx_comm_destroy_internal(vtx_ctx* ctx)
{
    if (ctx->comm && g_nccl.ok) g_nccl.CommDestroy(static_cast<nccl_comm>(ctx->comm));
    ctx->comm = nullptr;
}

int vtx_comm_unique_id(uint8_t id_out[128])
{
    std::string why;
    if (!id_out) return VTX_E_INVALID;
    if (!load_nccl(&why)) { g_create_error = why; return VTX_E_NCCL; }
    nccl_uid id;
    int r = g_nccl.GetUniqueId(&id);
    if (r != 0) { g_create_error = g_nccl.GetErrorString(r); return VTX_E_NCCL; }
    memcpy(id_out, id.internal, 128);
    return VTX_OK;
}

int vtx_comm_init(vtx_ctx* ctx, const uint8_t id[128], int32_t rank, int32_t n_ranks)
{
    if (!ctx || !id || n_ranks < 1 || rank < 0 || rank >= n_ranks) return ctx ? set_err(ctx, VTX_E_INVALID, "vtx_comm_init: bad arguments") : VTX_E_INVALID;
    std::string why;
    if (!load_nccl(&why)) return set_err(ctx, VTX_E_NCCL, "%s", why.c_str());
    CK(cudaSetDevice(ctx->device));
    nccl_uid uid; memcpy(uid.internal, id, 128);
    nccl_comm comm = nullptr;
    NK(g_nccl.CommInitRank(&comm, n_ranks, uid, rank));
    ctx->comm = comm; ctx->rank = rank; ctx->n_ranks = n_ranks;
    return VTX_OK;
}

int vtx_gather_start(vtx_ctx* ctx, int32_t root)
{
    Nvtx nvtx_range("vtx_gather_start");
    if (!ctx) return VTX_E_INVALID;
    if (!ctx->finished) return set_err(ctx, VTX_E_STATE, "vtx_gather must follow vtx_finish / vtx_finish_device");
    if (ctx->gather_pending) return set_err(ctx, VTX_E_STATE, "a gather is already in flight: call vtx_gather_wait first");
    const int nrk = ctx->n_ranks;
    if (root != VTX_GATHER_ALL && (root < 0 || root >= nrk)) return set_err(ctx, VTX_E_INVALID, "gather root %d out of range", root);
    if (nrk != 1 && !ctx->comm) return set_err(ctx, VTX_E_STATE, "vtx_comm_init has not been called");
    CK(cudaSetDevice(ctx->device));
    const size_t esz[7] = { 4, 4, 4, 4, 4, 8, 8 };
    DBuf* loc[7] = { &ctx->r_row, &ctx->r_col, &ctx->r_ref, &ctx->r_alt, &ctx->r_unk, &ctx->r_val, &ctx->r_val2 };
    const bool values_only = (ctx->cfg.flags & VTX_F_VALUES_ONLY) != 0;     // then only row / col / val (/ val2) travel
    const bool want[7] = { true, true, !values_only, !values_only, !values_only, true, !values_only || ctx->cfg.mode == VTX_MODE_COVERAGE };
    vtx_result& out = ctx->g_out;
    memset(&out, 0, sizeof(out));
    const void* src[7] = { nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr };
    if (nrk == 1) {
        for (int i = 0; i < 7; ++i) if (want[i]) src[i] = loc[i]->p;
        out.n = ctx->last_n; out.metrics = ctx->last_metrics;
    } else {
        if (!ctx->comm_stream) {
            CK(cudaStreamCreateWithFlags(&ctx->comm_stream, cudaStreamNonBlocking));
            CK(cudaEventCreateWithFlags(&ctx->ev_counts, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&ctx->ev_gather, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&ctx->ev_results, cudaEventDisableTiming));
            CK(cudaHostAlloc(reinterpret_cast<void**>(&ctx->h_counts), size_t(nrk + 1) * 32, cudaHostAllocDefault));
        }
        cudaStream_t cs = ctx->comm_stream;
        nccl_comm comm = static_cast<nccl_comm>(ctx->comm);
        // the local results are complete on the engine stream (vtx_finish synchronised it); order the comm stream behind it anyway
        CK(cudaEventRecord(ctx->ev_results, ctx->stream));
        CK(cudaStreamWaitEvent(cs, ctx->ev_results, 0));
        // 1. counts: {n, not_cell_bc, non_umi, scored} of every rank.  One tiny allgather; the host needs the sizes to post
        //    exact-size receives, and waits for this one event only (tens of microseconds, nothing else is blocked).
        ENS(ctx->g_counts, size_t(nrk + 1) * 32);
        uint64_t* mine = ctx->h_counts + size_t(nrk) * 4;
        mine[0] = ctx->last_n; mine[1] = ctx->last_metrics.num_not_cell_bc; mine[2] = ctx->last_metrics.num_non_umi; mine[3] = ctx->last_metrics.num_scored;
        uint64_t* dmine = P<uint64_t>(ctx->g_counts) + size_t(nrk) * 4;
        CK(cudaMemcpyAsync(dmine, mine, 32, cudaMemcpyHostToDevice, cs));
        NK(g_nccl.AllGather(dmine, ctx->g_counts.p, 4, kNcclUint64, comm, cs));
        CK(cudaMemcpyAsync(ctx->h_counts, ctx->g_counts.p, size_t(nrk) * 32, cudaMemcpyDeviceToHost, cs));
        CK(cudaEventRecord(ctx->ev_counts, cs));
        CK(cudaEventSynchronize(ctx->ev_counts));
        const uint64_t* counts = ctx->h_counts;
        size_t total = 0;
        std::vector<size_t> offs(nrk);
        vtx_metrics met{};
        for (int r = 0; r < nrk; ++r) {
            offs[r] = total; total += counts[size_t(r) * 4];
            met.num_not_cell_bc += counts[size_t(r) * 4 + 1]; met.num_non_umi += counts[size_t(r) * 4 + 2]; met.num_scored += counts[size_t(r) * 4 + 3];
        }
        out.n = total; out.metrics = met;
        const bool receiver = root == VTX_GATHER_ALL || root == ctx->rank;
        if (receiver) for (int i = 0; i < 7; ++i) if (want[i]) ENS(ctx->g_dev[i], (total ? total : 1) * esz[i]);
        // 2. the triplets, exact sizes, one NCCL group.  Rooted: ncclSend / ncclRecv, only the writer's GPU receives;
        //    all: one broadcast per (array, rank) = allgatherv.
        NK(g_nccl.GroupStart());
        for (int i = 0; i < 7; ++i) {
            if (!want[i]) continue;
            if (root == VTX_GATHER_ALL) {
                for (int r = 0; r < nrk; ++r) {
                    const size_t n = counts[size_t(r) * 4];
                    if (n) NK(g_nccl.Broadcast(loc[i]->p, static_cast<uint8_t*>(ctx->g_dev[i].p) + offs[r] * esz[i], n * esz[i], kNcclUint8, r, comm, cs));
                }
            } else if (ctx->rank == root) {
                for (int r = 0; r < nrk; ++r) {
                    const size_t n = counts[size_t(r) * 4];
                    if (!n) continue;
                    uint8_t* dst = static_cast<uint8_t*>(ctx->g_dev[i].p) + offs[r] * esz[i];
                    if (r == root) CK(cudaMemcpyAsync(dst, loc[i]->p, n * esz[i], cudaMemcpyDeviceToDevice, cs));
                    else NK(g_nccl.Recv(dst, n * esz[i], kNcclUint8, r, comm, cs));
                }
            } else if (ctx->last_n) {
                NK(g_nccl.Send(loc[i]->p, size_t(ctx->last_n) * esz[i], kNcclUint8, root, comm, cs));
            }
        }
        NK(g_nccl.GroupEnd());
        CK(cudaEventRecord(ctx->ev_gather, cs));
        ctx->gather_guard = true;
        if (receiver) for (int i = 0; i < 7; ++i) if (want[i]) src[i] = ctx->g_dev[i].p;
    }
    out.row = static_cast<const uint32_t*>(src[0]); out.col = static_cast<const uint32_t*>(src[1]);
    out.ref_cnt = static_cast<const uint32_t*>(src[2]); out.alt_cnt = static_cast<const uint32_t*>(src[3]);
    out.unk_cnt = static_cast<const uint32_t*>(src[4]);
    out.val = static_cast<const double*>(src[5]); out.val2 = static_cast<const double*>(src[6]);
    ctx->gather_pending = true;
    return VTX_OK;
}

int vtx_gather_wait(vtx_ctx* ctx, vtx_result* out)
{
    Nvtx nvtx_range("vtx_gather_wait");
    if (!ctx || !out) return VTX_E_INVALID;
    if (!ctx->gather_pending) return set_err(ctx, VTX_E_STATE, "no gather in flight");
    CK(cudaSetDevice(ctx->device));
    if (ctx->n_ranks > 1) CK(cudaEventSynchronize(ctx->ev_gather));
    ctx->gather_pending = false;
    *out = ctx->g_out;
    return VTX_OK;
}

int vtx_gather(vtx_ctx* ctx, vtx_result* out)
{
    if (!ctx || !out) return VTX_E_INVALID;
    const int rc = vtx_gather_start(ctx, VTX_GATHER_ALL);
    return rc ? rc : vtx_gather_wait(ctx, out);
}

}  // extern "C"
