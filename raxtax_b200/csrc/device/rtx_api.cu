// rtx_api.cu -- C ABI (include/raxtax_b200.h) of the sm_100a query-classification library.
// Host-side orchestration only: validation, HBM layout, kernel launches, result ordering.  No CPU compute path.

#include <dlfcn.h>
#include <nccl.h>  // types and prototypes only: libnccl is bound at run time (see the NCCL section below)

#include <algorithm>
#include <cmath>
#include <cstring>
#include <mutex>

#include "kernels.cuh"

using namespace rtx;

// ---------------------------------------------------------------------------------------------------------
struct EventPair {
    cudaEvent_t a, b;
    int kernel;
};

// Everything rtx_batch_upload sets up for ONE batch.  A context holds two of these ("slots", rtx_batch_slot): the active one is
// the BatchState base of rtx_ctx, the other is parked; switching swaps them.  While the kernels of one slot run on `stream`, the
// other slot can be uploaded (H2D on `stream_cp`) and its predecessor's results downloaded (D2H on `stream_cp` behind the slot's
// ev_done), so the device never waits for the host between batches.  Every slot has its own compute stream and its own per-sub-batch
// scratch (counts, prefixes, tables): the hit counting of the batch in one slot starts as soon as the hit counting of the batch in the
// other slot is through (ev_k2) and so runs under that batch's probability / prefix / walk kernels, whose tails (persistent CTAs, one
// CTA per query) leave most of the GPU idle -- what makes small batches cost no more than their share of a large one.
struct BatchState {
    cudaStream_t stream = nullptr;
    // sub-batch pipeline: hit counting of sub-batch i+1 (stream) overlaps probabilities / prefix sums / tree walk of sub-batch i
    // (stream2); the per-sub-batch buffers exist twice, events order the two streams
    cudaStream_t stream2 = nullptr;
    cudaEvent_t ev_hit[2] = {nullptr, nullptr}, ev_post[2] = {nullptr, nullptr};
    cudaEvent_t ev_k2 = nullptr;  // the last hit-count launch of the slot's current run has finished
    bool k2_recorded = false;
    // per-sub-batch scratch
    DevBuf d_counts, d_counts1, d_prob_big, d_cbuf, d_preb, d_ptab, d_segoff, d_preb1, d_ptab1, d_segoff1;
    bool has_batch = false;
    bool ran = false;
    BatchView bv{};
    u32 max_len = 0;
    u64 total_codes = 0, total_exact = 0;
    DevBuf d_seq_off, d_codes, d_exact_off, d_exact_ids, d_K, d_kmers, d_rows, d_nrows, d_hist;
    u32 sub_batch = 0;
    bool two_slots = false;  // this batch runs with the two-stream sub-batch pipeline
    // results
    ResultPool pool{};
    u32 pool_levels = 0;  // max_levels the pool arrays were sized for
    DevBuf d_pool_first, d_pool_nlev, d_pool_conf, d_pool_local, d_pool_used, d_res_off, d_res_cnt, d_global, d_status, d_hits;
    // prob scratch layout of this batch (the buffers themselves are shared between the slots, see bind_scratch)
    ProbScratch sc{}, sc1{};
    int prob_slots = 0;
    size_t prob_smem = 0, prob_big_bytes = 0, prefix_smem = 0;
    size_t need_counts = 0, need_cbuf = 0, need_preb = 0, need_ptab = 0, need_segoff = 0, need_prob_big = 0;
    // results in query order (result_scan_kernel / result_gather_kernel)
    DevBuf d_ord_begin, d_ord_first, d_ord_nlev, d_ord_conf, d_ord_local;
    int shard_phase = 0;
    u64 runs_since_download = 0;
    cudaEvent_t ev_up = nullptr, ev_done = nullptr;  // inputs are on the device / all kernels of the last run have finished
    bool up_pending = false;                          // ev_up was recorded and no run has waited for it yet
    // reference-sharded mode over NCCL
    bool sub_batch_agreed = false;  // the ranks settled on one sub-batch size for this batch
    bool merged = false;            // rtx_shard_gather ran: d_ord_* hold the merged lines (root) / nothing (other ranks)
    u64 merged_lines = 0;
};

struct rtx_ctx : BatchState {
    BatchState parked;  // the slot that is not active
    int cur_slot = 0;
    int device = 0;
    int n_sms = 148;
    cudaStream_t stream_cp = nullptr;  // host <-> device copies of the batch slots
    bool pipeline_opt = false;  // RTX_OPT_PIPELINE (off: measured 9.95-10.2 ms pipelined against 9.89 ms serial on C2, profiles/r01x_pipeline.txt)
    cudaStream_t cur_stream = nullptr;  // what the launch helpers use: stream / slot of the sub-batch being issued
    u16* cur_counts = nullptr;
    bool segmax_valid = false;  // the last hit-count launch left per-segment maxima in cur_sc's aux area
    ProbScratch* cur_sc = nullptr;
    std::string err;
    std::string hit_kernel;  // the hit-count kernel instantiation of the last launch (rtx_hitcount_kernel_name)
    // options
    int variant = RTX_HITCOUNT_BITROWS;
    int64_t sub_batch_opt = 0;
    bool keep_csr = false;
    bool profile = false;
    int hit_max_tiles = 0;
    int walk_variant = 0;  // RTX_OPT_WALK_VARIANT: 0 level-synchronous (+ depth-first retry), 1 depth-first only
    int walk_log_cap = 0;  // RTX_OPT_WALK_LOG_CAP
    int hit_group = 0;   // RTX_OPT_HITCOUNT_GROUP
    // index
    bool has_index = false;
    IndexView ix{};
    u32 n_rows = 0;
    u64 index_bytes = 0;
    u64 mem_free_after_index = 8ull << 30;
    DevBuf d_bitrows, d_rowmap, d_present, d_csr_off, d_csr_ids, d_node_lo, d_node_hi, d_node_type, d_child_first, d_child_count,
        d_ref_levels, d_lnfact, d_recs;
    DevBuf d_seq_codes, d_idx_off;  // reference sequences / their offsets while the index is built from them
    size_t walk_smem = 0, bfs_smem = 0;
    // reference-sharded mode
    ShardView sv{};
    DevBuf d_strad_of_node, d_strad_nodes, d_strad_parent, d_send, d_recv, d_sk, d_sany, d_sbest;
    // ... over NCCL (rtx_comm_init): exchange buffers per scratch slot, gather buffers of the root
    void* comm = nullptr;  // ncclComm_t
    int comm_rank = 0, comm_size = 0;
    DevBuf d_agree, d_send_s[2], d_recv_s[2], d_sk_s[2], d_sany_s[2], d_sbest_s[2], d_all_begin, d_rank_off, d_g_first, d_g_nlev, d_g_conf, d_g_local;
    // host staging: one pinned arena (device -> arena by DMA, arena -> caller memory by memcpy unless the caller's memory is pinned itself)
    unsigned char* h_arena = nullptr;
    size_t h_arena_cap = 0, h_arena_used = 0;
    struct PendingCopy {
        void* dst;
        size_t arena_off, bytes;
    };
    std::vector<PendingCopy> h_pending;
    // taps wired by rtx_classify_batch for sub-batched runs
    u16* tap_counts_host = nullptr;
    double* tap_probs_host = nullptr;
    u64 tap_prob_stride = 0;
    // profile
    rtx_profile prof{};
    std::vector<EventPair> events;
};

static std::string g_create_err;
static std::mutex g_create_mtx;

static int set_err(rtx_ctx* c, int code, const std::string& msg) {
    if (c) c->err = msg;
    else {
        std::lock_guard<std::mutex> g(g_create_mtx);
        g_create_err = msg;
    }
    return code;
}

#define CU(call)                                                                                              \
    do {                                                                                                      \
        cudaError_t e__ = (call);                                                                             \
        if (e__ != cudaSuccess)                                                                               \
            return set_err(ctx, RTX_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));           \
    } while (0)

#define REQUIRE(cond, msg)                                                \
    do {                                                                  \
        if (!(cond)) return set_err(ctx, RTX_ERR_INVALID, std::string(msg)); \
    } while (0)

static inline u32 round_up(u32 x, u32 a) { return (x + a - 1) / a * a; }

// ---- launch bookkeeping -------------------------------------------------------------------------------
struct LaunchTimer {
    rtx_ctx* c;
    int k;
    EventPair ep{};
    bool on;
    LaunchTimer(rtx_ctx* ctx, int kernel) : c(ctx), k(kernel), on(ctx->profile) {
        c->prof.kernel[k].launches += 1;
        if (on) {
            cudaEventCreate(&ep.a);
            cudaEventCreate(&ep.b);
            ep.kernel = k;
            cudaEventRecord(ep.a, c->cur_stream ? c->cur_stream : c->stream);
        }
    }
    ~LaunchTimer() {
        if (on) {
            cudaEventRecord(ep.b, c->cur_stream ? c->cur_stream : c->stream);
            c->events.push_back(ep);
        }
    }
};

static void drain_events(rtx_ctx* c) {
    for (auto& ep : c->events) {
        cudaEventSynchronize(ep.b);
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ep.a, ep.b) == cudaSuccess) c->prof.kernel[ep.kernel].total_ms += ms;
        cudaEventDestroy(ep.a);
        cudaEventDestroy(ep.b);
    }
    c->events.clear();
}

// ---- pinned staging ------------------------------------------------------------------------------------
static cudaError_t arena_reserve(rtx_ctx* c, size_t bytes) {  // only between downloads: nothing may be in flight into the arena
    c->h_arena_used = 0;
    c->h_pending.clear();
    if (bytes <= c->h_arena_cap) return cudaSuccess;
    if (c->h_arena) cudaFreeHost(c->h_arena);
    c->h_arena = nullptr;
    c->h_arena_cap = 0;
    const size_t cap = bytes + bytes / 4 + 4096;
    cudaError_t e = cudaHostAlloc((void**)&c->h_arena, cap, cudaHostAllocDefault);
    if (e == cudaSuccess) c->h_arena_cap = cap;
    return e;
}
static bool host_ptr_pinned(const void* p) {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}
// device -> caller memory: straight DMA when the caller's buffer is pinned, else DMA into the arena and a memcpy after the sync
static cudaError_t d2h(rtx_ctx* c, void* dst, const void* src, size_t bytes, bool dst_pinned) {
    if (!bytes) return cudaSuccess;
    if (dst_pinned) return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream_cp);
    const size_t off = (c->h_arena_used + 63) & ~(size_t)63;
    if (off + bytes > c->h_arena_cap) return cudaErrorMemoryAllocation;
    c->h_arena_used = off + bytes;
    c->h_pending.push_back({dst, off, bytes});
    return cudaMemcpyAsync(c->h_arena + off, src, bytes, cudaMemcpyDeviceToHost, c->stream_cp);
}
static void* arena_take(rtx_ctx* c, size_t bytes) {  // arena space the library reads itself
    const size_t off = (c->h_arena_used + 63) & ~(size_t)63;
    if (off + bytes > c->h_arena_cap) return nullptr;
    c->h_arena_used = off + bytes;
    return c->h_arena + off;
}
static cudaError_t d2h_finish(rtx_ctx* c) {
    cudaError_t e = cudaStreamSynchronize(c->stream_cp);
    if (e != cudaSuccess) return e;
    for (auto& pc : c->h_pending) memcpy(pc.dst, c->h_arena + pc.arena_off, pc.bytes);
    c->h_pending.clear();
    return cudaSuccess;
}

// ---------------------------------------------------------------------------------------------------------
#define RTX_API extern "C" __attribute__((visibility("default")))

RTX_API int rtx_abi_version(void) { return RTX_ABI_VERSION; }

RTX_API const char* rtx_last_error(const rtx_ctx* ctx) {
    if (ctx) return ctx->err.c_str();
    std::lock_guard<std::mutex> g(g_create_mtx);
    return g_create_err.c_str();
}

RTX_API int rtx_ctx_create(int device_ordinal, rtx_ctx** out) {
    rtx_ctx* ctx = nullptr;  // for the macros: errors land in the global slot
    if (!out) return set_err(nullptr, RTX_ERR_INVALID, "rtx_ctx_create: out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return set_err(nullptr, RTX_ERR_NO_DEVICE,
                       std::string("no CUDA device available (") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count 0") +
                           "); raxtax_b200 has no CPU fallback");
    if (device_ordinal < 0 || device_ordinal >= n) return set_err(nullptr, RTX_ERR_INVALID, "device ordinal out of range");
    CU(cudaSetDevice(device_ordinal));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device_ordinal));
    if (prop.major < 10)
        return set_err(nullptr, RTX_ERR_NO_DEVICE, std::string("device ") + prop.name + " is not sm_100-class; this library is built for sm_100a only");
    rtx_ctx* c = new rtx_ctx();
    c->device = device_ordinal;
    c->n_sms = prop.multiProcessorCount;
    e = cudaStreamCreateWithFlags(&c->stream_cp, cudaStreamNonBlocking);
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
        BatchState& b = i ? c->parked : static_cast<BatchState&>(*c);
        e = cudaStreamCreateWithFlags(&b.stream, cudaStreamNonBlocking);
        // the second stream carries the short kernels behind hit counting: its CTAs go first whenever an SM frees up
        if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&b.stream2, cudaStreamNonBlocking, prio_hi);
        for (int k = 0; k < 2 && e == cudaSuccess; ++k) {
            e = cudaEventCreateWithFlags(&b.ev_hit[k], cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b.ev_post[k], cudaEventDisableTiming);
        }
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b.ev_up, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b.ev_done, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b.ev_k2, cudaEventDisableTiming);
    }
    if (e != cudaSuccess) {
        std::string m = std::string("stream / event creation: ") + cudaGetErrorString(e);
        rtx_ctx_destroy(c);
        return set_err(nullptr, RTX_ERR_CUDA, m);
    }
    c->cur_stream = c->stream;
    // ln n! table: exact factorials up to 170, lgamma beyond (the reference's statrs::ln_factorial does the same)
    const u32 len = 98304 + 8;  // K + t <= 65535 + 32767
    std::vector<double> lf(len);
    double f = 1.0;
    lf[0] = 0.0;
    for (u32 i = 1; i < len; ++i) {
        if (i <= 170) {
            f *= (double)i;
            lf[i] = std::log(f);
        } else lf[i] = std::lgamma((double)i + 1.0);
    }
    ctx = c;
    e = c->d_lnfact.ensure(len * sizeof(double));
    if (e == cudaSuccess) e = cudaMemcpy(c->d_lnfact.p, lf.data(), len * sizeof(double), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        std::string m = std::string("lnfact upload: ") + cudaGetErrorString(e);
        rtx_ctx_destroy(c);
        return set_err(nullptr, RTX_ERR_CUDA, m);
    }
    c->ix.lnfact = c->d_lnfact.as<double>();
    c->ix.lnfact_len = len;
    *out = c;
    return RTX_OK;
}

RTX_API void rtx_ctx_destroy(rtx_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    for (int i = 0; i < 2; ++i) {
        BatchState& s = i ? c->parked : static_cast<BatchState&>(*c);
        if (s.stream) cudaStreamSynchronize(s.stream);
        if (s.stream2) cudaStreamSynchronize(s.stream2);
    }
    drain_events(c);
    if (c->stream_cp) cudaStreamSynchronize(c->stream_cp);
    rtx_comm_destroy(c);
    for (int i = 0; i < 2; ++i) {
        DevBuf* xb[] = {&c->d_send_s[i], &c->d_recv_s[i], &c->d_sk_s[i], &c->d_sany_s[i], &c->d_sbest_s[i]};
        for (DevBuf* b : xb) b->release();
    }
    DevBuf* gb[] = {&c->d_agree, &c->d_all_begin, &c->d_rank_off, &c->d_g_first, &c->d_g_nlev, &c->d_g_conf, &c->d_g_local};
    for (DevBuf* b : gb) b->release();
    DevBuf* bufs[] = {&c->d_bitrows, &c->d_rowmap, &c->d_present, &c->d_csr_off, &c->d_csr_ids, &c->d_node_lo, &c->d_node_hi,
                      &c->d_node_type, &c->d_child_first, &c->d_child_count, &c->d_ref_levels, &c->d_lnfact, &c->d_seq_codes, &c->d_idx_off, &c->d_recs, &c->d_strad_of_node,
                      &c->d_strad_nodes, &c->d_strad_parent, &c->d_send, &c->d_recv, &c->d_sk, &c->d_sany, &c->d_sbest};
    for (DevBuf* b : bufs) b->release();
    for (int i = 0; i < 2; ++i) {
        BatchState& s = i ? c->parked : static_cast<BatchState&>(*c);
        DevBuf* sb[] = {&s.d_seq_off, &s.d_codes, &s.d_exact_off, &s.d_exact_ids, &s.d_K, &s.d_kmers, &s.d_rows, &s.d_nrows, &s.d_hist,
                        &s.d_pool_first, &s.d_pool_nlev, &s.d_pool_conf, &s.d_pool_local, &s.d_pool_used, &s.d_res_off, &s.d_res_cnt,
                        &s.d_global, &s.d_status, &s.d_hits, &s.d_ord_begin, &s.d_ord_first, &s.d_ord_nlev, &s.d_ord_conf, &s.d_ord_local,
                        &s.d_counts, &s.d_counts1, &s.d_prob_big, &s.d_cbuf, &s.d_preb, &s.d_ptab, &s.d_segoff, &s.d_preb1, &s.d_ptab1, &s.d_segoff1};
        for (DevBuf* b : sb) b->release();
        if (s.ev_up) cudaEventDestroy(s.ev_up);
        if (s.ev_done) cudaEventDestroy(s.ev_done);
        if (s.ev_k2) cudaEventDestroy(s.ev_k2);
        for (int k = 0; k < 2; ++k) {
            if (s.ev_hit[k]) cudaEventDestroy(s.ev_hit[k]);
            if (s.ev_post[k]) cudaEventDestroy(s.ev_post[k]);
        }
        if (s.stream2) cudaStreamDestroy(s.stream2);
        if (s.stream) cudaStreamDestroy(s.stream);
    }
    if (c->h_arena) cudaFreeHost(c->h_arena);
    if (c->stream_cp) cudaStreamDestroy(c->stream_cp);
    delete c;
}

RTX_API int rtx_ctx_set_option(rtx_ctx* ctx, int option, int64_t value) {
    if (!ctx) return RTX_ERR_INVALID;
    switch (option) {
        case RTX_OPT_HITCOUNT_VARIANT:
            REQUIRE(value == RTX_HITCOUNT_BITROWS || value == RTX_HITCOUNT_CSR, "unknown hit-count variant");
            ctx->variant = (int)value;
            return RTX_OK;
        case RTX_OPT_SUB_BATCH:
            REQUIRE(value >= 0 && value <= 65535, "sub-batch must be in [0, 65535]");
            ctx->sub_batch_opt = value;
            return RTX_OK;
        case RTX_OPT_KEEP_CSR:
            ctx->keep_csr = value != 0;
            return RTX_OK;
        case RTX_OPT_PROFILE:
            ctx->profile = value != 0;
            return RTX_OK;
        case RTX_OPT_HITCOUNT_MAX_TILES:
            REQUIRE(value >= 0 && value <= 4096, "bad max tiles per CTA");
            ctx->hit_max_tiles = (int)value;
            return RTX_OK;
        case RTX_OPT_PIPELINE:
            ctx->pipeline_opt = value != 0;
            return RTX_OK;
        case RTX_OPT_WALK_VARIANT:
            REQUIRE(value >= 0 && value <= 4 && value != 2, "unknown walk variant");  // 3: without the large-frontier paths, 4: with them forced
            ctx->walk_variant = (int)value;
            return RTX_OK;
        case RTX_OPT_WALK_LOG_CAP:
            REQUIRE(value >= 0 && value <= (int64_t)kBfsEntries, "bad walk log cap");
            ctx->walk_log_cap = (int)value;
            return RTX_OK;
        case RTX_OPT_HITCOUNT_GROUP:
            REQUIRE(value >= 0 && value <= kHitGroupMaxThreads / 32, "bad query group size");
            ctx->hit_group = (int)value;
            return RTX_OK;
        default:
            return set_err(ctx, RTX_ERR_INVALID, "unknown option");
    }
}

RTX_API void* rtx_ctx_stream(rtx_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
RTX_API int rtx_ctx_device(const rtx_ctx* ctx) { return ctx ? ctx->device : -1; }

RTX_API int rtx_ctx_synchronize(rtx_ctx* ctx) {
    if (!ctx) return RTX_ERR_INVALID;
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream2));
    CU(cudaStreamSynchronize(ctx->parked.stream));
    CU(cudaStreamSynchronize(ctx->parked.stream2));
    CU(cudaStreamSynchronize(ctx->stream_cp));
    return RTX_OK;
}

RTX_API int rtx_batch_slot(rtx_ctx* ctx, int slot) {
    if (!ctx) return RTX_ERR_INVALID;
    REQUIRE(slot == 0 || slot == 1, "rtx_batch_slot: a context has the batch slots 0 and 1");
    if (slot != ctx->cur_slot) {
        std::swap(static_cast<BatchState&>(*ctx), ctx->parked);
        ctx->cur_slot = slot;
    }
    return RTX_OK;
}

RTX_API int rtx_host_alloc(size_t bytes, void** out) {
    if (!out) return RTX_ERR_INVALID;
    *out = nullptr;
    cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault);
    if (e != cudaSuccess) return set_err(nullptr, RTX_ERR_CUDA, std::string("cudaHostAlloc: ") + cudaGetErrorString(e));
    return RTX_OK;
}
RTX_API int rtx_host_free(void* p) {
    if (!p) return RTX_OK;
    return cudaFreeHost(p) == cudaSuccess ? RTX_OK : RTX_ERR_CUDA;
}

RTX_API uint64_t rtx_index_n_refs(const rtx_ctx* c) { return c && c->has_index ? c->ix.n_refs : 0; }
RTX_API uint64_t rtx_index_shard_refs(const rtx_ctx* c) { return c && c->has_index ? c->ix.shard_refs : 0; }
RTX_API uint32_t rtx_index_max_levels(const rtx_ctx* c) { return c && c->has_index ? c->ix.max_levels : 0; }
RTX_API uint64_t rtx_index_device_bytes(const rtx_ctx* c) { return c && c->has_index ? c->index_bytes : 0; }
RTX_API uint32_t rtx_batch_sub_batch(const rtx_ctx* c) { return c && c->has_batch ? c->sub_batch : 0; }
RTX_API uint64_t rtx_index_bitrow_bytes(const rtx_ctx* c) { return c && c->has_index ? (uint64_t)c->n_rows * c->ix.row_words * 4 : 0; }
RTX_API const char* rtx_hitcount_kernel_name(const rtx_ctx* c) { return c ? c->hit_kernel.c_str() : ""; }

// ---------------------------------------------------------------------------------------------------------
// index upload
// ---------------------------------------------------------------------------------------------------------
template <typename T>
static cudaError_t upload_vec(DevBuf& buf, const T* src, size_t n, u64* acc) {
    cudaError_t e = buf.ensure(std::max<size_t>(n, 1) * sizeof(T));
    if (e != cudaSuccess) return e;
    if (n) e = cudaMemcpy(buf.p, src, n * sizeof(T), cudaMemcpyHostToDevice);
    if (acc) *acc += n * sizeof(T);
    return e;
}

RTX_API int rtx_index_upload(rtx_ctx* ctx, const rtx_index_desc* d) {
    if (!ctx) return RTX_ERR_INVALID;
    REQUIRE(d != nullptr, "rtx_index_upload: desc is NULL");
    REQUIRE(d->n_refs >= 1 && d->n_refs <= 0xFFFFFFFFull, "n_refs must be in [1, 2^32) (tree.rs:24-31)");
    REQUIRE(d->n_nodes >= 1 && d->node_lo && d->node_hi && d->node_type && d->child_first && d->child_count && d->ref_levels,
            "rtx_index_upload: NULL array");
    const bool from_seq = d->csr_offsets == nullptr;  // build the index on the device from the sorted reference sequences
    REQUIRE(!from_seq || (d->ref_seq_offsets && (d->ref_seq_codes || d->ref_seq_offsets[d->n_refs] == d->ref_seq_offsets[0])),
            "rtx_index_upload: neither a CSR (csr_offsets) nor reference sequences (ref_seq_offsets / ref_seq_codes) given");
    REQUIRE(!(from_seq && ctx->keep_csr), "RTX_OPT_KEEP_CSR (CSR hit-count variant) needs an index described by its CSR");
    const u64 N = d->n_refs;
    u64 s0 = d->ref_shard_begin, s1 = d->ref_shard_end ? d->ref_shard_end : N;
    const u32 n_shards = d->n_shards > 1 ? d->n_shards : 1;
    if (n_shards > 1) {
        REQUIRE(d->shard_cuts != nullptr && d->shard_rank < n_shards, "shard_cuts / shard_rank invalid");
        REQUIRE(d->shard_cuts[0] == 0 && d->shard_cuts[n_shards] == N, "shard_cuts must span [0, n_refs]");
        for (u32 r = 0; r < n_shards; ++r) REQUIRE(d->shard_cuts[r] < d->shard_cuts[r + 1], "shard_cuts must be strictly increasing");
        s0 = d->shard_cuts[d->shard_rank];
        s1 = d->shard_cuts[d->shard_rank + 1];
    }
    REQUIRE(s0 < s1 && s1 <= N, "bad reference shard range");
    const u64 nnz = from_seq ? 0 : d->csr_offsets[65536];
    if (!from_seq) {
        REQUIRE(d->csr_offsets[0] == 0, "csr_offsets[0] must be 0");
        for (u32 k = 0; k < 65536; ++k) REQUIRE(d->csr_offsets[k] <= d->csr_offsets[k + 1], "csr_offsets must be non-decreasing");
        REQUIRE(nnz == 0 || d->csr_ids, "csr_ids is NULL");
    } else {
        for (u64 r = s0; r < s1; ++r) REQUIRE(d->ref_seq_offsets[r] <= d->ref_seq_offsets[r + 1], "ref_seq_offsets must be non-decreasing");
    }
    REQUIRE(d->node_lo[0] == 0 && d->node_hi[0] == N, "node 0 must be the root with range [0, n_refs)");
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaStreamSynchronize(ctx->parked.stream));
    CU(cudaStreamSynchronize(ctx->stream2));
    CU(cudaStreamSynchronize(ctx->parked.stream2));
    CU(cudaStreamSynchronize(ctx->stream_cp));
    ctx->has_index = false;
    ctx->has_batch = false;
    ctx->parked.has_batch = false;

    // ---- tree checks, depth --------------------------------------------------------------------------
    const u32 nn = d->n_nodes;
    std::vector<u32> depth(nn, 0);
    u32 max_depth = 0;
    u64 child_total = 0;
    for (u32 i = 0; i < nn; ++i) {
        REQUIRE(d->node_lo[i] < d->node_hi[i] && d->node_hi[i] <= N, "node range out of bounds");
        REQUIRE(d->child_count[i] < (1u << 30), "too many children");
        REQUIRE(d->node_type[i] <= 2, "node_type must be 0 (Inner), 1 (Taxon) or 2 (Sequence with children)");
        const u32 cf = d->child_first[i], cc = d->child_count[i];
        child_total += cc;
        if (cc) {
            REQUIRE(cf > i && (u64)cf + cc <= nn, "children must follow their parent and stay in range");
            for (u32 c = cf; c < cf + cc; ++c) {
                depth[c] = depth[i] + 1;
                max_depth = std::max(max_depth, depth[c]);
                REQUIRE(d->node_lo[c] >= d->node_lo[i] && d->node_hi[c] <= d->node_hi[i], "child range outside its parent");
            }
        } else {
            REQUIRE(d->node_type[i] != 0, "an Inner node must have children (lineage.rs:162 unwrap)");
        }
    }
    REQUIRE(child_total == nn - 1, "every node except the root must be the child of exactly one node");
    u32 max_levels = std::max(1u, max_depth);
    for (u64 r = 0; r < N; ++r) max_levels = std::max<u32>(max_levels, d->ref_levels[r]);
    if (max_levels > RTX_MAX_LEVELS) return set_err(ctx, RTX_ERR_UNSUPPORTED, "lineage deeper than RTX_MAX_LEVELS");

    IndexView& ix = ctx->ix;
    const u64 Ns = s1 - s0;
    const u32 row_words = round_up((u32)((Ns + 31) / 32), kRowAlignWords);
    u64 bytes = 0;

    // ---- row map: k-mers with at least one posting inside the shard ------------------------------------
    std::vector<u32> rowmap(65536, 0), present(2048, 0);
    u32 n_rows = 1;
    // upload chunks of the sequence path: whole references, at most ~256 MB of codes each
    std::vector<u64> seq_chunks;  // reference ids where a chunk starts, + s1
    if (from_seq) {
        const u64 cap = 256ull << 20;
        seq_chunks.push_back(s0);
        u64 begin = s0;
        for (u64 r = s0; r < s1; ++r) {
            if (d->ref_seq_offsets[r + 1] - d->ref_seq_offsets[begin] > cap && r > begin) {
                seq_chunks.push_back(r);
                begin = r;
            }
        }
        seq_chunks.push_back(s1);
        u64 max_codes = 1, max_refs = 1;
        for (size_t c = 0; c + 1 < seq_chunks.size(); ++c) {
            max_codes = std::max(max_codes, d->ref_seq_offsets[seq_chunks[c + 1]] - d->ref_seq_offsets[seq_chunks[c]]);
            max_refs = std::max(max_refs, seq_chunks[c + 1] - seq_chunks[c]);
        }
        CU(ctx->d_seq_codes.ensure(max_codes + 16));
        CU(ctx->d_idx_off.ensure((max_refs + 1) * 8));
        CU(ctx->d_present.ensure(2048 * 4));
        CU(cudaMemsetAsync(ctx->d_present.p, 0, 2048 * 4, ctx->stream));
    }
    // one chunk of reference sequences -> device (offsets rebased to the chunk)
    std::vector<u64> reb;
    auto seq_chunk_to_device = [&](size_t c) -> cudaError_t {
        const u64 r0 = seq_chunks[c], r1 = seq_chunks[c + 1];
        const u64 o0 = d->ref_seq_offsets[r0], bytes_c = d->ref_seq_offsets[r1] - o0;
        reb.resize(r1 - r0 + 1);
        for (u64 r = r0; r <= r1; ++r) reb[r - r0] = d->ref_seq_offsets[r] - o0;
        cudaError_t e = cudaMemcpyAsync(ctx->d_idx_off.p, reb.data(), reb.size() * 8, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess && bytes_c) e = cudaMemcpyAsync(ctx->d_seq_codes.p, d->ref_seq_codes + o0, bytes_c, cudaMemcpyHostToDevice, ctx->stream);
        return e;
    };
    if (from_seq) {
        for (size_t c = 0; c + 1 < seq_chunks.size(); ++c) {
            CU(seq_chunk_to_device(c));
            {
                LaunchTimer lt(ctx, RTX_K_INDEX);
                kmer_presence_kernel<<<ctx->n_sms * 4, 256, 0, ctx->stream>>>(ctx->d_idx_off.as<u64>(), ctx->d_seq_codes.as<u8>(),
                                                                            (u32)(seq_chunks[c + 1] - seq_chunks[c]), ctx->d_present.as<u32>());
            }
            CU(cudaGetLastError());
            CU(cudaStreamSynchronize(ctx->stream));  // reb / the pageable source are reused by the next chunk
        }
        CU(cudaMemcpy(present.data(), ctx->d_present.p, 2048 * 4, cudaMemcpyDeviceToHost));
        for (u32 k = 0; k < 65536; ++k)
            if (present[k >> 5] >> (k & 31) & 1u) rowmap[k] = n_rows++;
        bytes += 2048 * 4;
    } else {
        for (u32 k = 0; k < 65536; ++k) {
            const u64 o0 = d->csr_offsets[k], o1 = d->csr_offsets[k + 1];
            if (o0 == o1) continue;
            bool in = true;
            if (s0 != 0 || s1 != N) {
                const u32* it = std::lower_bound(d->csr_ids + o0, d->csr_ids + o1, (u32)s0);
                in = (it != d->csr_ids + o1) && (*it < s1);
            }
            if (in) {
                rowmap[k] = n_rows++;
                present[k >> 5] |= 1u << (k & 31);
            }
        }
        CU(upload_vec(ctx->d_present, present.data(), 2048, &bytes));
    }
    CU(upload_vec(ctx->d_rowmap, rowmap.data(), 65536, &bytes));

    // ---- lineage tree ------------------------------------------------------------------------------------
    auto clampu = [&](u64 x) { return std::min(std::max(x, s0), s1); };
    CU(upload_vec(ctx->d_node_lo, d->node_lo, nn, &bytes));
    CU(upload_vec(ctx->d_node_hi, d->node_hi, nn, &bytes));
    CU(upload_vec(ctx->d_node_type, d->node_type, nn, &bytes));
    CU(upload_vec(ctx->d_child_first, d->child_first, nn, &bytes));
    CU(upload_vec(ctx->d_child_count, d->child_count, nn, &bytes));
    {
        std::vector<NodeRec> recs(nn);
        auto seg_of = [&](u64 pos) -> u32 { return pos > s0 ? (u32)((pos - s0 - 1) / kPrefixSeg) : 0u; };  // segment of the reference in front of pos
        for (u32 i = 0; i < nn; ++i)
            recs[i] = NodeRec{(u32)(clampu(d->node_lo[i]) - s0), (u32)(clampu(d->node_hi[i]) - s0), d->child_first[i], d->child_count[i] | ((u32)d->node_type[i] << 30),
                              seg_of(clampu(d->node_lo[i])), seg_of(clampu(d->node_hi[i])), d->node_lo[i], d->node_hi[i] - d->node_lo[i]};
        CU(upload_vec(ctx->d_recs, recs.data(), nn, &bytes));
    }
    CU(upload_vec(ctx->d_ref_levels, d->ref_levels, N, &bytes));

    // ---- bit rows -----------------------------------------------------------------------------------------
    const size_t row_bytes = (size_t)row_words * 4;
    CU(ctx->d_bitrows.ensure((size_t)n_rows * row_bytes));
    CU(cudaMemsetAsync(ctx->d_bitrows.p, 0, (size_t)n_rows * row_bytes, ctx->stream));
    bytes += (u64)n_rows * row_bytes;
    if (from_seq) {
        for (size_t c = 0; c + 1 < seq_chunks.size(); ++c) {
            CU(seq_chunk_to_device(c));
            {
                LaunchTimer lt(ctx, RTX_K_INDEX);
                bitrows_from_seq_kernel<<<ctx->n_sms * 8, 256, 0, ctx->stream>>>(ctx->d_idx_off.as<u64>(), ctx->d_seq_codes.as<u8>(),
                                                                                (u32)(seq_chunks[c + 1] - seq_chunks[c]), seq_chunks[c] - s0,
                                                                                ctx->d_rowmap.as<u32>(), ctx->d_bitrows.as<u32>(), row_words);
            }
            CU(cudaGetLastError());
            CU(cudaStreamSynchronize(ctx->stream));
        }
        ctx->d_seq_codes.release();
        ctx->d_idx_off.release();
    } else
        CU(upload_vec(ctx->d_csr_off, d->csr_offsets, 65537, nullptr));
    if (nnz) {
        if (ctx->keep_csr) {
            CU(upload_vec(ctx->d_csr_ids, d->csr_ids, nnz, &bytes));
            bytes += 65537 * 8;
            LaunchTimer lt(ctx, RTX_K_INDEX);
            build_bitrows_kernel<<<ctx->n_sms * 8, 256, 0, ctx->stream>>>(ctx->d_csr_off.as<u64>(), ctx->d_csr_ids.as<u32>(), nnz,
                                                                         ctx->d_rowmap.as<u32>(), ctx->d_bitrows.as<u32>(), row_words,
                                                                         s0, s1);
        } else {
            // stream the postings through a bounded device buffer; offsets are rebased per chunk on the device side
            const u64 chunk = 64ull << 20;  // postings per chunk (256 MB)
            CU(ctx->d_csr_ids.ensure(std::min(nnz, chunk) * 4));
            std::vector<u64> off_chunk(65537);
            for (u64 p0 = 0; p0 < nnz; p0 += chunk) {
                const u64 cn = std::min(chunk, nnz - p0);
                CU(cudaMemcpyAsync(ctx->d_csr_ids.p, d->csr_ids + p0, cn * 4, cudaMemcpyHostToDevice, ctx->stream));
                for (u32 k = 0; k <= 65536; ++k) {
                    u64 o = d->csr_offsets[k];
                    off_chunk[k] = o <= p0 ? 0 : std::min(o - p0, cn);
                }
                // csr_off[k] <= p  <=> posting p of this chunk belongs to a k-mer >= k
                CU(cudaMemcpyAsync(ctx->d_csr_off.p, off_chunk.data(), 65537 * 8, cudaMemcpyHostToDevice, ctx->stream));
                {
                    LaunchTimer lt(ctx, RTX_K_INDEX);
                    build_bitrows_kernel<<<ctx->n_sms * 8, 256, 0, ctx->stream>>>(ctx->d_csr_off.as<u64>(), ctx->d_csr_ids.as<u32>(),
                                                                                 cn, ctx->d_rowmap.as<u32>(), ctx->d_bitrows.as<u32>(),
                                                                                 row_words, s0, s1);
                }
                CU(cudaStreamSynchronize(ctx->stream));  // off_chunk / pageable source reused next iteration
            }
        }
    }
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(ctx->stream));
    if (!ctx->keep_csr) {
        ctx->d_csr_ids.release();
        ctx->d_csr_off.release();
    }

    // ---- straddling nodes (reference-sharded mode) -----------------------------------------------------------
    {
        std::vector<int> strad_of(nn, -1), strad_parent;
        std::vector<u32> strad_nodes;
        if (n_shards > 1) {
            std::vector<int> parent(nn, -1);
            for (u32 i = 0; i < nn; ++i)
                for (u32 c = d->child_first[i]; c < d->child_first[i] + d->child_count[i]; ++c) parent[c] = (int)i;
            for (u32 i = 0; i < nn; ++i) {  // BFS order: parents precede children
                const u64 lo = d->node_lo[i], hi = d->node_hi[i];
                bool crosses = false;
                for (u32 r = 1; r < n_shards && !crosses; ++r) crosses = lo < d->shard_cuts[r] && d->shard_cuts[r] < hi;
                if (crosses) {
                    strad_of[i] = (int)strad_nodes.size();
                    strad_nodes.push_back(i);
                    strad_parent.push_back(parent[i] >= 0 ? strad_of[parent[i]] : -1);
                }
            }
        }
        CU(upload_vec(ctx->d_strad_of_node, strad_of.data(), nn, &bytes));
        CU(upload_vec(ctx->d_strad_nodes, strad_nodes.data(), strad_nodes.size(), &bytes));
        CU(upload_vec(ctx->d_strad_parent, strad_parent.data(), strad_parent.size(), &bytes));
        ctx->sv = ShardView{};
        ctx->sv.n_strad = (u32)strad_nodes.size();
        ctx->sv.n_shards = n_shards;
        ctx->sv.rank = n_shards > 1 ? d->shard_rank : 0;
        ctx->sv.strad_of_node = ctx->d_strad_of_node.as<int>();
        ctx->sv.strad_nodes = ctx->d_strad_nodes.as<u32>();
        ctx->sv.strad_parent = ctx->d_strad_parent.as<int>();
    }

    ix.bitrows = ctx->d_bitrows.as<u32>();
    ix.rowmap = ctx->d_rowmap.as<u32>();
    ix.present = ctx->d_present.as<u32>();
    ix.csr_off = ctx->keep_csr ? ctx->d_csr_off.as<u64>() : nullptr;
    ix.csr_ids = ctx->keep_csr ? ctx->d_csr_ids.as<u32>() : nullptr;
    ix.row_words = row_words;
    ix.n_refs = N;
    ix.shard_begin = s0;
    ix.shard_refs = Ns;
    ix.n_pad = (u64)row_words * 32;
    ix.node_lo = ctx->d_node_lo.as<u32>();
    ix.node_hi = ctx->d_node_hi.as<u32>();
    ix.node_type = ctx->d_node_type.as<u8>();
    ix.child_first = ctx->d_child_first.as<u32>();
    ix.child_count = ctx->d_child_count.as<u32>();
    ix.n_nodes = nn;
    ix.max_levels = max_levels;
    ix.ref_levels = ctx->d_ref_levels.as<u8>();
    ctx->n_rows = n_rows;
    ctx->index_bytes = bytes;
    {
        for (int i = 0; i < 2; ++i) {  // sized for the previous index
            BatchState& st = i ? ctx->parked : static_cast<BatchState&>(*ctx);
            DevBuf* scratch[] = {&st.d_counts, &st.d_counts1, &st.d_preb, &st.d_preb1, &st.d_segoff, &st.d_segoff1, &st.d_ptab, &st.d_ptab1, &st.d_cbuf};
            for (DevBuf* b : scratch) b->release();
        }
        size_t mem_free = 0, mem_total = 0;
        if (cudaMemGetInfo(&mem_free, &mem_total) != cudaSuccess) mem_free = 8ull << 30;
        ctx->mem_free_after_index = mem_free;
    }
    ctx->has_index = true;
    return RTX_OK;
}

// ---------------------------------------------------------------------------------------------------------
// batch upload
// ---------------------------------------------------------------------------------------------------------
static int ensure_pool(rtx_ctx* ctx, u64 cap) {
    const u32 ML = ctx->ix.max_levels;
    CU(ctx->d_pool_first.ensure(cap * 4));
    CU(ctx->d_pool_nlev.ensure(cap));
    CU(ctx->d_pool_conf.ensure(cap * ML * 8));
    CU(ctx->d_pool_local.ensure(cap * 8));
    CU(ctx->d_pool_used.ensure(8));
    CU(ctx->d_ord_first.ensure(cap * 4));
    CU(ctx->d_ord_nlev.ensure(cap));
    CU(ctx->d_ord_conf.ensure(cap * ML * 8));
    CU(ctx->d_ord_local.ensure(cap * 8));
    ctx->pool.first_ref = ctx->d_pool_first.as<u32>();
    ctx->pool.n_levels = ctx->d_pool_nlev.as<u8>();
    ctx->pool.conf = ctx->d_pool_conf.as<double>();
    ctx->pool.local = ctx->d_pool_local.as<double>();
    ctx->pool.used = ctx->d_pool_used.as<unsigned long long>();
    ctx->pool.cap = cap;
    ctx->pool_levels = ML;
    return RTX_OK;
}

// Before a slot's kernels are issued: its per-sub-batch scratch large enough for the batch's layout, its ProbScratch pointed at it, the
// per-function shared-memory ceilings set for this layout.  Growing a buffer goes through cudaFree, which waits for the device.
static int bind_scratch(rtx_ctx* ctx) {
    CU(ctx->d_counts.ensure(std::max<size_t>(ctx->need_counts, 1)));
    CU(ctx->d_cbuf.ensure(std::max<size_t>(ctx->need_cbuf, 1)));
    CU(ctx->d_preb.ensure(std::max<size_t>(ctx->need_preb, 1)));
    CU(ctx->d_ptab.ensure(std::max<size_t>(ctx->need_ptab, 1)));
    CU(ctx->d_segoff.ensure(std::max<size_t>(ctx->need_segoff, 1)));
    if (ctx->need_prob_big) CU(ctx->d_prob_big.ensure(ctx->need_prob_big));
    ctx->sc.ptab = ctx->d_ptab.as<double>();
    ctx->sc.cbuf = ctx->d_cbuf.as<double>();
    ctx->sc.blk = ctx->d_preb.as<double>();
    ctx->sc.counts = ctx->d_counts.as<u16>();
    ctx->sc.counts_stride = (size_t)ctx->ix.n_pad;
    ctx->sc.hstride = ctx->bv.hstride;
    ctx->sc.segoff = ctx->d_segoff.as<double>();
    ctx->sc.big = ctx->need_prob_big ? ctx->d_prob_big.as<unsigned char>() : nullptr;
    ctx->sc1 = ctx->sc;
    if (ctx->two_slots) {
        CU(ctx->d_counts1.ensure(std::max<size_t>(ctx->need_counts, 1)));
        CU(ctx->d_preb1.ensure(std::max<size_t>(ctx->need_preb, 1)));
        CU(ctx->d_ptab1.ensure(std::max<size_t>(ctx->need_ptab, 1)));
        CU(ctx->d_segoff1.ensure(std::max<size_t>(ctx->need_segoff, 1)));
        ctx->sc1.blk = ctx->d_preb1.as<double>();
        ctx->sc1.counts = ctx->d_counts1.as<u16>();
        ctx->sc1.ptab = ctx->d_ptab1.as<double>();
        ctx->sc1.segoff = ctx->d_segoff1.as<double>();
        // the log-CMF scratch is indexed by CTA slot of prob_table_kernel, which only ever runs on stream2: shared
    }
    // dynamic shared memory ceilings are per function, not per launch: set them for this slot's layout
    if (!ctx->prob_big_bytes) CU(cudaFuncSetAttribute(prob_table_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->prob_smem));
    CU(cudaFuncSetAttribute(prefix_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->prefix_smem));
    CU(cudaFuncSetAttribute(lineage_walk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->walk_smem));
    CU(cudaFuncSetAttribute(lineage_walk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->walk_smem));
    CU(cudaFuncSetAttribute(lineage_bfs_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->bfs_smem));
    CU(cudaFuncSetAttribute(lineage_bfs_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->bfs_smem));
    ctx->cur_stream = ctx->stream;
    ctx->cur_counts = ctx->d_counts.as<u16>();
    ctx->cur_sc = &ctx->sc;
    return RTX_OK;
}

RTX_API int rtx_batch_upload(rtx_ctx* ctx, const rtx_batch* batch) {
    if (!ctx) return RTX_ERR_INVALID;
    if (!ctx->has_index) return set_err(ctx, RTX_ERR_NO_INDEX, "rtx_batch_upload: no index uploaded");
    REQUIRE(batch != nullptr, "batch is NULL");
    const u32 nq = batch->n_queries;
    REQUIRE(nq == 0 || batch->seq_offsets, "seq_offsets is NULL");
    CU(cudaSetDevice(ctx->device));
    ctx->has_batch = false;
    ctx->ran = false;
    BatchView& bv = ctx->bv;
    bv = BatchView{};
    bv.n_queries = nq;
    bv.flags = batch->flags;
    if (nq == 0) {
        ctx->has_batch = true;
        return RTX_OK;
    }
    u32 max_len = 0;
    for (u32 q = 0; q < nq; ++q) {
        REQUIRE(batch->seq_offsets[q] <= batch->seq_offsets[q + 1], "seq_offsets must be non-decreasing");
        u64 l = batch->seq_offsets[q + 1] - batch->seq_offsets[q];
        REQUIRE(l <= 0x7FFFFFFFull, "query too long");
        max_len = std::max<u32>(max_len, (u32)l);
    }
    const u64 total = batch->seq_offsets[nq] - batch->seq_offsets[0];
    REQUIRE(total == 0 || batch->seq_codes, "seq_codes is NULL");
    const u32 kmax = max_len >= 8 ? max_len - 7 : 0;  // upper bound on unique 8-mers of one query
    if (kmax > 65535) return set_err(ctx, RTX_ERR_UNSUPPORTED, "query with more than 65535 8-mer windows (raxtax.rs:56 asserts the same)");
    const u32 kstride = round_up(std::max(kmax, 1u), 16);
    const u32 hstride = round_up(kmax + 1, 4);
    // probability tables in shared memory: per-warp partial sums and the ln n! table while they fit, else the compact layout
    int nprod = kProbWarps, lf_smem = 1;
    size_t smem = ProbSmem::bytes(hstride, hstride / 2 + 1, nprod, lf_smem);
    if (smem > 100 * 1024) {
        nprod = 1;
        lf_smem = 0;
        smem = ProbSmem::bytes(hstride, hstride / 2 + 1, nprod, lf_smem);
    }
    const bool big = smem > 200 * 1024;  // queries beyond ~6.4 kb: the tables of K3 move to global scratch (ProbScratch::big)
    ctx->prob_big_bytes = big ? (smem + 255) & ~(size_t)255 : 0;
    if (big) smem = 0;
    ctx->sc = ProbScratch{};
    ctx->sc.nprod = nprod;
    ctx->sc.lf_smem = lf_smem;
    ctx->max_len = max_len;
    ctx->total_codes = total;
    u64 total_exact = 0;
    if (batch->exact_offsets) {
        for (u32 q = 0; q < nq; ++q) REQUIRE(batch->exact_offsets[q] <= batch->exact_offsets[q + 1], "exact_offsets must be non-decreasing");
        REQUIRE(batch->exact_offsets[0] == 0, "exact_offsets[0] must be 0");
        total_exact = batch->exact_offsets[nq];
        REQUIRE(total_exact == 0 || batch->exact_ids, "exact_ids is NULL");
        for (u64 e = 0; e < total_exact; ++e) REQUIRE(batch->exact_ids[e] < ctx->ix.n_refs, "exact id out of range");
    }
    ctx->total_exact = total_exact;

    // H2D on the copy stream (offsets are rebased to 0 so that callers may pass a window of a larger array); the kernels of the
    // slot's next run wait for ev_up, the kernels of the OTHER slot, possibly running right now, are not disturbed
    cudaStream_t cs = ctx->stream_cp;
    CU(ctx->d_seq_off.ensure((nq + 1) * 8));
    CU(ctx->d_codes.ensure(std::max<u64>(total, 1)));
    if (batch->seq_offsets[0] == 0) {
        CU(cudaMemcpyAsync(ctx->d_seq_off.p, batch->seq_offsets, (nq + 1) * 8, cudaMemcpyHostToDevice, cs));
    } else {
        std::vector<u64> reb(nq + 1);
        for (u32 q = 0; q <= nq; ++q) reb[q] = batch->seq_offsets[q] - batch->seq_offsets[0];
        CU(cudaMemcpyAsync(ctx->d_seq_off.p, reb.data(), (nq + 1) * 8, cudaMemcpyHostToDevice, cs));
        CU(cudaStreamSynchronize(cs));
    }
    if (total) CU(cudaMemcpyAsync(ctx->d_codes.p, batch->seq_codes + batch->seq_offsets[0], total, cudaMemcpyHostToDevice, cs));
    ctx->prof.h2d_bytes += (nq + 1) * 8 + total;
    if (batch->exact_offsets) {
        CU(ctx->d_exact_off.ensure((nq + 1) * 4));
        CU(ctx->d_exact_ids.ensure(std::max<u64>(total_exact, 1) * 4));
        CU(cudaMemcpyAsync(ctx->d_exact_off.p, batch->exact_offsets, (nq + 1) * 4, cudaMemcpyHostToDevice, cs));
        if (total_exact) CU(cudaMemcpyAsync(ctx->d_exact_ids.p, batch->exact_ids, total_exact * 4, cudaMemcpyHostToDevice, cs));
        ctx->prof.h2d_bytes += (nq + 1) * 4 + total_exact * 4;
        bv.exact_off = ctx->d_exact_off.as<u32>();
        bv.exact_ids = ctx->d_exact_ids.as<u32>();
    }
    CU(cudaEventRecord(ctx->ev_up, cs));
    ctx->up_pending = true;
    bv.seq_off = ctx->d_seq_off.as<u64>();
    bv.codes = ctx->d_codes.as<u8>();
    bv.kstride = kstride;
    bv.hstride = hstride;

    // per-query device arrays
    CU(ctx->d_K.ensure(nq * 2));
    CU(ctx->d_kmers.ensure((size_t)nq * kstride * 2));
    CU(ctx->d_rows.ensure((size_t)nq * kstride * 4));
    CU(ctx->d_nrows.ensure(nq * 4));
    CU(ctx->d_hist.ensure((size_t)nq * hstride * 4));
    bv.K = ctx->d_K.as<u16>();
    bv.kmers = ctx->d_kmers.as<u16>();
    bv.rows = ctx->d_rows.as<u32>();
    bv.nrows = ctx->d_nrows.as<u32>();
    bv.hist = ctx->d_hist.as<u32>();
    CU(ctx->d_res_off.ensure(nq * 4));
    CU(ctx->d_res_cnt.ensure(nq * 4));
    CU(ctx->d_ord_begin.ensure(((size_t)nq + 1) * 4));
    CU(ctx->d_global.ensure(nq * 8));
    CU(ctx->d_status.ensure(nq * 4));
    CU(ctx->d_hits.ensure(16));  // [0] postings-touched counter, [1] work counter of prob_table_kernel
    ctx->pool.res_off = ctx->d_res_off.as<u32>();
    ctx->pool.res_cnt = ctx->d_res_cnt.as<u32>();
    ctx->pool.global_sig = ctx->d_global.as<double>();
    ctx->pool.status = ctx->d_status.as<int>();
    // the pool's confidence arrays are sized cap x max_levels: a new index with deeper lineages needs them re-sized as well
    if (ctx->pool.cap < (u64)nq * 8 + 1024 || ctx->pool_levels != ctx->ix.max_levels) {
        int rc = ensure_pool(ctx, std::max<u64>(ctx->pool.cap, (u64)nq * 8 + 1024));
        if (rc) return rc;
    }

    // sub-batch: the per-query scratch (count vector, block prefixes, segment offsets, P(m) table) of one sub-batch may take a
    // quarter of the memory that is free now, at most 48 GB and at least 2 GiB -- large sub-batches amortise the launch tails of
    // the walk and probability kernels (C3: 1 069 queries per sub-batch at the old fixed 2 GiB, ~6 000 now)
    const u64 per_query = ctx->ix.n_pad * 2;
    u64 sb = (u64)ctx->sub_batch_opt;
    if (!sb) {
        const u64 mem_free = ctx->mem_free_after_index;  // sampled once per index upload (cudaMemGetInfo costs ~1 ms per call)
        u64 budget = std::min<u64>(std::max<u64>(mem_free / 4, 2ull << 30), 48ull << 30);
        if (ctx->comm != nullptr && ctx->sv.n_shards > 1) budget = std::min<u64>(budget, std::max<u64>(mem_free / 5, 1ull << 30));  // two scratch slots
        const u64 scratch_per_query = per_query + ((u64)ctx->ix.n_pad / kBlkRefs + ctx->ix.n_pad / kPrefixSeg + ctx->ix.n_pad / kPrefixSeg / 64 + ctx->ix.n_pad / kPrefixSeg / 4 + 8 + hstride) * 8;
        sb = std::max<u64>(1, budget / scratch_per_query);
    }
    const bool may_pipe = ctx->pipeline_opt && ctx->sv.n_shards <= 1;
    if (!ctx->sub_batch_opt && may_pipe && nq >= 4096) sb = std::min<u64>(sb, std::max<u64>(1024, (nq + 3) / 4));  // >= 4 pipeline stages
    sb = std::min<u64>(std::min<u64>(sb, nq), 65535);
    ctx->sub_batch = (u32)sb;
    ctx->two_slots = (may_pipe && nq > sb) || (ctx->comm != nullptr && ctx->sv.n_shards > 1 && nq > 1);
    ctx->sub_batch_agreed = false;
    ctx->merged = false;
    ctx->need_counts = sb * per_query;

    // probability kernel scratch
    ctx->prob_smem = smem;
    int occ = 0;
    if (big) {
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, prob_table_kernel<true>, kProbThreads, 0));
    } else {
        CU(cudaFuncSetAttribute(prob_table_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, prob_table_kernel<false>, kProbThreads, smem));
    }
    if (occ < 1) return set_err(ctx, RTX_ERR_CUDA, "prob_table_kernel does not fit on an SM");
    {
        const size_t n_seg = ctx->ix.n_pad / kPrefixSeg;
        ctx->prefix_smem = ((ctx->prob_big_bytes ? (size_t)0 : (size_t)hstride) + ((n_seg + 1) & ~(size_t)1)) * 8 +
                           ((n_seg + 31) / 32) * 4 + 16;
        if (ctx->prefix_smem > 220 * 1024)
            return set_err(ctx, RTX_ERR_UNSUPPORTED, "reference shard too large for the prefix kernel's segment table (more than ~11 M references per GPU): shard the references");
    }
    ctx->walk_smem = (size_t)kWalkWarps * WalkSmem::bytes(ctx->ix.max_levels);
    ctx->bfs_smem = BfsSmem::bytes(ctx->ix.max_levels) + bfs_ptab_smem(hstride) + bfs_skip_smem(ctx->ix.n_pad);
    ctx->shard_phase = 0;
    int slots = (int)std::min<u64>((u64)ctx->n_sms * occ, sb);
    const u32 tstride = round_up(hstride / 2 + 1, 4);
    ctx->sc.tstride = tstride;
    ctx->sc.cbuf_stride = (size_t)hstride * tstride;
    ctx->sc.big = nullptr;
    ctx->sc.big_stride = 0;
    ctx->need_prob_big = 0;
    if (ctx->prob_big_bytes) {
        // long queries: the log-CMF scratch of one CTA slot is hstride x tstride doubles (1 GB at 16 k 8-mers); as many slots as fit a
        // quarter of the free memory (at most 16 GB), at least one
        const u64 per_slot = (u64)ctx->sc.cbuf_stride * 8 + ctx->prob_big_bytes;
        const u64 budget = std::min<u64>(ctx->mem_free_after_index / 4, 16ull << 30);
        if (per_slot > budget)
            return set_err(ctx, RTX_ERR_UNSUPPORTED, "query too long: the probability scratch of one query (" + std::to_string(per_slot >> 20) +
                                                         " MB) does not fit a quarter of the free device memory");
        slots = (int)std::max<u64>(1, std::min<u64>((u64)slots, budget / per_slot));
        ctx->need_prob_big = (size_t)slots * ctx->prob_big_bytes;
        ctx->sc.big_stride = ctx->prob_big_bytes;
    }
    ctx->prob_slots = slots;
    ctx->sc.blk_stride = (size_t)ctx->ix.n_pad / kBlkRefs;  // one value per block of references
    ctx->need_cbuf = (size_t)slots * ctx->sc.cbuf_stride * 8;
    ctx->need_preb = (size_t)sb * ctx->sc.blk_stride * 8;
    ctx->need_ptab = (size_t)sb * hstride * 8;
    {   // per query: n_seg segment offsets | u32 aux[2 + n_seg/32] (m_min, skip bitmap; ProbScratch::seg_aux_off)
        const u32 n_seg = (u32)(ctx->ix.n_pad / kPrefixSeg);
        ctx->sc.seg_aux_off = round_up(n_seg, 2);
        ctx->sc.segoff_stride = round_up(ctx->sc.seg_aux_off + 1 + ((n_seg + 31) / 32 + 1) / 2 + (n_seg + 3) / 4, 4);  // + u16 segmax[n_seg]
    }
    ctx->need_segoff = (size_t)sb * ctx->sc.segoff_stride * 8;
    ctx->has_batch = true;
    int rc = bind_scratch(ctx);  // allocation failures surface here, at upload time
    if (rc) {
        ctx->has_batch = false;
        return rc;
    }
    return RTX_OK;
}

// ---------------------------------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------------------------------
// L2 blocking shared by both bit-row kernels: CTAs are scheduled query-fastest, so all queries of one reference tile group
// run together; the group's slice of the bit matrix (n_rows x tiles x 256 bytes) should stay resident in the 126 MB L2.
static void hit_tile_groups(const rtx_ctx* c, int* n_tiles, int* groups, int* tiles_per_cta) {
    *n_tiles = (int)(c->ix.row_words / (32 * kLaneWords));
    int max_tiles = c->hit_max_tiles;
    if (max_tiles <= 0) {
        const double slice_bytes_per_tile = (double)c->n_rows * 32.0 * kLaneWords * 4.0;
        max_tiles = (int)std::min(64.0, std::max(4.0, std::floor(64e6 / slice_bytes_per_tile)));
    }
    *groups = (*n_tiles + max_tiles - 1) / max_tiles;
    *tiles_per_cta = (*n_tiles + *groups - 1) / *groups;
}

// single-query kernel: one query per CTA, its tile group's tiles spread over the warps
template <int NP>
static cudaError_t launch_hitcount(rtx_ctx* c, int q_base, int qb) {
    int n_tiles, groups, tiles_per_cta;
    hit_tile_groups(c, &n_tiles, &groups, &tiles_per_cta);
    // warps per CTA: the count in [4, 8] that wastes the fewest warp slots in the last round
    int nwarps = 0;
    double best = -1.0;
    for (int w = 8; w >= 4; --w) {
        const int rounds = (tiles_per_cta + w - 1) / w;
        const double eff = (double)tiles_per_cta / (rounds * w);
        if (eff > best + 1e-9) {
            best = eff;
            nwarps = w;
        }
    }
    const bool hist_global = (size_t)(kRowListCap + c->bv.hstride) * 4 > 200 * 1024;  // tens of thousands of 8-mers per query
    const size_t smem = (size_t)(kRowListCap + (hist_global ? 0 : c->bv.hstride)) * 4;
    cudaError_t e = cudaFuncSetAttribute(hitcount_bitrows_kernel<NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    dim3 grid(qb, groups);
    c->hit_kernel = "hitcount_bitrows_kernel<" + std::to_string(NP) + ">";
    hitcount_bitrows_kernel<NP><<<grid, nwarps * 32, smem, c->cur_stream>>>(c->ix, c->bv, c->cur_counts, q_base, tiles_per_cta, n_tiles,
                                                                          hist_global ? 1 : 0);
    return cudaGetLastError();
}

// query-group kernel: G queries per CTA (one per warp) over the same reference tiles
template <int NP>
static cudaError_t launch_hitcount_group(rtx_ctx* c, int q_base, int qb, int G) {
    int n_tiles, groups, tiles_per_cta;
    hit_tile_groups(c, &n_tiles, &groups, &tiles_per_cta);
    const size_t smem = (size_t)G * (c->bv.kstride + c->bv.hstride) * 4;
    cudaError_t e = cudaFuncSetAttribute(hitcount_group_kernel<NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    dim3 grid((qb + G - 1) / G, groups);
    const u32 n_seg = (u32)(c->ix.n_pad / kPrefixSeg);
    u16* segmax = const_cast<u16*>(seg_max(*c->cur_sc, 0, n_seg));
    c->hit_kernel = "hitcount_group_kernel<" + std::to_string(NP) + "> (" + std::to_string(G) + " queries per CTA)";
    hitcount_group_kernel<NP><<<grid, G * 32, smem, c->cur_stream>>>(c->ix, c->bv, c->cur_counts, q_base, qb, tiles_per_cta, n_tiles, segmax,
                                                                   c->cur_sc->segoff_stride * 4);
    c->segmax_valid = true;
    return cudaGetLastError();
}

// kmax: the most 8-mers of a query in the sub-batch, which bounds the counts and so the bit planes (NP) the kernels keep
static cudaError_t launch_hitcount_bitrows(rtx_ctx* c, int q_base, int qb, u32 kmax) {
    // queries per CTA: 4 on indexes of a few GB, 16 on large ones -- measured (profiles/r2_hitcount_group_by_index_size.txt): on 1 M x 650 bp
    // references (8.2 GB of bit rows) 16 queries per CTA are 5.8 % faster than 4 (more rows shared through the L1, less L2 traffic), on
    // 100 k references (0.8 GB) and on 500 k x 1500 bp (4.1 GB) they are 1-5 % slower
    int G = c->hit_group;  // 0 = default
    if (G == 0) G = ((u64)c->n_rows * c->ix.row_words * 4 >= (6ull << 30)) ? 16 : 4;
    while (G > 1 && (size_t)G * (c->bv.kstride + c->bv.hstride) * 4 > 150 * 1024) G /= 2;  // long queries: smaller groups
    const bool single = G == 1 || qb < G;
    const int NP = kmax < (1u << 8) ? 8 : kmax < (1u << 10) ? 10 : kmax < (1u << 11) ? 11 : kmax < (1u << 13) ? 13 : 16;
    switch (NP) {
        case 8: return single ? launch_hitcount<8>(c, q_base, qb) : launch_hitcount_group<8>(c, q_base, qb, G);
        case 10: return single ? launch_hitcount<10>(c, q_base, qb) : launch_hitcount_group<10>(c, q_base, qb, G);
        case 11: return single ? launch_hitcount<11>(c, q_base, qb) : launch_hitcount_group<11>(c, q_base, qb, G);
        case 13: return single ? launch_hitcount<13>(c, q_base, qb) : launch_hitcount_group<13>(c, q_base, qb, G);
        default: return single ? launch_hitcount<16>(c, q_base, qb) : launch_hitcount_group<16>(c, q_base, qb, G);
    }
}

static int run_phase1(rtx_ctx* ctx, int q_base, int qb) {
    const u32 kmax = ctx->max_len >= 8 ? ctx->max_len - 7 : 0;
    LaunchTimer lt(ctx, RTX_K_HITCOUNT);
    ctx->segmax_valid = false;  // only the query-group bit-row kernel leaves per-segment maxima for K4
    if (ctx->variant == RTX_HITCOUNT_CSR) {
        if (!ctx->ix.csr_ids && kmax > 0 && ctx->n_rows > 1)
            return set_err(ctx, RTX_ERR_INVALID, "CSR hit-count variant needs RTX_OPT_KEEP_CSR set before rtx_index_upload");
        const size_t smem = (size_t)(kCsrTileRefs / 2 + ctx->bv.hstride) * 4;
        CU(cudaFuncSetAttribute(hitcount_csr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        dim3 grid(qb, (unsigned)((ctx->ix.shard_refs + kCsrTileRefs - 1) / kCsrTileRefs));
        ctx->hit_kernel = "hitcount_csr_kernel";
        hitcount_csr_kernel<<<grid, kCsrThreads, smem, ctx->cur_stream>>>(ctx->ix, ctx->bv, ctx->cur_counts, q_base);
        CU(cudaGetLastError());
    } else {
        CU(launch_hitcount_bitrows(ctx, q_base, qb, kmax));
    }
    return RTX_OK;
}

// K3 (P(m) tables) + K4 (prefix sums at node boundaries) of one sub-batch
static int launch_prob(rtx_ctx* ctx, int q0, int qb) {
    {
        CU(cudaMemsetAsync(ctx->d_hits.as<unsigned long long>() + 1, 0, 8, ctx->cur_stream));  // the kernel's work counter
        LaunchTimer lt(ctx, RTX_K_PROB);
        const int grid = std::min(ctx->prob_slots, qb);
        if (ctx->cur_sc->big)
            prob_table_kernel<true><<<grid, kProbThreads, 0, ctx->cur_stream>>>(ctx->ix, ctx->bv, ctx->pool, *ctx->cur_sc, q0, qb,
                                                                                ctx->d_hits.as<unsigned long long>(),
                                                                                ctx->d_hits.as<unsigned long long>() + 1);
        else
            prob_table_kernel<false><<<grid, kProbThreads, ctx->prob_smem, ctx->cur_stream>>>(ctx->ix, ctx->bv, ctx->pool, *ctx->cur_sc, q0, qb,
                                                                                            ctx->d_hits.as<unsigned long long>(),
                                                                                            ctx->d_hits.as<unsigned long long>() + 1);
        CU(cudaGetLastError());
    }
    {
        LaunchTimer lt(ctx, RTX_K_PREFIX);
        prefix_kernel<<<qb, kPrefixThreads, ctx->prefix_smem, ctx->cur_stream>>>(ctx->ix, ctx->bv, *ctx->cur_sc, ctx->cur_counts, q0, qb,
                                                                                 ctx->segmax_valid ? 1 : 0);
        CU(cudaGetLastError());
    }
    return RTX_OK;
}

// the batch's result lines into query order (d_ord_*); part of every run, so that a download is plain copies
static int order_results(rtx_ctx* ctx) {
    const u32 nq = ctx->bv.n_queries;
    {
        LaunchTimer lt(ctx, RTX_K_WALK);
        result_scan_kernel<<<1, kScanThreads, 0, ctx->stream>>>(ctx->pool, ctx->d_ord_begin.as<u32>(), nq);
        CU(cudaGetLastError());
    }
    {
        LaunchTimer lt(ctx, RTX_K_WALK);
        result_gather_kernel<<<(nq + 7) / 8, 256, 0, ctx->stream>>>(ctx->pool, ctx->d_ord_begin.as<u32>(), ctx->d_ord_first.as<u32>(),
                                                                    ctx->d_ord_nlev.as<u8>(), ctx->d_ord_conf.as<double>(),
                                                                    ctx->d_ord_local.as<double>(), nq, ctx->ix.max_levels);
        CU(cudaGetLastError());
    }
    return RTX_OK;
}

// before the first kernel of a slot's run: scratch bound to this slot's layout, inputs (H2D on the copy stream) in place
static int begin_run(rtx_ctx* ctx) {
    int rc = bind_scratch(ctx);
    if (rc) return rc;
    if (ctx->up_pending) {
        CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_up, 0));
        ctx->up_pending = false;
    }
    // two hit-count kernels side by side would only halve each other's L2 share: this batch's kernels start when the hit counting of
    // the batch in the other slot is through, i.e. under that batch's tail kernels
    if (ctx->parked.k2_recorded) CU(cudaStreamWaitEvent(ctx->stream, ctx->parked.ev_k2, 0));
    ctx->k2_recorded = false;
    return RTX_OK;
}

// tree walk of a sub-batch (SH: of this shard's part of the tree): the level-synchronous kernel, then the depth-first walker for the
// queries it handed back (RTX_OPT_WALK_VARIANT 1: depth-first walker only)
template <bool SH>
static int launch_walk(rtx_ctx* ctx, const ShardView& sv, const ProbScratch& sc, int q0, int qb, cudaStream_t st) {
    LaunchTimer lt(ctx, RTX_K_WALK);
    const bool bfs = ctx->walk_variant != 1;
    if (bfs) {
        const u32 cap = ctx->walk_log_cap ? (u32)ctx->walk_log_cap : kBfsEntries;
        lineage_bfs_kernel<SH><<<qb, kBfsThreads, ctx->bfs_smem, st>>>(ctx->ix, ctx->d_recs.as<NodeRec>(), ctx->bv, ctx->pool, sc, sv, q0, qb, cap,
                                                                     ctx->walk_variant == 3 ? 0 : ctx->walk_variant == 4 ? 2 : 1);
        CU(cudaGetLastError());
    }
    lineage_walk_kernel<SH><<<(qb + kWalkWarps - 1) / kWalkWarps, kWalkWarps * 32, ctx->walk_smem, st>>>(
        ctx->ix, ctx->d_recs.as<NodeRec>(), ctx->bv, ctx->pool, sc, sv, q0, qb, bfs ? 1 : 0);
    CU(cudaGetLastError());
    return RTX_OK;
}

static int run_all(rtx_ctx* ctx) {
    BatchView& bv = ctx->bv;
    const u32 nq = bv.n_queries;
    if (nq == 0) return RTX_OK;
    if (ctx->sv.n_shards > 1)
        return set_err(ctx, RTX_ERR_INVALID, "this context holds one shard of a reference-sharded index: use the rtx_shard_phase* calls");
    {
        int rc = begin_run(ctx);
        if (rc) return rc;
    }
    CU(cudaMemsetAsync(ctx->d_hist.p, 0, (size_t)nq * bv.hstride * 4, ctx->stream));
    CU(cudaMemsetAsync(ctx->d_pool_used.p, 0, 8, ctx->stream));
    CU(cudaMemsetAsync(ctx->d_hits.p, 0, 8, ctx->stream));
    {
        LaunchTimer lt(ctx, RTX_K_KMERS);
        kmers_kernel<<<nq, kKmerThreads, 0, ctx->stream>>>(ctx->ix, bv);
        CU(cudaGetLastError());
    }
    // Sub-batch pipeline: hit counting of sub-batch i runs on `stream`, everything behind it (probabilities, prefix sums,
    // tree walk, taps) on `stream2` with the buffers of slot i & 1, so that the L2/ALU-bound hit counting of the next
    // sub-batch overlaps the FP64/latency-bound tail of this one.
    const bool pipe = ctx->two_slots;
    u32 i_sub = 0;
    for (u32 q0 = 0; q0 < nq; q0 += ctx->sub_batch, ++i_sub) {
        const int qb = (int)std::min<u32>(ctx->sub_batch, nq - q0);
        const int slot = pipe ? (int)(i_sub & 1u) : 0;
        ctx->cur_counts = slot ? ctx->d_counts1.as<u16>() : ctx->d_counts.as<u16>();
        ctx->cur_sc = slot ? &ctx->sc1 : &ctx->sc;
        ctx->cur_stream = ctx->stream;
        if (pipe && i_sub >= 2) CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_post[slot], 0));  // the slot's previous tenant is done
        int rc = run_phase1(ctx, (int)q0, qb);
        if (rc) return rc;
        if ((bv.flags & RTX_SKIP_EXACT_MATCHES) && bv.exact_off) {
            LaunchTimer lt(ctx, RTX_K_FIXUP);
            fixup_exact_kernel<<<(qb + 127) / 128, 128, 0, ctx->cur_stream>>>(ctx->ix, bv, ctx->cur_counts, (int)q0, qb);
            CU(cudaGetLastError());
        }
        if (q0 + ctx->sub_batch >= nq) {  // the run's last hit-count launch: the batch in the other slot may start counting behind it
            CU(cudaEventRecord(ctx->ev_k2, ctx->stream));
            ctx->k2_recorded = true;
        }
        if (pipe) {
            CU(cudaEventRecord(ctx->ev_hit[slot], ctx->stream));
            ctx->cur_stream = ctx->stream2;
            CU(cudaStreamWaitEvent(ctx->stream2, ctx->ev_hit[slot], 0));
        }
        {
            int rc2 = launch_prob(ctx, (int)q0, qb);
            if (rc2) return rc2;
        }
        {
            int rc2 = launch_walk<false>(ctx, ShardView{}, *ctx->cur_sc, (int)q0, qb, ctx->cur_stream);
            if (rc2) return rc2;
        }
        if (ctx->tap_counts_host) {
            const u64 Ns = ctx->ix.shard_refs;
            CU(cudaMemcpy2DAsync(ctx->tap_counts_host + (size_t)q0 * Ns, Ns * 2, ctx->cur_counts, ctx->ix.n_pad * 2, Ns * 2, qb,
                                 cudaMemcpyDeviceToHost, ctx->cur_stream));
            ctx->prof.d2h_bytes += (u64)qb * Ns * 2;
        }
        if (ctx->tap_probs_host) {
            const u64 w = std::min<u64>(ctx->tap_prob_stride, bv.hstride);
            CU(cudaMemcpy2DAsync(ctx->tap_probs_host + (size_t)q0 * ctx->tap_prob_stride, ctx->tap_prob_stride * 8, ctx->cur_sc->ptab,
                                 (size_t)bv.hstride * 8, w * 8, qb, cudaMemcpyDeviceToHost, ctx->cur_stream));
            ctx->prof.d2h_bytes += (u64)qb * w * 8;
        }
        if (pipe) CU(cudaEventRecord(ctx->ev_post[slot], ctx->stream2));
    }
    if (pipe) {  // everything issued later on `stream` (downloads, the next run) is ordered behind both slots
        CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_post[0], 0));
        if (i_sub >= 2) CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_post[1], 0));
    }
    ctx->cur_stream = ctx->stream;
    ctx->cur_counts = ctx->d_counts.as<u16>();
    ctx->cur_sc = &ctx->sc;
    {
        int rc = order_results(ctx);
        if (rc) return rc;
    }
    CU(cudaEventRecord(ctx->ev_done, ctx->stream));
    ctx->prof.queries += nq;
    ctx->runs_since_download += 1;
    ctx->ran = true;
    return RTX_OK;
}

RTX_API int rtx_batch_run(rtx_ctx* ctx) {
    if (!ctx) return RTX_ERR_INVALID;
    if (!ctx->has_batch) return set_err(ctx, RTX_ERR_INVALID, "rtx_batch_run: no batch uploaded");
    CU(cudaSetDevice(ctx->device));
    return run_all(ctx);
}

// ---------------------------------------------------------------------------------------------------------
// download
// ---------------------------------------------------------------------------------------------------------
RTX_API int rtx_batch_download(rtx_ctx* ctx, rtx_results* res) {
    if (!ctx) return RTX_ERR_INVALID;
    REQUIRE(res != nullptr, "results is NULL");
    if (!ctx->has_batch || (!ctx->ran && ctx->bv.n_queries)) return set_err(ctx, RTX_ERR_INVALID, "rtx_batch_download: nothing was run");
    CU(cudaSetDevice(ctx->device));
    const BatchView& bv = ctx->bv;
    const u32 nq = bv.n_queries;
    res->n_results = 0;
    if (nq == 0) {
        if (res->result_begin) res->result_begin[0] = 0;
        return RTX_OK;
    }
    REQUIRE(res->result_begin && res->n_kmers && res->global_signal, "result_begin / n_kmers / global_signal must be provided");
    const u32 ML = ctx->ix.max_levels;
    cudaStream_t cs = ctx->stream_cp;
    CU(cudaStreamWaitEvent(cs, ctx->ev_done, 0));  // this slot's kernels; the other slot may be running on `stream` meanwhile
    // round 1: per-query metadata through the pinned arena, one synchronisation
    const size_t meta_bytes = 2 * 64 + ((size_t)nq + 1) * 4 + (size_t)nq * (4 + 4 + 2 + 8) + 6 * 64;
    CU(arena_reserve(ctx, meta_bytes));
    unsigned long long* h_used = (unsigned long long*)arena_take(ctx, 16);
    u32* h_begin = (u32*)arena_take(ctx, ((size_t)nq + 1) * 4);
    int* h_status = (int*)arena_take(ctx, (size_t)nq * 4);
    u32* h_nrows = (u32*)arena_take(ctx, (size_t)nq * 4);
    CU(cudaMemcpyAsync(&h_used[0], ctx->d_pool_used.p, 8, cudaMemcpyDeviceToHost, cs));
    CU(cudaMemcpyAsync(&h_used[1], ctx->d_hits.p, 8, cudaMemcpyDeviceToHost, cs));
    CU(cudaMemcpyAsync(h_begin, ctx->d_ord_begin.p, ((size_t)nq + 1) * 4, cudaMemcpyDeviceToHost, cs));
    CU(cudaMemcpyAsync(h_status, ctx->d_status.p, (size_t)nq * 4, cudaMemcpyDeviceToHost, cs));
    CU(cudaMemcpyAsync(h_nrows, ctx->d_nrows.p, (size_t)nq * 4, cudaMemcpyDeviceToHost, cs));
    CU(d2h(ctx, res->n_kmers, ctx->d_K.p, (size_t)nq * 2, host_ptr_pinned(res->n_kmers)));
    CU(d2h(ctx, res->global_signal, ctx->d_global.p, (size_t)nq * 8, host_ptr_pinned(res->global_signal)));
    CU(d2h_finish(ctx));
    const unsigned long long used = ctx->merged ? (unsigned long long)h_begin[nq] : h_used[0], hits = h_used[1];
    ctx->prof.d2h_bytes += 16 + 4 + (u64)nq * (3 * 4 + 2 + 8);
    {
        // every run since the last download processed this same batch: account them all
        const u64 runs = ctx->runs_since_download;
        ctx->runs_since_download = 0;
        u64 rows = 0;
        for (u32 q = 0; q < nq; ++q) rows += h_nrows[q];
        ctx->prof.hits += hits * runs;
        ctx->prof.bitrow_bytes += runs * (rows * (u64)ctx->ix.row_words * 4 + (u64)nq * ctx->ix.n_pad * 2);
        ctx->prof.csr_equiv_bytes += runs * (4 * (u64)hits + (u64)nq * ctx->ix.shard_refs * 2);
    }
    bool pool_overflow = false;
    for (u32 q = 0; q < nq; ++q) {
        switch (h_status[q]) {
            case kQOk: break;
            case kQPoolOverflow: pool_overflow = true; break;
            case kQProbSumZero:
                return set_err(ctx, RTX_ERR_ASSERT, "query " + std::to_string(q) + ": probs_sum > 0.0 violated (prob.rs:98)");
            case kQEmptyResult:
                return set_err(ctx, RTX_ERR_ASSERT, "query " + std::to_string(q) + ": empty evaluation result (raxtax.rs:72)");
            case kQTooManyResults:
                return set_err(ctx, RTX_ERR_UNSUPPORTED, "query " + std::to_string(q) + ": more than RTX_MAX_RESULTS_PER_QUERY result lines");
            default: return set_err(ctx, RTX_ERR_CUDA, "query " + std::to_string(q) + ": unknown device status");
        }
    }
    if (pool_overflow && ctx->merged)
        return set_err(ctx, RTX_ERR_CUDA, "result pool overflow after rtx_shard_gather (the gather sizes the pools of all ranks before merging)");
    if (pool_overflow) {
        // grow the pool and redo the whole batch once (counts of earlier sub-batches are gone)
        int rc = ensure_pool(ctx, used + used / 4 + 1024);
        if (rc) return rc;
        if (ctx->sv.n_shards > 1) {  // counts and prefixes are still resident: only the walk has to be repeated
            CU(cudaMemsetAsync(ctx->d_pool_used.p, 0, 8, ctx->stream));
            ctx->shard_phase = 2;
            rc = rtx_shard_phase3(ctx);
            if (rc) return rc;
            return rtx_batch_download(ctx, res);
        }
        rc = run_all(ctx);
        if (rc) return rc;
        return rtx_batch_download(ctx, res);
    }
    res->n_results = used;
    if ((u64)h_begin[nq] != used) return set_err(ctx, RTX_ERR_CUDA, "result accounting mismatch");
    if (used > res->result_capacity) return set_err(ctx, RTX_ERR_INVALID, "result_capacity too small; n_results holds the needed size");
    memcpy(res->result_begin, h_begin, ((size_t)nq + 1) * 4);  // before the arena is recycled for round 2
    if (used) {
        // round 2: the result lines, already in query order on the device
        REQUIRE(res->first_ref && res->n_levels && res->confidence && res->local_signal, "per-result output arrays must be provided");
        CU(arena_reserve(ctx, used * (4 + 1 + 8 + (size_t)ML * 8) + 4 * 64));
        CU(d2h(ctx, res->first_ref, ctx->d_ord_first.p, used * 4, host_ptr_pinned(res->first_ref)));
        CU(d2h(ctx, res->n_levels, ctx->d_ord_nlev.p, used, host_ptr_pinned(res->n_levels)));
        CU(d2h(ctx, res->confidence, ctx->d_ord_conf.p, used * ML * 8, host_ptr_pinned(res->confidence)));
        CU(d2h(ctx, res->local_signal, ctx->d_ord_local.p, used * 8, host_ptr_pinned(res->local_signal)));
        CU(d2h_finish(ctx));
        ctx->prof.d2h_bytes += used * (4 + 1 + 8 + (u64)ML * 8);
    }
    // taps
    if (res->tap_hist) {
        REQUIRE(res->tap_hist_stride >= bv.hstride || res->tap_hist_stride >= (u64)(ctx->max_len >= 8 ? ctx->max_len - 7 : 0) + 1,
                "tap_hist_stride too small");
        const u64 w = std::min<u64>(res->tap_hist_stride, bv.hstride);
        CU(cudaMemcpy2DAsync(res->tap_hist, res->tap_hist_stride * 4, ctx->d_hist.p, (size_t)bv.hstride * 4, w * 4, nq, cudaMemcpyDeviceToHost,
                             cs));
        ctx->prof.d2h_bytes += (u64)nq * w * 4;
    }
    if (res->tap_kmers) {
        const u64 w = std::min<u64>(res->tap_kmer_stride, bv.kstride);
        CU(cudaMemcpy2DAsync(res->tap_kmers, res->tap_kmer_stride * 2, ctx->d_kmers.p, (size_t)bv.kstride * 2, w * 2, nq,
                             cudaMemcpyDeviceToHost, cs));
        ctx->prof.d2h_bytes += (u64)nq * w * 2;
    }
    if (res->tap_probs && !ctx->tap_probs_host) {
        REQUIRE(ctx->sub_batch >= nq, "tap_probs through rtx_batch_download needs the whole batch in one sub-batch; use rtx_classify_batch");
        const u64 w = std::min<u64>(res->tap_prob_stride, bv.hstride);
        CU(cudaMemcpy2DAsync(res->tap_probs, res->tap_prob_stride * 8, ctx->d_ptab.p, (size_t)bv.hstride * 8, w * 8, nq, cudaMemcpyDeviceToHost,
                             cs));
        ctx->prof.d2h_bytes += (u64)nq * w * 8;
    }
    if (res->tap_counts && !ctx->tap_counts_host) {
        REQUIRE(ctx->sub_batch >= nq, "tap_counts through rtx_batch_download needs the whole batch in one sub-batch; use rtx_classify_batch");
        const u64 Ns = ctx->ix.shard_refs;
        CU(cudaMemcpy2DAsync(res->tap_counts, Ns * 2, ctx->d_counts.p, ctx->ix.n_pad * 2, Ns * 2, nq, cudaMemcpyDeviceToHost, cs));
        ctx->prof.d2h_bytes += (u64)nq * Ns * 2;
    }
    CU(cudaStreamSynchronize(cs));
    return RTX_OK;
}

RTX_API int rtx_classify_batch(rtx_ctx* ctx, const rtx_batch* batch, rtx_results* results) {
    if (!ctx) return RTX_ERR_INVALID;
    REQUIRE(results != nullptr, "results is NULL");
    int rc = rtx_batch_upload(ctx, batch);
    if (rc) return rc;
    ctx->tap_counts_host = results->tap_counts;
    ctx->tap_probs_host = results->tap_probs;
    ctx->tap_prob_stride = results->tap_prob_stride;
    rc = rtx_batch_run(ctx);
    if (rc == RTX_OK) rc = rtx_batch_download(ctx, results);
    ctx->tap_counts_host = nullptr;
    ctx->tap_probs_host = nullptr;
    return rc;
}

// ---- sharded mode ------------------------------------------------------------------------------------------
static int shard_precheck(rtx_ctx* ctx, int want_phase, const char* who) {
    if (!ctx) return RTX_ERR_INVALID;
    if (!ctx->has_batch) return set_err(ctx, RTX_ERR_INVALID, std::string(who) + ": no batch uploaded");
    if (ctx->bv.n_queries > ctx->sub_batch) return set_err(ctx, RTX_ERR_INVALID, std::string(who) + ": the batch must fit one sub-batch in sharded mode");
    if (want_phase == 0 && ctx->shard_phase == 3) ctx->shard_phase = 0;  // a finished pass may be repeated on the resident batch
    if (ctx->shard_phase != want_phase) return set_err(ctx, RTX_ERR_INVALID, std::string(who) + ": phases must run in order 1, 2, 3 after rtx_batch_upload");
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) return set_err(ctx, RTX_ERR_CUDA, cudaGetErrorString(e));
    return RTX_OK;
}

RTX_API int rtx_shard_phase1(rtx_ctx* ctx) {
    int rc = shard_precheck(ctx, 0, "rtx_shard_phase1");
    if (rc) return rc;
    BatchView& bv = ctx->bv;
    const u32 nq = bv.n_queries;
    ctx->shard_phase = 1;
    if (nq == 0) return RTX_OK;
    rc = begin_run(ctx);
    if (rc) return rc;
    CU(cudaMemsetAsync(ctx->d_hist.p, 0, (size_t)nq * bv.hstride * 4, ctx->stream));
    CU(cudaMemsetAsync(ctx->d_pool_used.p, 0, 8, ctx->stream));
    CU(cudaMemsetAsync(ctx->d_hits.p, 0, 8, ctx->stream));
    {
        LaunchTimer lt(ctx, RTX_K_KMERS);
        kmers_kernel<<<nq, kKmerThreads, 0, ctx->stream>>>(ctx->ix, bv);
        CU(cudaGetLastError());
    }
    rc = run_phase1(ctx, 0, (int)nq);
    if (rc) return rc;
    if ((bv.flags & RTX_SKIP_EXACT_MATCHES) && bv.exact_off) {
        LaunchTimer lt(ctx, RTX_K_FIXUP);
        fixup_exact_kernel<<<(nq + 127) / 128, 128, 0, ctx->stream>>>(ctx->ix, bv, ctx->d_counts.as<u16>(), 0, (int)nq);
        CU(cudaGetLastError());
    }
    // exchange buffers
    const size_t S = ctx->sv.n_strad;
    CU(ctx->d_send.ensure(std::max<size_t>(1, (size_t)nq * S) * sizeof(ShardRec)));
    CU(ctx->d_recv.ensure(std::max<size_t>(1, (size_t)nq * S) * sizeof(ShardRec) * ctx->sv.n_shards));
    CU(ctx->d_sk.ensure(std::max<size_t>(1, (size_t)nq * S)));
    CU(ctx->d_sany.ensure(std::max<size_t>(1, (size_t)nq * S)));
    CU(ctx->d_sbest.ensure(std::max<size_t>(1, (size_t)nq * S) * 4));
    ctx->sv.send = ctx->d_send.as<ShardRec>();
    ctx->sv.recv = ctx->d_recv.as<ShardRec>();
    ctx->sv.sk = ctx->d_sk.as<u8>();
    ctx->sv.sany = ctx->d_sany.as<u8>();
    ctx->sv.sbest = ctx->d_sbest.as<u32>();
    CU(cudaStreamSynchronize(ctx->stream));
    return RTX_OK;
}

RTX_API int rtx_shard_hist_buffer(rtx_ctx* ctx, void** dev_ptr, uint64_t* n_elems) {
    if (!ctx || !dev_ptr || !n_elems) return RTX_ERR_INVALID;
    if (!ctx->has_batch) return set_err(ctx, RTX_ERR_INVALID, "rtx_shard_hist_buffer: no batch uploaded");
    *dev_ptr = ctx->d_hist.p;
    *n_elems = (uint64_t)ctx->bv.n_queries * ctx->bv.hstride;
    return RTX_OK;
}

RTX_API int rtx_shard_phase2(rtx_ctx* ctx) {
    int rc = shard_precheck(ctx, 1, "rtx_shard_phase2");
    if (rc) return rc;
    BatchView& bv = ctx->bv;
    const u32 nq = bv.n_queries;
    ctx->shard_phase = 2;
    if (nq == 0) return RTX_OK;
    rc = launch_prob(ctx, 0, (int)nq);
    if (rc) return rc;
    if (ctx->sv.n_strad) {
        const long long warps = (long long)nq * ctx->sv.n_strad;
        shard_records_kernel<<<(unsigned)((warps * 32 + 127) / 128), 128, 0, ctx->stream>>>(ctx->ix, ctx->d_recs.as<NodeRec>(), ctx->sc, ctx->sv, (int)nq);
        CU(cudaGetLastError());
    }
    CU(cudaStreamSynchronize(ctx->stream));
    return RTX_OK;
}

RTX_API int rtx_shard_records_buffers(rtx_ctx* ctx, void** send_ptr, uint64_t* send_bytes, void** recv_ptr, uint64_t* recv_bytes) {
    if (!ctx || !send_ptr || !send_bytes || !recv_ptr || !recv_bytes) return RTX_ERR_INVALID;
    if (!ctx->has_batch || ctx->shard_phase < 1) return set_err(ctx, RTX_ERR_INVALID, "rtx_shard_records_buffers: run rtx_shard_phase1 first");
    const uint64_t b = (uint64_t)ctx->bv.n_queries * ctx->sv.n_strad * sizeof(ShardRec);
    *send_ptr = ctx->d_send.p;
    *send_bytes = b;
    *recv_ptr = ctx->d_recv.p;
    *recv_bytes = b * ctx->sv.n_shards;
    return RTX_OK;
}

RTX_API int rtx_shard_phase3(rtx_ctx* ctx) {
    int rc = shard_precheck(ctx, 2, "rtx_shard_phase3");
    if (rc) return rc;
    BatchView& bv = ctx->bv;
    const u32 nq = bv.n_queries;
    ctx->shard_phase = 3;
    if (nq == 0) return RTX_OK;
    if (ctx->sv.n_strad) {
        shard_combine_kernel<<<(nq + 127) / 128, 128, 0, ctx->stream>>>(ctx->sv, ctx->d_recs.as<NodeRec>(), (int)nq);
        CU(cudaGetLastError());
    }
    rc = launch_walk<true>(ctx, ctx->sv, ctx->sc, 0, (int)nq, ctx->stream);
    if (rc) return rc;
    ctx->cur_stream = ctx->stream;
    rc = order_results(ctx);
    if (rc) return rc;
    CU(cudaEventRecord(ctx->ev_done, ctx->stream));
    ctx->prof.queries += nq;
    ctx->runs_since_download += 1;
    ctx->ran = true;
    return RTX_OK;
}

// =========================================================================================================
// Reference-sharded mode over NCCL (BASELINE config 5; north_star: "an NCCL-over-NVLink allreduce of the small per-query count
// histograms and a gather of the above-threshold hits").  One rank = one context = one GPU; the ranks may be processes (torchrun,
// MPI) or threads of one process.  The exchange prob.rs:62-73 forces -- cmf_prod_components needs the count histogram over ALL
// references -- is an in-place ncclAllReduce(ncclUint32, ncclSum) on the sub-batch's rows of the histogram buffer; the straddler
// records travel by ncclAllGather; the result lines reach the root by ncclSend / ncclRecv and are merged there on the device.
// libnccl is bound at run time (dlopen: the copy a host framework already loaded, else the system's), so that the library has no
// link-time dependency for the single-GPU and query-partitioned cases.
// =========================================================================================================
namespace {
struct NcclApi {
    void* lib = nullptr;
    std::string err;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool ok() const { return lib != nullptr && err.empty(); }
};

NcclApi load_nccl() {
    NcclApi a;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {  // the copy already in the process (e.g. the one a Python framework bundles) wins
        a.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL | RTLD_NOLOAD);
        if (a.lib) break;
    }
    for (const char* n : names) {
        if (a.lib) break;
        a.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    }
    if (!a.lib) {
        a.err = std::string("libnccl.so.2 not found: ") + (dlerror() ? dlerror() : "");
        return a;
    }
    auto sym = [&](const char* n) -> void* {
        void* p = dlsym(a.lib, n);
        if (!p && a.err.empty()) a.err = std::string("libnccl lacks ") + n;
        return p;
    };
    a.GetUniqueId = (decltype(a.GetUniqueId))sym("ncclGetUniqueId");
    a.CommInitRank = (decltype(a.CommInitRank))sym("ncclCommInitRank");
    a.CommDestroy = (decltype(a.CommDestroy))sym("ncclCommDestroy");
    a.AllReduce = (decltype(a.AllReduce))sym("ncclAllReduce");
    a.AllGather = (decltype(a.AllGather))sym("ncclAllGather");
    a.Send = (decltype(a.Send))sym("ncclSend");
    a.Recv = (decltype(a.Recv))sym("ncclRecv");
    a.GroupStart = (decltype(a.GroupStart))sym("ncclGroupStart");
    a.GroupEnd = (decltype(a.GroupEnd))sym("ncclGroupEnd");
    a.GetErrorString = (decltype(a.GetErrorString))sym("ncclGetErrorString");
    return a;
}
NcclApi& nccl() {
    static NcclApi api = load_nccl();
    return api;
}
}  // namespace

#define NC(call)                                                                                                                  \
    do {                                                                                                                          \
        ncclResult_t r__ = (call);                                                                                                \
        if (r__ != ncclSuccess) return set_err(ctx, RTX_ERR_CUDA, std::string(#call) + ": " + nccl().GetErrorString(r__));        \
    } while (0)

RTX_API int rtx_comm_unique_id(void* out) {
    rtx_ctx* ctx = nullptr;
    if (!out) return set_err(nullptr, RTX_ERR_INVALID, "rtx_comm_unique_id: out is NULL");
    if (!nccl().ok()) return set_err(nullptr, RTX_ERR_UNSUPPORTED, "NCCL unavailable: " + nccl().err);
    ncclUniqueId id;
    NC(nccl().GetUniqueId(&id));
    static_assert(sizeof(id) == RTX_COMM_UNIQUE_ID_BYTES, "ncclUniqueId size");
    memcpy(out, &id, sizeof id);
    return RTX_OK;
}

RTX_API int rtx_comm_init(rtx_ctx* ctx, const void* unique_id, int rank, int nranks) {
    if (!ctx) return RTX_ERR_INVALID;
    REQUIRE(unique_id != nullptr && nranks >= 1 && rank >= 0 && rank < nranks, "rtx_comm_init: bad rank / nranks / id");
    if (!nccl().ok()) return set_err(ctx, RTX_ERR_UNSUPPORTED, "NCCL unavailable: " + nccl().err);
    CU(cudaSetDevice(ctx->device));
    if (ctx->comm) {
        nccl().CommDestroy((ncclComm_t)ctx->comm);
        ctx->comm = nullptr;
    }
    ncclUniqueId id;
    memcpy(&id, unique_id, sizeof id);
    ncclComm_t comm = nullptr;
    NC(nccl().CommInitRank(&comm, nranks, id, rank));
    ctx->comm = comm;
    ctx->comm_rank = rank;
    ctx->comm_size = nranks;
    return RTX_OK;
}

RTX_API int rtx_comm_destroy(rtx_ctx* ctx) {
    if (!ctx) return RTX_ERR_INVALID;
    if (ctx->comm) {
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        cudaStreamSynchronize(ctx->stream2);
        nccl().CommDestroy((ncclComm_t)ctx->comm);
        ctx->comm = nullptr;
    }
    ctx->comm_size = 0;
    return RTX_OK;
}

static int comm_precheck(rtx_ctx* ctx, const char* who) {
    if (!ctx) return RTX_ERR_INVALID;
    if (!ctx->comm) return set_err(ctx, RTX_ERR_INVALID, std::string(who) + ": no communicator (rtx_comm_init)");
    if ((int)ctx->sv.n_shards != ctx->comm_size || (int)ctx->sv.rank != ctx->comm_rank)
        return set_err(ctx, RTX_ERR_INVALID, std::string(who) + ": the index must be uploaded as shard `rank` of `nranks` shards of the communicator");
    if (!ctx->has_batch) return set_err(ctx, RTX_ERR_INVALID, std::string(who) + ": no batch uploaded");
    return RTX_OK;
}

// All phases of the uploaded batch.  The batch is cut into sub-batches (the same cut on every rank: the smallest of the ranks'
// own choices) that alternate between two scratch slots: hit counting of sub-batch i+1 runs on `stream` while the histogram
// all-reduce, the probability / prefix / record kernels, the record all-gather and the tree walk of sub-batch i run on `stream2`.
RTX_API int rtx_shard_run(rtx_ctx* ctx) {
    int rc = comm_precheck(ctx, "rtx_shard_run");
    if (rc) return rc;
    CU(cudaSetDevice(ctx->device));
    BatchView& bv = ctx->bv;
    const u32 nq = bv.n_queries;
    ncclComm_t comm = (ncclComm_t)ctx->comm;
    ctx->merged = false;
    // the ranks agree on the sub-batch size (each sized its own from its free memory) -- once per upload
    if (!ctx->sub_batch_agreed) {
        CU(ctx->d_agree.ensure(8));
        const u32 mine = nq ? ctx->sub_batch : 0xFFFFFFFFu;
        CU(cudaMemcpyAsync(ctx->d_agree.p, &mine, 4, cudaMemcpyHostToDevice, ctx->stream));
        NC(nccl().AllReduce(ctx->d_agree.p, ctx->d_agree.p, 1, ncclUint32, ncclMin, comm, ctx->stream));
        u32 agreed = 0;
        CU(cudaMemcpyAsync(&agreed, ctx->d_agree.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        if (nq) ctx->sub_batch = std::max(1u, std::min(agreed, ctx->sub_batch));
        ctx->sub_batch_agreed = true;
    }
    if (nq == 0) {
        ctx->shard_phase = 3;
        ctx->ran = true;
        return RTX_OK;
    }
    const u32 sb = ctx->sub_batch;
    const bool pipe = ctx->two_slots && nq > sb;
    rc = begin_run(ctx);
    if (rc) return rc;
    const size_t S = ctx->sv.n_strad;
    const u32 R = ctx->sv.n_shards;
    const int n_slots = pipe ? 2 : 1;
    for (int s = 0; s < n_slots; ++s) {  // exchange buffers per scratch slot, sized for one sub-batch
        CU(ctx->d_send_s[s].ensure(std::max<size_t>(1, (size_t)sb * S) * sizeof(ShardRec)));
        CU(ctx->d_recv_s[s].ensure(std::max<size_t>(1, (size_t)sb * S) * sizeof(ShardRec) * R));
        CU(ctx->d_sk_s[s].ensure(std::max<size_t>(1, (size_t)sb * S)));
        CU(ctx->d_sany_s[s].ensure(std::max<size_t>(1, (size_t)sb * S)));
        CU(ctx->d_sbest_s[s].ensure(std::max<size_t>(1, (size_t)sb * S) * 4));
    }
    CU(cudaMemsetAsync(ctx->d_hist.p, 0, (size_t)nq * bv.hstride * 4, ctx->stream));
    CU(cudaMemsetAsync(ctx->d_pool_used.p, 0, 8, ctx->stream));
    CU(cudaMemsetAsync(ctx->d_hits.p, 0, 8, ctx->stream));
    {
        LaunchTimer lt(ctx, RTX_K_KMERS);
        kmers_kernel<<<nq, kKmerThreads, 0, ctx->stream>>>(ctx->ix, bv);
        CU(cudaGetLastError());
    }
    u32 i_sub = 0;
    for (u32 q0 = 0; q0 < nq; q0 += sb, ++i_sub) {
        const int qb = (int)std::min<u32>(sb, nq - q0);
        const int slot = pipe ? (int)(i_sub & 1u) : 0;
        ctx->cur_counts = slot ? ctx->d_counts1.as<u16>() : ctx->d_counts.as<u16>();
        ctx->cur_sc = slot ? &ctx->sc1 : &ctx->sc;
        ctx->cur_stream = ctx->stream;
        if (pipe && i_sub >= 2) CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_post[slot], 0));  // the slot's previous tenant is done
        rc = run_phase1(ctx, (int)q0, qb);
        if (rc) return rc;
        if ((bv.flags & RTX_SKIP_EXACT_MATCHES) && bv.exact_off) {
            LaunchTimer lt(ctx, RTX_K_FIXUP);
            fixup_exact_kernel<<<(qb + 127) / 128, 128, 0, ctx->stream>>>(ctx->ix, bv, ctx->cur_counts, (int)q0, qb);
            CU(cudaGetLastError());
        }
        if (pipe) {
            CU(cudaEventRecord(ctx->ev_hit[slot], ctx->stream));
            ctx->cur_stream = ctx->stream2;
            CU(cudaStreamWaitEvent(ctx->stream2, ctx->ev_hit[slot], 0));
        }
        cudaStream_t st = ctx->cur_stream;
        {   // prob.rs:62-73 needs the histogram over all references
            LaunchTimer lt(ctx, RTX_K_ALLREDUCE);
            u32* h = ctx->d_hist.as<u32>() + (size_t)q0 * bv.hstride;
            NC(nccl().AllReduce(h, h, (size_t)qb * bv.hstride, ncclUint32, ncclSum, comm, st));
            ctx->prof.allreduce_bytes += (u64)qb * bv.hstride * 4;
        }
        rc = launch_prob(ctx, (int)q0, qb);
        if (rc) return rc;
        ShardView sv = ctx->sv;
        sv.send = ctx->d_send_s[slot].as<ShardRec>();
        sv.recv = ctx->d_recv_s[slot].as<ShardRec>();
        sv.sk = ctx->d_sk_s[slot].as<u8>();
        sv.sany = ctx->d_sany_s[slot].as<u8>();
        sv.sbest = ctx->d_sbest_s[slot].as<u32>();
        if (S) {
            {
                LaunchTimer lt(ctx, RTX_K_SHARD);
                const long long warps = (long long)qb * (long long)S;
                shard_records_kernel<<<(unsigned)((warps * 32 + 127) / 128), 128, 0, st>>>(ctx->ix, ctx->d_recs.as<NodeRec>(), *ctx->cur_sc, sv, qb);
                CU(cudaGetLastError());
            }
            {
                LaunchTimer lt(ctx, RTX_K_ALLGATHER);
                NC(nccl().AllGather(sv.send, (void*)sv.recv, (size_t)qb * S * sizeof(ShardRec), ncclUint8, comm, st));
                ctx->prof.allgather_bytes += (u64)qb * S * sizeof(ShardRec) * R;
            }
            {
                LaunchTimer lt(ctx, RTX_K_SHARD);
                shard_combine_kernel<<<(qb + 127) / 128, 128, 0, st>>>(sv, ctx->d_recs.as<NodeRec>(), qb);
                CU(cudaGetLastError());
            }
        }
        rc = launch_walk<true>(ctx, sv, *ctx->cur_sc, (int)q0, qb, st);
        if (rc) return rc;
        if (pipe) CU(cudaEventRecord(ctx->ev_post[slot], ctx->stream2));
    }
    if (pipe) {
        CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_post[0], 0));
        if (i_sub >= 2) CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_post[1], 0));
    }
    ctx->cur_stream = ctx->stream;
    ctx->cur_counts = ctx->d_counts.as<u16>();
    ctx->cur_sc = &ctx->sc;
    rc = order_results(ctx);
    if (rc) return rc;
    CU(cudaEventRecord(ctx->ev_done, ctx->stream));
    ctx->shard_phase = 3;
    ctx->prof.queries += nq;
    ctx->runs_since_download += 1;
    ctx->ran = true;
    return RTX_OK;
}

// The ranks' result lines -> root, merged there (shard_merge_*_kernel): afterwards rtx_batch_download returns the batch's final lines
// on the root and no lines on the other ranks.
RTX_API int rtx_shard_gather(rtx_ctx* ctx, int root) {
    int rc = comm_precheck(ctx, "rtx_shard_gather");
    if (rc) return rc;
    REQUIRE(root >= 0 && root < ctx->comm_size, "rtx_shard_gather: bad root");
    if (!ctx->ran) return set_err(ctx, RTX_ERR_INVALID, "rtx_shard_gather: nothing was run");
    CU(cudaSetDevice(ctx->device));
    const u32 nq = ctx->bv.n_queries;
    const u32 R = (u32)ctx->comm_size, ML = ctx->ix.max_levels;
    const bool is_root = ctx->comm_rank == root;
    ncclComm_t comm = (ncclComm_t)ctx->comm;
    cudaStream_t st = ctx->stream;
    if (nq == 0) {
        ctx->merged = true;
        ctx->merged_lines = 0;
        return RTX_OK;
    }
    // a result pool that overflowed on ANY rank is grown there and the batch re-run on ALL ranks (the collectives need everybody)
    CU(ctx->d_agree.ensure(16));
    for (int attempt = 0;; ++attempt) {
        unsigned long long h[2] = {0, 0}, g[2] = {0, 0};
        CU(cudaMemcpyAsync(&h[0], ctx->d_pool_used.p, 8, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        h[1] = h[0] > ctx->pool.cap ? 1ull : 0ull;
        CU(cudaMemcpyAsync(ctx->d_agree.p, h, 16, cudaMemcpyHostToDevice, st));
        NC(nccl().AllReduce(ctx->d_agree.p, ctx->d_agree.p, 2, ncclUint64, ncclMax, comm, st));
        CU(cudaMemcpyAsync(g, ctx->d_agree.p, 16, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        if (!g[1]) break;
        if (attempt >= 2) return set_err(ctx, RTX_ERR_CUDA, "rtx_shard_gather: the result pool keeps overflowing");
        if (h[1]) {
            rc = ensure_pool(ctx, h[0] + h[0] / 4 + 1024);
            if (rc) return rc;
        }
        rc = rtx_shard_run(ctx);
        if (rc) return rc;
    }
    // every rank's per-query offsets everywhere (4 bytes per query and rank), then the totals on the host
    CU(ctx->d_all_begin.ensure((size_t)R * (nq + 1) * 4));
    {
        LaunchTimer lt(ctx, RTX_K_ALLGATHER);
        NC(nccl().AllGather(ctx->d_ord_begin.p, ctx->d_all_begin.p, (size_t)nq + 1, ncclUint32, comm, st));
        ctx->prof.allgather_bytes += (u64)R * (nq + 1) * 4;
    }
    std::vector<u32> tot(R), off(R + 1, 0);
    CU(cudaMemcpy2DAsync(tot.data(), 4, ctx->d_all_begin.as<u32>() + nq, (size_t)(nq + 1) * 4, 4, R, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (u32 r = 0; r < R; ++r) off[r + 1] = off[r] + tot[r];
    const u64 all = off[R];
    const u32 mine = tot[ctx->comm_rank];
    if (is_root) {
        CU(ctx->d_g_first.ensure(std::max<u64>(all, 1) * 4));
        CU(ctx->d_g_nlev.ensure(std::max<u64>(all, 1)));
        CU(ctx->d_g_conf.ensure(std::max<u64>(all, 1) * ML * 8));
        CU(ctx->d_g_local.ensure(std::max<u64>(all, 1) * 8));
        CU(ctx->d_rank_off.ensure((R + 1) * 4));
        CU(cudaMemcpyAsync(ctx->d_rank_off.p, off.data(), (R + 1) * 4, cudaMemcpyHostToDevice, st));
    }
    {
        LaunchTimer lt(ctx, RTX_K_GATHER);
        NC(nccl().GroupStart());
        if (!is_root) {
            if (mine) {
                NC(nccl().Send(ctx->d_ord_first.p, (size_t)mine * 4, ncclUint8, root, comm, st));
                NC(nccl().Send(ctx->d_ord_nlev.p, (size_t)mine, ncclUint8, root, comm, st));
                NC(nccl().Send(ctx->d_ord_conf.p, (size_t)mine * ML * 8, ncclUint8, root, comm, st));
                NC(nccl().Send(ctx->d_ord_local.p, (size_t)mine * 8, ncclUint8, root, comm, st));
            }
        } else {
            for (u32 r = 0; r < R; ++r) {
                if ((int)r == root || !tot[r]) continue;
                NC(nccl().Recv(ctx->d_g_first.as<u32>() + off[r], (size_t)tot[r] * 4, ncclUint8, (int)r, comm, st));
                NC(nccl().Recv(ctx->d_g_nlev.as<u8>() + off[r], (size_t)tot[r], ncclUint8, (int)r, comm, st));
                NC(nccl().Recv(ctx->d_g_conf.as<double>() + (size_t)off[r] * ML, (size_t)tot[r] * ML * 8, ncclUint8, (int)r, comm, st));
                NC(nccl().Recv(ctx->d_g_local.as<double>() + off[r], (size_t)tot[r] * 8, ncclUint8, (int)r, comm, st));
            }
        }
        NC(nccl().GroupEnd());
        ctx->prof.gather_bytes += is_root ? (all - mine) * (4 + 1 + 8 + (u64)ML * 8) : (u64)mine * (4 + 1 + 8 + (u64)ML * 8);
    }
    if (!is_root) {
        CU(cudaMemsetAsync(ctx->d_ord_begin.p, 0, ((size_t)nq + 1) * 4, st));
        CU(cudaEventRecord(ctx->ev_done, st));
        ctx->merged = true;
        ctx->merged_lines = 0;
        return RTX_OK;
    }
    if (mine) {  // the root's own lines take their place among the gathered ones
        CU(cudaMemcpyAsync(ctx->d_g_first.as<u32>() + off[root], ctx->d_ord_first.p, (size_t)mine * 4, cudaMemcpyDeviceToDevice, st));
        CU(cudaMemcpyAsync(ctx->d_g_nlev.as<u8>() + off[root], ctx->d_ord_nlev.p, (size_t)mine, cudaMemcpyDeviceToDevice, st));
        CU(cudaMemcpyAsync(ctx->d_g_conf.as<double>() + (size_t)off[root] * ML, ctx->d_ord_conf.p, (size_t)mine * ML * 8, cudaMemcpyDeviceToDevice, st));
        CU(cudaMemcpyAsync(ctx->d_g_local.as<double>() + off[root], ctx->d_ord_local.p, (size_t)mine * 8, cudaMemcpyDeviceToDevice, st));
    }
    // the merged lines go where the root's own were: those arrays are sized for the pool's capacity
    if (all > ctx->pool.cap) {
        rc = ensure_pool(ctx, all + all / 4 + 1024);
        if (rc) return rc;
    }
    MergeView mv{ctx->d_all_begin.as<u32>(), ctx->d_rank_off.as<u32>(), ctx->d_g_first.as<u32>(), ctx->d_g_nlev.as<u8>(), ctx->d_g_conf.as<double>(),
                 ctx->d_g_local.as<double>(), R, nq, ML, 0};
    {
        LaunchTimer lt(ctx, RTX_K_SHARD);
        shard_merge_count_kernel<<<(nq + 255) / 256, 256, 0, st>>>(mv, ctx->bv, ctx->pool);
        CU(cudaGetLastError());
        result_scan_kernel<<<1, kScanThreads, 0, st>>>(ctx->pool, ctx->d_ord_begin.as<u32>(), nq);
        CU(cudaGetLastError());
        shard_merge_write_kernel<<<(nq + 7) / 8, 256, 0, st>>>(mv, ctx->bv, ctx->ix, ctx->d_ord_begin.as<u32>(), ctx->d_ord_first.as<u32>(),
                                                              ctx->d_ord_nlev.as<u8>(), ctx->d_ord_conf.as<double>(), ctx->d_ord_local.as<double>());
        CU(cudaGetLastError());
    }
    CU(cudaEventRecord(ctx->ev_done, st));
    ctx->merged = true;
    ctx->merged_lines = ~0ull;  // read from ord_begin[nq] by the download
    return RTX_OK;
}

RTX_API int rtx_shard_classify(rtx_ctx* ctx, const rtx_batch* batch, rtx_results* results, int root) {
    if (!ctx) return RTX_ERR_INVALID;
    REQUIRE(results != nullptr, "results is NULL");
    int rc = rtx_batch_upload(ctx, batch);
    if (rc == RTX_OK) rc = rtx_shard_run(ctx);
    if (rc == RTX_OK) rc = rtx_shard_gather(ctx, root);
    if (rc == RTX_OK) rc = rtx_batch_download(ctx, results);
    return rc;
}

// ---- in-process exchange between the shards of one process (stand-ins for ncclAllReduce / ncclAllGather) ---------------------
static int exchange_precheck(rtx_ctx* const* ctxs, uint32_t n, int want_phase, const char* who) {
    if (!ctxs || n == 0 || !ctxs[0]) return RTX_ERR_INVALID;
    rtx_ctx* ctx = ctxs[0];
    for (uint32_t r = 0; r < n; ++r) {
        rtx_ctx* c = ctxs[r];
        if (!c || !c->has_batch || c->shard_phase != want_phase) return set_err(ctx, RTX_ERR_INVALID, std::string(who) + ": every context must have finished phase " + std::to_string(want_phase));
        if (c->sv.n_shards != n || c->sv.rank != r) return set_err(ctx, RTX_ERR_INVALID, std::string(who) + ": contexts must be passed in shard order, one per shard");
        if (c->bv.n_queries != ctx->bv.n_queries || c->bv.hstride != ctx->bv.hstride || c->sv.n_strad != ctx->sv.n_strad)
            return set_err(ctx, RTX_ERR_INVALID, std::string(who) + ": the contexts hold different batches");
    }
    return RTX_OK;
}

RTX_API int rtx_shard_exchange_hist_local(rtx_ctx* const* ctxs, uint32_t n) {
    int rc = exchange_precheck(ctxs, n, 1, "rtx_shard_exchange_hist_local");
    if (rc) return rc;
    rtx_ctx* ctx = ctxs[0];
    const size_t n_el = (size_t)ctx->bv.n_queries * ctx->bv.hstride;
    if (n_el == 0 || n == 1) return RTX_OK;
    CU(cudaSetDevice(ctx->device));
    CU(arena_reserve(ctx, (size_t)n * n_el * 4 + 64 * (size_t)n));
    std::vector<u32*> part(n);
    for (uint32_t r = 0; r < n; ++r) {
        part[r] = (u32*)arena_take(ctx, n_el * 4);
        CU(cudaSetDevice(ctxs[r]->device));
        CU(cudaMemcpyAsync(part[r], ctxs[r]->d_hist.p, n_el * 4, cudaMemcpyDeviceToHost, ctxs[r]->stream));
    }
    for (uint32_t r = 0; r < n; ++r) {
        CU(cudaSetDevice(ctxs[r]->device));
        CU(cudaStreamSynchronize(ctxs[r]->stream));
    }
    for (uint32_t r = 1; r < n; ++r)
        for (size_t i = 0; i < n_el; ++i) part[0][i] += part[r][i];
    for (uint32_t r = 0; r < n; ++r) {
        CU(cudaSetDevice(ctxs[r]->device));
        CU(cudaMemcpyAsync(ctxs[r]->d_hist.p, part[0], n_el * 4, cudaMemcpyHostToDevice, ctxs[r]->stream));
    }
    for (uint32_t r = 0; r < n; ++r) {  // the arena is reused by the next exchange / download
        CU(cudaSetDevice(ctxs[r]->device));
        CU(cudaStreamSynchronize(ctxs[r]->stream));
    }
    return RTX_OK;
}

RTX_API int rtx_shard_exchange_records_local(rtx_ctx* const* ctxs, uint32_t n) {
    int rc = exchange_precheck(ctxs, n, 2, "rtx_shard_exchange_records_local");
    if (rc) return rc;
    rtx_ctx* ctx = ctxs[0];
    const size_t b = (size_t)ctx->bv.n_queries * ctx->sv.n_strad * sizeof(ShardRec);
    if (b == 0) return RTX_OK;
    CU(cudaSetDevice(ctx->device));
    CU(arena_reserve(ctx, (size_t)n * b + 64));
    unsigned char* all = (unsigned char*)arena_take(ctx, (size_t)n * b);
    for (uint32_t r = 0; r < n; ++r) {
        CU(cudaSetDevice(ctxs[r]->device));
        CU(cudaMemcpyAsync(all + (size_t)r * b, ctxs[r]->d_send.p, b, cudaMemcpyDeviceToHost, ctxs[r]->stream));
    }
    for (uint32_t r = 0; r < n; ++r) {
        CU(cudaSetDevice(ctxs[r]->device));
        CU(cudaStreamSynchronize(ctxs[r]->stream));
    }
    for (uint32_t r = 0; r < n; ++r) {
        CU(cudaSetDevice(ctxs[r]->device));
        CU(cudaMemcpyAsync(ctxs[r]->d_recv.p, all, (size_t)n * b, cudaMemcpyHostToDevice, ctxs[r]->stream));
    }
    for (uint32_t r = 0; r < n; ++r) {
        CU(cudaSetDevice(ctxs[r]->device));
        CU(cudaStreamSynchronize(ctxs[r]->stream));
    }
    return RTX_OK;
}

// ---- measurement -------------------------------------------------------------------------------------------
RTX_API int rtx_profile_reset(rtx_ctx* ctx) {
    if (!ctx) return RTX_ERR_INVALID;
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaStreamSynchronize(ctx->parked.stream));
    CU(cudaStreamSynchronize(ctx->stream_cp));
    drain_events(ctx);
    ctx->prof = rtx_profile{};
    ctx->runs_since_download = 0;
    ctx->parked.runs_since_download = 0;
    return RTX_OK;
}

RTX_API int rtx_profile_get(rtx_ctx* ctx, rtx_profile* out) {
    if (!ctx || !out) return RTX_ERR_INVALID;
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaStreamSynchronize(ctx->parked.stream));
    drain_events(ctx);
    *out = ctx->prof;
    return RTX_OK;
}

