/* raxtax_b200.h -- C ABI of the B200 (sm_100a) query-classification library.
 *
 * Drop-in boundary for the per-query body of raxtax's driver loop: reference src/raxtax.rs:41-84
 * (`intersect_buffer.fill(0)` ... the one-exact-match override), i.e. everything between "a parsed query"
 * and "a Vec<EvaluationResult>" (src/lineage.rs:7-14).  FASTA parsing, Tree construction, the exact-match
 * hash map, string formatting, logging and checkpointing stay on the host side of this boundary
 * (see include/raxtax_host.h for the C++ host that mirrors the reference's `raxtax()` signature and
 * INTEGRATION.md for the Rust `extern "C"` block a maintainer would add in src/raxtax.rs).
 *
 * Conventions: plain pointers and sizes, little-endian, caller owns every host buffer, the library owns
 * every device allocation.  Every call returns 0 on success and a negative rtx_status on failure;
 * rtx_last_error() gives the message.  One rtx_ctx per GPU, used from one host thread at a time; contexts
 * are independent, so N GPUs = N contexts driven by N threads or N processes.  There is no CPU fallback:
 * without a usable CUDA device rtx_ctx_create fails.
 */
#ifndef RAXTAX_B200_H
#define RAXTAX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTX_ABI_VERSION 4
#define RTX_MAX_LEVELS 32 /* deepest lineage (comma-separated ranks) the device tree walk supports */
#define RTX_MAX_RESULTS_PER_QUERY 256 /* >= the 200 lines a query can produce with the 0.01 cutoff */

typedef enum {
    RTX_OK = 0,
    RTX_ERR_INVALID = -1,     /* bad argument / violated input contract */
    RTX_ERR_CUDA = -2,        /* CUDA runtime error (message has the CUDA string) */
    RTX_ERR_NO_DEVICE = -3,   /* no CUDA device: the library has no CPU path */
    RTX_ERR_NO_INDEX = -4,    /* classify before rtx_index_upload */
    RTX_ERR_UNSUPPORTED = -5, /* input outside the supported envelope (e.g. > 8191 unique 8-mers in one query) */
    RTX_ERR_ASSERT = -6       /* an invariant the reference asserts on failed (raxtax.rs:72, prob.rs:98) */
} rtx_status;

typedef struct rtx_ctx rtx_ctx;

/* flags of rtx_batch.flags -- the two switches that reach the hot path (raxtax.rs:17-18) */
#define RTX_SKIP_EXACT_MATCHES 1u /* --skip-exact-matches: zero the counters of exact matches (raxtax.rs:65-68) */
#define RTX_RAW_CONFIDENCE 2u     /* --raw-confidence: disable the one-exact-match override (raxtax.rs:73-84) */

/* hit-count kernel variants (rtx_ctx_set_option(RTX_OPT_HITCOUNT_VARIANT)) */
#define RTX_HITCOUNT_BITROWS 0 /* bit-row positional popcount (default) */
#define RTX_HITCOUNT_CSR 1     /* CSR postings + shared-memory counters (the reference's data structure) */

typedef enum {
    RTX_OPT_HITCOUNT_VARIANT = 1,
    RTX_OPT_SUB_BATCH = 2,      /* queries per device sub-batch (0 = auto) */
    RTX_OPT_KEEP_CSR = 3,       /* keep the CSR postings resident after building bit rows (needed for variant CSR) */
    RTX_OPT_PROFILE = 4,        /* record a CUDA event pair around every kernel launch (rtx_profile_get) */
    RTX_OPT_HITCOUNT_MAX_TILES = 6, /* warp tiles (64 words each) per CTA; fewer = more reference tile groups (L2 blocking); 0 = default */
    RTX_OPT_HITCOUNT_GROUP = 7,     /* queries per CTA (one per warp) of the query-group bit-row kernel: 0 = library default (4; 16 when the
                                       bit rows reach 6 GB), 1 = single-query kernel (one query per CTA), 2..16 = group size; the size is
                                       halved for long queries, and a sub-batch smaller than it runs the single-query kernel */
    RTX_OPT_WALK_VARIANT = 9,       /* tree walk: 0 = level-synchronous kernel + depth-first retry of overflowing queries (default),
                                       1 = depth-first walker only, 3 = level-synchronous without the large-frontier paths (every child
                                       of a frontier node is evaluated), 4 = test hook: those paths (mass-pruned search, arg-max over the
                                       kept segments) forced on every frontier */
    RTX_OPT_PIPELINE = 11,          /* 1: batches of >= 4096 queries are cut into >= 4 sub-batches and hit counting of sub-batch i+1 overlaps
                                       probabilities / prefix sums / tree walk of sub-batch i on a second, higher-priority stream;
                                       0 (default) = serial: on B200 the overlap only recovers what the shorter launches lose */
    RTX_OPT_WALK_LOG_CAP = 10       /* test hook: significant-node log capacity of the level-synchronous walk (0 = full); queries that
                                       exceed it take the depth-first retry path */
} rtx_option;

/* ---- context ------------------------------------------------------------------------------------------- */
int rtx_abi_version(void);
int rtx_ctx_create(int device_ordinal, rtx_ctx** out);
void rtx_ctx_destroy(rtx_ctx* ctx);
const char* rtx_last_error(const rtx_ctx* ctx); /* ctx may be NULL: error of the last failed rtx_ctx_create */
int rtx_ctx_set_option(rtx_ctx* ctx, int option, int64_t value);
/* the CUDA stream (cudaStream_t) all of this context's work is issued on; lets a caller record its own events */
void* rtx_ctx_stream(rtx_ctx* ctx);
int rtx_ctx_device(const rtx_ctx* ctx); /* the CUDA device ordinal the context was created on */
int rtx_ctx_synchronize(rtx_ctx* ctx);
/* Page-locked host memory for batch inputs and result arrays.  Optional: every call accepts ordinary memory (results then pass
 * through the context's own pinned staging arena and one memcpy); buffers from rtx_host_alloc -- or registered by the caller with
 * cudaHostRegister -- are written by DMA directly.  No counterpart in the reference (its results are owned Strings, raxtax.rs:85-88). */
int rtx_host_alloc(size_t bytes, void** out);
int rtx_host_free(void* p);

/* ---- reference index ("Tree", src/tree.rs:36-43) --------------------------------------------------------
 * Flattened form of what Tree::new (tree.rs:47-140) builds:
 *  - reference ids are positions in the lineage-sorted order (tree.rs:53-54), n_refs = Tree.num_tips;
 *  - k_mer_map (tree.rs:41,134-137) as CSR: csr_offsets[65537], csr_ids ascending and unique per list -- or, instead,
 *    the sorted reference sequences (ref_seq_*), from which the device builds its index directly;
 *  - the Node tree (tree.rs:189-194) without its childless Sequence leaves (they never influence
 *    Lineage::evaluate, lineage.rs:119-179, because their parent is never Inner), numbered so that the children of node i are the consecutive
 *    nodes child_first[i] .. child_first[i]+child_count[i]-1 in the reference's child order; node 0 = root;
 *    node_lo/node_hi = confidence_range (global reference ids);
 *  - ref_levels[r] = number of comma-separated ranks of lineages[r] (used by the override, raxtax.rs:79).
 * Reference sharding: this context holds the postings of references [ref_shard_begin, ref_shard_end) only;
 * csr_ids outside that range are ignored.  The node tree and ref_levels are always the full ones.
 */
typedef struct {
    uint64_t n_refs;
    const uint64_t* csr_offsets;
    const uint32_t* csr_ids;
    uint32_t n_nodes;
    const uint32_t* node_lo;
    const uint32_t* node_hi;
    const uint8_t* node_type; /* 0 = Inner, 1 = Taxon, 2 = Sequence node that has children (degenerate lineages only) (tree.rs:181-186) */
    const uint32_t* child_first;
    const uint32_t* child_count;
    const uint8_t* ref_levels;
    uint64_t ref_shard_begin;
    uint64_t ref_shard_end; /* 0 = n_refs */
    /* reference-sharded operation over several contexts / ranks (0 or 1 = off): shard r holds references
     * [shard_cuts[r], shard_cuts[r+1]); when n_shards > 1 ref_shard_begin/end are taken from shard_cuts[shard_rank]. */
    uint32_t n_shards;
    uint32_t shard_rank;
    const uint64_t* shard_cuts; /* [n_shards + 1], shard_cuts[0] = 0, shard_cuts[n_shards] = n_refs */
    /* Alternative to the CSR (used when csr_offsets == NULL): the lineage-sorted reference sequences themselves, 4-bit codes as
     * parser.rs:11-34, reference r = ref_seq_codes[ref_seq_offsets[r] .. ref_seq_offsets[r+1]).  The library then does the windowing
     * and de-duplication of tree.rs:114-123,134-137 on the device and never materialises k_mer_map (the CSR hit-count variant
     * is unavailable for such an index). */
    const uint64_t* ref_seq_offsets; /* [n_refs + 1] */
    const uint8_t* ref_seq_codes;
} rtx_index_desc;

int rtx_index_upload(rtx_ctx* ctx, const rtx_index_desc* desc);
/* sizes a caller needs to allocate tap buffers */
uint64_t rtx_index_n_refs(const rtx_ctx* ctx);       /* global N */
uint64_t rtx_index_shard_refs(const rtx_ctx* ctx);   /* references held by this context */
uint32_t rtx_batch_sub_batch(const rtx_ctx* ctx);     /* queries per device sub-batch of the uploaded batch (0 = no batch) */
uint32_t rtx_index_max_levels(const rtx_ctx* ctx);   /* stride of rtx_results.confidence */
uint64_t rtx_index_device_bytes(const rtx_ctx* ctx); /* HBM held by the index */
uint64_t rtx_index_bitrow_bytes(const rtx_ctx* ctx); /* of which: the bit rows (k-mer x reference matrix) */
/* the hit-count kernel instantiation the last launch used, as ncu names it (measurement records) */
const char* rtx_hitcount_kernel_name(const rtx_ctx* ctx);

/* ---- query batch (src/raxtax.rs:14-22: `queries: &[(String, Vec<u8>)]` minus the labels) ----------------
 * seq_codes are the 4-bit one-hot codes of parser.rs:11-34.  exact_ids[exact_offsets[q]..exact_offsets[q+1])
 * is `tree.sequences.get(query_sequence)` (raxtax.rs:42) looked up by the host; exact_offsets may be NULL
 * when no query has an exact match.
 */
typedef struct {
    uint32_t n_queries;
    const uint64_t* seq_offsets; /* [n_queries + 1] */
    const uint8_t* seq_codes;
    const uint32_t* exact_offsets; /* [n_queries + 1] or NULL */
    const uint32_t* exact_ids;
    uint32_t flags;
} rtx_batch;

/* ---- results (`Vec<EvaluationResult>` per query, src/lineage.rs:7-14, in the reference's order) ----------
 * Results of query q are entries [result_begin[q], result_begin[q+1]) of the per-result arrays.
 * confidence has row stride rtx_index_max_levels(); values are already rounded to 0.01 (lineage.rs:129)
 * or 1.0 for the override.  Tap buffers are optional (NULL = skip) and exist for parity tests:
 *   tap_counts[q * shard_refs + r]  = intersect_buffer after the skip-zeroing (raxtax.rs:58-68), u16
 *   tap_hist[q * tap_hist_stride + m] = number of references with count m (prob.rs:13-19), this shard only
 *   tap_kmers[q * tap_kmer_stride + i] = sorted unique 8-mers (utils.rs:27-40)
 *   tap_probs[q * tap_prob_stride + m] = normalised probability of a reference with count m (prob.rs:92-102),
 *                                        valid where tap_hist (the global histogram) is non-zero
 */
typedef struct {
    uint16_t* n_kmers;       /* [n_queries] */
    uint32_t* result_begin;  /* [n_queries + 1] */
    double* global_signal;   /* [n_queries] */
    uint64_t result_capacity;
    uint32_t* first_ref;     /* [result_capacity] index into Tree.lineages */
    uint8_t* n_levels;       /* [result_capacity] */
    double* confidence;      /* [result_capacity * max_levels] */
    double* local_signal;    /* [result_capacity] */
    uint64_t n_results;      /* out: total results written (if > result_capacity nothing past capacity is written
                                and the call returns RTX_ERR_INVALID with the needed size here) */
    uint16_t* tap_counts;
    uint32_t* tap_hist;
    uint64_t tap_hist_stride;
    uint16_t* tap_kmers;
    uint64_t tap_kmer_stride;
    double* tap_probs;
    uint64_t tap_prob_stride;
} rtx_results;

/* One call = H2D of the batch, all kernels, D2H of the results (the end-to-end path). */
int rtx_classify_batch(rtx_ctx* ctx, const rtx_batch* batch, rtx_results* results);

/* The same path split so that a caller can keep a batch resident in HBM and time the device part alone:
 * upload (H2D) -> run (kernels only, asynchronous on rtx_ctx_stream) -> download (D2H + host-side ordering). */
int rtx_batch_upload(rtx_ctx* ctx, const rtx_batch* batch);
int rtx_batch_run(rtx_ctx* ctx);
int rtx_batch_download(rtx_ctx* ctx, rtx_results* results);
/* Two batch slots per context (0 = default, 1): rtx_batch_slot selects the slot that rtx_batch_upload / _run / _download (and
 * rtx_classify_batch) act on.  The slots share the context's stream for kernels, but inputs and results move on a separate copy
 * stream, so a caller can keep the device busy: upload + run slot B while slot A's kernels are still executing, then download A
 * (waits for A only) while B runs -- see rxh_raxtax in raxtax_host.cpp.  The reference's counterpart is rayon keeping every core
 * busy with the next chunk (raxtax.rs:35-39). */
int rtx_batch_slot(rtx_ctx* ctx, int slot);

/* ---- reference-sharded mode (north_star: NCCL all-reduce of the per-query count histograms) -------------
 * Every rank uploads the same batch.  Per batch (which must fit one sub-batch):
 *   rtx_shard_phase1      k-mers, local hit counts, local histograms
 *   [all-reduce SUM, in place, of the hist buffer: uint32 [n_queries * hist_stride]]     <- the only O(Q*K) exchange
 *   rtx_shard_phase2      P(count) from the global histogram, local block prefixes, one record per
 *                         (query, straddling node): local mass, local best child, local significant children
 *   [all-gather of the records buffer: send_bytes from every rank -> recv = n_shards * send_bytes, rank order]
 *   rtx_shard_phase3      combines the records, walks the part of the tree this rank owns
 *   rtx_batch_download    this rank's result lines WITHOUT the one-exact-match override; the caller merges the
 *                         ranks' lines per query (sort by confidence vector descending, first_ref ascending) and
 *                         applies the override (raxtax.rs:73-84) -- see raxtax_b200/dist.py.
 * The buffers are device pointers owned by the library, valid until the next rtx_batch_upload.
 */
int rtx_shard_phase1(rtx_ctx* ctx);
int rtx_shard_hist_buffer(rtx_ctx* ctx, void** dev_ptr, uint64_t* n_elems);
int rtx_shard_phase2(rtx_ctx* ctx);
int rtx_shard_records_buffers(rtx_ctx* ctx, void** send_ptr, uint64_t* send_bytes, void** recv_ptr, uint64_t* recv_bytes);
int rtx_shard_phase3(rtx_ctx* ctx);
/* In-process stand-ins for the two collectives when ONE process drives all the shards (several GPUs of a box, or several contexts
 * on one GPU): ctxs[r] is shard r of n.  ..._hist_local: element-wise sum of the histogram buffers, written back to every context
 * (between phase 1 and 2).  ..._records_local: the straddler records of all shards, in shard order, into every context's receive
 * buffer (between phase 2 and 3).  Staged through pinned host memory (~2.6 KB of histogram per query and shard).  With one process
 * per GPU use ncclAllReduce / ncclAllGather on the buffers above instead (raxtax_b200/dist.py). */
int rtx_shard_exchange_hist_local(rtx_ctx* const* ctxs, uint32_t n);
int rtx_shard_exchange_records_local(rtx_ctx* const* ctxs, uint32_t n);

/* ---- reference-sharded mode over NCCL, inside the library ------------------------------------------------
 * One rank = one context = one GPU (processes under torchrun / MPI, or threads of one process).  rtx_comm_unique_id (any one rank;
 * the 128 bytes reach the others out of band) + rtx_comm_init on every rank build the communicator; the index is uploaded as
 * shard `rank` of `nranks` (rtx_index_desc.n_shards / shard_rank / shard_cuts).  Then per batch, on EVERY rank with the same batch:
 *   rtx_batch_upload
 *   rtx_shard_run     k-mers, then per sub-batch: local hit counts | ncclAllReduce(ncclUint32, ncclSum) of the sub-batch's histogram
 *                     rows (in place; the exchange prob.rs:62-73 forces: the product over ALL references) | P(count), local prefixes,
 *                     straddler records | ncclAllGather of the records | combine + tree walk.  Two scratch slots: the collectives and
 *                     the tail kernels of sub-batch i run on a second stream under the hit counting of sub-batch i+1.
 *   rtx_shard_gather  the ranks' result lines -> root (ncclSend / ncclRecv), merged on the root's device in the order of
 *                     lineage.rs:93, then the one-exact-match override (raxtax.rs:73-84)
 *   rtx_batch_download  root: the final lines of the batch, exactly what an unsharded context returns; other ranks: no lines
 * rtx_shard_classify = the four in one call.  libnccl.so.2 is bound at run time (the copy already loaded into the process wins);
 * without it rtx_comm_* fail with RTX_ERR_UNSUPPORTED and everything else works. */
#define RTX_COMM_UNIQUE_ID_BYTES 128
int rtx_comm_unique_id(void* out /* RTX_COMM_UNIQUE_ID_BYTES */);
int rtx_comm_init(rtx_ctx* ctx, const void* unique_id, int rank, int nranks);
int rtx_comm_destroy(rtx_ctx* ctx);
int rtx_shard_run(rtx_ctx* ctx);
int rtx_shard_gather(rtx_ctx* ctx, int root);
int rtx_shard_classify(rtx_ctx* ctx, const rtx_batch* batch, rtx_results* results, int root);

/* ---- measurement ---------------------------------------------------------------------------------------- */
typedef struct {
    uint64_t launches;   /* kernel launches since the last reset */
    double total_ms;     /* sum of CUDA-event durations (only with RTX_OPT_PROFILE) */
} rtx_kernel_stat;

enum { RTX_K_KMERS = 0, RTX_K_HITCOUNT = 1, RTX_K_FIXUP = 2, RTX_K_PROB = 3, RTX_K_INDEX = 4, RTX_K_WALK = 5, RTX_K_PREFIX = 6,
       RTX_K_ALLREDUCE = 7 /* histogram all-reduce */, RTX_K_ALLGATHER = 8 /* straddler records, result offsets */,
       RTX_K_SHARD = 9 /* record / combine / merge kernels */, RTX_K_GATHER = 10 /* result lines -> root */, RTX_K_COUNT = 11 };

typedef struct {
    rtx_kernel_stat kernel[RTX_K_COUNT];
    uint64_t queries;          /* queries run since the last reset */
    uint64_t hits;             /* sum over queries of sum_r count[r] = postings a CSR walk would touch */
    uint64_t bitrow_bytes;     /* bytes of bit rows + count vectors the hit-count launches had to move */
    uint64_t csr_equiv_bytes;  /* 4*hits + 2*N per query: the reference data structure's traffic (SURVEY 8d) */
    uint64_t h2d_bytes, d2h_bytes;
    uint64_t allreduce_bytes, allgather_bytes, gather_bytes; /* payload of the collectives (reference-sharded mode over NCCL) */
} rtx_profile;

int rtx_profile_reset(rtx_ctx* ctx);
int rtx_profile_get(rtx_ctx* ctx, rtx_profile* out);

#ifdef __cplusplus
}
#endif
#endif /* RAXTAX_B200_H */
